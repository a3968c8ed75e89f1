"""CPU: lane-level numpy emulation of csr_generic_kernel / sell_generic_kernel (csrc/spmv_generic.cu) against the oracle.

The emulation follows the kernel statement by statement -- the warp-uniform outer loop over groups of 32 / L rows, the lanes
striding through their row, the shuffle tree with `width = L` (a lane whose partner would fall outside its L-lane segment
gets its own value back, as __shfl_down_sync does), lane 0 of a segment writing y -- so it pins the index arithmetic and
the reduction pattern: every row written exactly once, with the complete row sum, for every lane count and for grids
smaller than the matrix (several trips of the loop).  The second half of the file goes further: it compiles the kernels' OWN SOURCE for
the host and runs it (see there).  The GPU parity proper is tests/test_generic_gpu.py."""
import ctypes as C

import generic_emu
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import oracle as O


def shfl_down(v, o, width):
    lane = np.arange(32)
    src = np.where((lane % width) + o < width, lane + o, lane)
    return v[src]


def emulate_csr_generic(off, col, val, x, y, alpha, beta, base, lanes_log2, ctas, block=256):
    lanes = 1 << lanes_log2
    rows = off.size - 1
    rows_per_warp = 32 >> lanes_log2
    nwarps = ctas * block // 32
    written = np.zeros(rows, int)
    lane = np.arange(32)
    sub = lane & (lanes - 1)
    for warp in range(nwarps):
        w0 = warp * rows_per_warp
        while w0 < rows:                                   # warp-uniform trip count
            row = w0 + (lane >> lanes_log2)
            s = np.zeros(32)
            for l in range(32):
                if row[l] < rows:
                    beg, end = int(off[row[l]]) - base, int(off[row[l] + 1]) - base
                    k = beg + sub[l]
                    while k < end:
                        s[l] += val[k] * x[int(col[k]) - base]
                        k += lanes
            o = lanes >> 1
            while o > 0:
                s = s + shfl_down(s, o, lanes)
                o >>= 1
            for l in range(32):
                if row[l] < rows and sub[l] == 0:
                    r = row[l]
                    y[r] = alpha * s[l] if beta == 0 else alpha * s[l] + beta * y[r]
                    written[r] += 1
            w0 += nwarps * rows_per_warp
    return written


@pytest.mark.parametrize("lanes_log2", [2, 3, 4, 5])
@pytest.mark.parametrize("base", [0, 1])
def test_csr_generic_lane_logic(lanes_log2, base):
    rows = 700
    off, col, val = O.rmat_csr(rows, avg_nnz=9, seed=11, val_seed=12)
    x, y0 = O.uniform(13, rows), O.uniform(14, rows)
    want = O.spmv_csr(off, col, val, x, y0, -1.5, 0.5)
    y = y0.copy()
    # one CTA = 8 warps: far fewer rows per sweep than the matrix has -> several trips of the outer loop
    written = emulate_csr_generic(off.astype(np.int64) + base, col.astype(np.int64) + base, val, x, y, -1.5, 0.5, base, lanes_log2, ctas=1)
    assert np.all(written == 1)
    assert np.linalg.norm(y - want) <= 1e-13 * np.linalg.norm(want)


def test_csr_generic_rows_not_a_multiple_of_the_group_and_empty_rows():
    lens = np.array([0, 5, 0, 0, 33, 1, 64, 0, 7, 129, 0])            # 11 rows: the last group of every lane count is partial
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    rng = np.random.default_rng(3)
    col = rng.integers(0, 50, off[-1]).astype(np.int64)
    val = rng.uniform(-1, 1, off[-1])
    x, y0 = rng.uniform(-1, 1, 50), rng.uniform(-1, 1, lens.size)
    want = O.spmv_csr(off.astype(np.int32), col.astype(np.int32), val, x, y0, 2.0, 0.0)
    for lanes_log2 in (2, 3, 4, 5):
        y = np.full(lens.size, np.nan)                                 # beta = 0 never reads y
        written = emulate_csr_generic(off, col, val, x, y, 2.0, 0.0, 0, lanes_log2, ctas=1)
        assert np.all(written == 1)
        assert np.linalg.norm(y - want) <= 1e-13 * np.linalg.norm(want)


def emulate_sell_generic(rows, S, so, sc, sv, x, y, alpha, beta, base):
    for row in range(rows):
        s, r = divmod(row, S)
        beg, end = int(so[s]) - base, int(so[s + 1]) - base
        width = (end - beg) // S
        acc = 0.0
        for k in range(width):
            i = beg + k * S + r
            c = int(sc[i]) - base
            if c < 0:
                continue
            acc += sv[i] * x[c]
        y[row] = alpha * acc if beta == 0 else alpha * acc + beta * y[row]


@pytest.mark.parametrize("S", [2, 7, 32])
def test_sell_generic_index_arithmetic(S):
    rows = 203                                                         # partial last slice
    off, col, val = O.rmat_csr(rows, avg_nnz=5, seed=21, val_seed=22)
    so, sc, sv = O.csr_to_sell(off, col, val, S)
    x, y0 = O.uniform(23, rows), O.uniform(24, rows)
    y = y0.copy()
    emulate_sell_generic(rows, S, so.astype(np.int64), sc.astype(np.int64), sv, x, y, 1.0, 2.0, 0)
    want = O.spmv_csr(off, col, val, x, y0, 1.0, 2.0)
    assert np.linalg.norm(y - want) <= 1e-13 * np.linalg.norm(want)
    assert np.linalg.norm(O.spmv_sell(rows, S, so, sc, sv, x, y0, 1.0, 2.0) - want) <= 1e-13 * np.linalg.norm(want)


# ------------------------------------------------------------------------------------------------------------------
# The kernels' OWN SOURCE on the CPU: csrc/spmv_generic_kernels.cuh compiled for the host on top of
# tests/host_emulation/cuda_emulation.h (a real thread per lane, a barrier-based __shfl_down_sync, a locked atomicAdd) and run
# with the device's launch geometry against scipy / the oracle.  Covers the kernels whose first hardware run is still pending
# (COO, Sliced-ELL, their transposes) as well as the CSR ones already validated on a B200.
# ------------------------------------------------------------------------------------------------------------------
NPI = {0: np.int32, 1: np.int64}
NPF = {0: np.float32, 1: np.float64}
CTF = {0: C.c_float, 1: C.c_double}
# (offsets 64-bit, columns 64-bit, A fp64, x / y fp64): the nine instantiations of spmv_generic.cu's dispatch
COMBOS = [(0, 0, 0, 0), (0, 0, 0, 1), (0, 0, 1, 1), (1, 0, 0, 0), (1, 0, 0, 1), (1, 0, 1, 1), (1, 1, 0, 0), (1, 1, 0, 1), (1, 1, 1, 1)]


@pytest.fixture(scope="module")
def emu():
    return generic_emu.load()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _case(rows, cols, avg, seed, a_dt, xy_dt, transpose, base):
    off, col, val = O.rmat_csr(rows, avg_nnz=avg, seed=seed, val_seed=seed + 1)
    col = col % cols
    val = val.astype(NPF[a_dt])
    nx, ny = (rows, cols) if transpose else (cols, rows)
    x, y0 = O.uniform(seed + 2, nx).astype(NPF[xy_dt]), O.uniform(seed + 3, ny).astype(NPF[xy_dt])
    A = sp.csr_matrix((val.astype(np.float64), col, off), shape=(rows, cols))
    return off, col, val, x, y0, (A.T if transpose else A)


def _tol(xy_dt):
    return 1e-12 if xy_dt else 2e-5


@pytest.mark.parametrize("off64,col64,a_dt,xy_dt", COMBOS)
@pytest.mark.parametrize("transpose", [0, 1])
def test_csr_generic_source_on_the_host(emu, off64, col64, a_dt, xy_dt, transpose):
    rows, cols, base = 300, 211, 1
    off, col, val, x, y0, M = _case(rows, cols, 7, 40 + off64 + 2 * col64, a_dt, xy_dt, transpose, base)
    ct = CTF[xy_dt]
    for lanes_log2, (alpha, beta) in zip((2, 3, 4, 5), ((-1.5, 0.5), (1.0, 0.0), (2.0, 1.0), (0.75, -2.0))):
        y = y0.copy() if beta != 0 else np.full_like(y0, np.nan)          # beta = 0 never reads y
        o, c = (off + base).astype(NPI[off64]), (col + base).astype(NPI[col64])
        rc = emu.emu_csr_generic(off64, col64, a_dt, xy_dt, transpose, lanes_log2, 1, C.c_longlong(rows), C.c_longlong(cols),
                                 C.c_longlong(col.size), _p(o), _p(c), _p(val), C.c_longlong(base), C.byref(ct(alpha)), C.byref(ct(beta)),
                                 _p(x), _p(y))
        assert rc == 0
        want = alpha * (M @ x.astype(np.float64)) + (beta * y0.astype(np.float64) if beta != 0 else 0.0)
        assert np.linalg.norm(y - want) <= _tol(xy_dt) * np.linalg.norm(want), (lanes_log2, alpha, beta)


@pytest.mark.parametrize("idx64,a_dt,xy_dt", [(0, 0, 0), (0, 0, 1), (0, 1, 1), (1, 0, 0), (1, 0, 1), (1, 1, 1)])
@pytest.mark.parametrize("transpose", [0, 1])
def test_coo_generic_source_on_the_host(emu, idx64, a_dt, xy_dt, transpose):
    """Entries in random order; A^T is the same kernel with the index arrays and the shape swapped (the shim's generic_mv)."""
    rows, cols, base = 300, 211, 1
    off, col, val, x, y0, M = _case(rows, cols, 7, 60 + idx64, a_dt, xy_dt, transpose, base)
    row = np.repeat(np.arange(rows), np.diff(off))
    perm = np.random.default_rng(1).permutation(col.size)
    r, c, v = (row[perm] + base).astype(NPI[idx64]), (col[perm] + base).astype(NPI[idx64]), val[perm]
    ct = CTF[xy_dt]
    for alpha, beta in ((-1.5, 0.5), (1.0, 0.0), (2.0, 1.0)):
        y = y0.copy() if beta != 0 else np.full_like(y0, np.nan)
        args = (rows, cols, r, c) if not transpose else (cols, rows, c, r)
        rc = emu.emu_coo_generic(idx64, a_dt, xy_dt, 1, C.c_longlong(args[0]), C.c_longlong(args[1]), C.c_longlong(col.size), _p(args[2]),
                                 _p(args[3]), _p(v), C.c_longlong(base), C.byref(ct(alpha)), C.byref(ct(beta)), _p(x), _p(y))
        assert rc == 0
        want = alpha * (M @ x.astype(np.float64)) + (beta * y0.astype(np.float64) if beta != 0 else 0.0)
        assert np.linalg.norm(y - want) <= _tol(xy_dt) * np.linalg.norm(want), (alpha, beta)


@pytest.mark.parametrize("off64,col64,a_dt,xy_dt", COMBOS)
@pytest.mark.parametrize("transpose,S", [(0, 32), (0, 7), (1, 32), (1, 2)])
def test_sell_generic_source_on_the_host(emu, off64, col64, a_dt, xy_dt, transpose, S):
    rows, cols, base = 203, 150, 1                                       # partial last slice; base 1: padding column is 0
    off, col, val, x, y0, M = _case(rows, cols, 5, 80 + S, a_dt, xy_dt, transpose, base)
    so, sc, sv = O.csr_to_sell((off + base).astype(np.int32), (col + base).astype(np.int32), val, S, base=base)
    ct = CTF[xy_dt]
    for alpha, beta in ((-1.5, 0.5), (1.0, 0.0)):
        y = y0.copy() if beta != 0 else np.full_like(y0, np.nan)
        o, c = so.astype(NPI[off64]), sc.astype(NPI[col64])
        rc = emu.emu_sell_generic(off64, col64, a_dt, xy_dt, transpose, 1, C.c_longlong(rows), C.c_longlong(cols), C.c_longlong(S),
                                  _p(o), _p(c), _p(sv), C.c_longlong(base), C.byref(ct(alpha)), C.byref(ct(beta)), _p(x), _p(y))
        assert rc == 0
        want = alpha * (M @ x.astype(np.float64)) + (beta * y0.astype(np.float64) if beta != 0 else 0.0)
        assert np.linalg.norm(y - want) <= _tol(xy_dt) * np.linalg.norm(want), (alpha, beta)


def _lens_matrix(lens, cols, seed):
    rng = np.random.default_rng(seed)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, max(cols, 1), int(off[-1])).astype(np.int64)
    val = rng.uniform(-1, 1, int(off[-1]))
    return off, col, val


EDGE_SHAPES = {
    "one_by_one_empty": ([0], 1),
    "one_by_one": ([1], 1),
    "single_row": ([37], 50),
    "single_column": ([1] * 40, 1),
    "all_rows_empty": ([0] * 33, 7),
    "first_and_last_rows_empty": ([0, 0, 5, 1, 0, 9, 0], 12),
    "33_rows_one_long": ([1] * 32 + [300], 64),
    "duplicate_columns": ([4, 4, 4], 2),
}


@pytest.mark.parametrize("name", list(EDGE_SHAPES))
def test_generic_sources_on_degenerate_shapes(emu, name):
    """CSR (every lane count), COO and Sliced-ELL (slice sizes below, at and above the row count), A and A^T, on the shapes where
    index arithmetic goes wrong first; fp64 with 64-bit indices, base 0; grid of one CTA."""
    lens, cols = EDGE_SHAPES[name]
    rows = len(lens)
    off, col, val = _lens_matrix(np.array(lens), cols, 7)
    A = sp.csr_matrix((val, col, off), shape=(rows, cols))
    row = np.repeat(np.arange(rows, dtype=np.int64), np.diff(off))
    one, half = C.c_double(1.25), C.c_double(-0.5)
    LL = C.c_longlong
    for transpose in (0, 1):
        M = A.T if transpose else A
        nx, ny = (rows, cols) if transpose else (cols, rows)
        x, y0 = O.uniform(1, nx), O.uniform(2, ny)
        want = 1.25 * (M @ x) - 0.5 * y0
        tol = 1e-13 * max(np.linalg.norm(want), 1.0)
        for lanes_log2 in (2, 3, 4, 5):
            y = y0.copy()
            assert emu.emu_csr_generic(1, 1, 1, 1, transpose, lanes_log2, 1, LL(rows), LL(cols), LL(col.size), _p(off), _p(col), _p(val), LL(0),
                                       C.byref(one), C.byref(half), _p(x), _p(y)) == 0
            assert np.linalg.norm(y - want) <= tol, ("csr", transpose, lanes_log2)
        y = y0.copy()
        a = (rows, cols, row, col) if not transpose else (cols, rows, col, row)
        assert emu.emu_coo_generic(1, 1, 1, 1, LL(a[0]), LL(a[1]), LL(col.size), _p(a[2]), _p(a[3]), _p(val), LL(0), C.byref(one), C.byref(half),
                                   _p(x), _p(y)) == 0
        assert np.linalg.norm(y - want) <= tol, ("coo", transpose)
        for S in (1, 2, 32, 64):
            so, sc, sv = O.csr_to_sell(off.astype(np.int32), col.astype(np.int32), val, S)
            so, sc = so.astype(np.int64), sc.astype(np.int64)
            y = y0.copy()
            assert emu.emu_sell_generic(1, 1, 1, 1, transpose, 1, LL(rows), LL(cols), LL(S), _p(so), _p(sc), _p(sv), LL(0), C.byref(one),
                                        C.byref(half), _p(x), _p(y)) == 0
            assert np.linalg.norm(y - want) <= tol, ("sell", transpose, S)
