"""CPU half of the element-wise checks (tests/elementwise_check.py).

1. Self-test of the comparator: it accepts every correct summation order (scipy, the oracle, a reversed and a pairwise sum
   in the arithmetic type) on `cancel`, `wide` and `nonfinite` inputs, and rejects each planted fault: an fp64 product
   accumulated in fp32, one element moved by 4x its bound, a NaN moved to the neighbouring row, an Inf with its sign flipped,
   one changed bit in a guard band, and the masked-lane defect of SpMM (0 * B(0, j) added for the slots past a row's end).
2. The same regimes and guard bands on the generic kernels' own source compiled for the host (tests/generic_emu.py): CSR,
   COO and Sliced-ELL, every instantiation, A and A^T; Sliced-ELL also with NaN stored in every padding slot.
"""
import ctypes as C

import generic_emu
import numpy as np
import pytest

from elementwise_check import (F64, GUARDS, SCALARS, assert_elementwise, bad_elements, bands_intact, cases, csr_of,
                               guarded, lens_to_csr, reference, row_bound, start_y, transpose_csr, values)
from oracle import oracle as O

# every row length mod 4, empty rows, rows longer than one 32-entry step
LENS = np.array([0, 1, 2, 3, 4, 5, 6, 7, 0, 31, 33, 34, 35, 64, 9, 10, 11, 0, 1, 2, 13, 45, 3, 70, 0, 8, 17, 18, 19])


def structure(seed=1, cols=97):
    off, col = lens_to_csr(LENS, cols, seed)
    return csr_of(off, col, np.ones(col.size), (LENS.size, cols))


def in_type(M, x, y0, alpha, beta, T, order):
    """y = alpha * (sum of M_ij x_j) + beta * y0 with every operation rounded to T, the row sums taken in `order`."""
    T = np.dtype(T).type
    out = np.empty(M.shape[0], T)
    with np.errstate(all="ignore"):
        for i in range(M.shape[0]):
            p = [T(v) * T(x[j]) for v, j in zip(M.data[M.indptr[i]:M.indptr[i + 1]], M.indices[M.indptr[i]:M.indptr[i + 1]])]
            if order == "reversed":
                s = T(0)
                for t in reversed(p):
                    s = T(s + t)
            else:                                   # pairwise
                while len(p) > 1:
                    p = [T(p[k] + p[k + 1]) if k + 1 < len(p) else p[k] for k in range(0, len(p), 2)]
                s = p[0] if p else T(0)
            out[i] = T(T(alpha) * s) if beta == 0 else T(T(T(alpha) * s) + T(T(beta) * T(y0[i])))
    return out


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("regime", ["cancel", "wide", "nonfinite"])
def test_comparator_accepts_every_correct_summation_order(dtype, regime):
    M0 = structure()
    for _, alpha, beta, val, x, y0, ref, bound in cases(M0, (M0.shape[1],), (M0.shape[0],), dtype, dtype, 5, regimes=(regime,)):
        M = csr_of(M0.indptr, M0.indices, val, M0.shape)
        with np.errstate(all="ignore"):
            scipy_y = alpha * (M @ x.astype(np.float64)) + (beta * y0.astype(np.float64) if beta != 0 else 0.0)
        oracle_y = O.spmv_csr(M0.indptr.astype(np.int32), M0.indices.astype(np.int32), val, x, start_y(y0, beta), alpha, beta)
        assert oracle_y.dtype == dtype
        for name, got in (("scipy", scipy_y.astype(dtype)), ("oracle", oracle_y),
                          ("reversed", in_type(M, x, y0, alpha, beta, dtype, "reversed")),
                          ("pairwise", in_type(M, x, y0, alpha, beta, dtype, "pairwise"))):
            assert_elementwise(got, ref, bound, f"{name} {regime} alpha={alpha} beta={beta}")
        if regime == "nonfinite":
            assert np.isnan(ref).any() and np.isinf(ref).any() and np.isfinite(ref[np.diff(M.indptr) > 0]).any()


def _case(regime, dtype=np.float64, beta_nonzero=True):
    M0 = structure()
    for _, alpha, beta, val, x, y0, ref, bound in cases(M0, (M0.shape[1],), (M0.shape[0],), dtype, dtype, 5, regimes=(regime,)):
        if (beta != 0) == beta_nonzero:
            return csr_of(M0.indptr, M0.indices, val, M0.shape), alpha, beta, x, y0, ref, bound


@pytest.mark.parametrize("regime", ["uniform", "cancel", "wide"])
def test_comparator_rejects_fp64_accumulated_in_fp32(regime):
    M, alpha, beta, x, y0, ref, bound = _case(regime)
    got = in_type(M, x, y0, alpha, beta, np.float32, "reversed")
    assert bad_elements(got, ref, bound).size > 0


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("regime", ["uniform", "cancel", "wide", "nonfinite"])
def test_comparator_rejects_one_row_moved_by_four_bounds(dtype, regime):
    M, alpha, beta, x, y0, ref, bound = _case(regime, dtype)
    i = int(np.flatnonzero(np.isfinite(ref) & (np.diff(M.indptr) > 0))[0])
    got = ref.copy()
    got[i] += 4 * bound[i]
    assert list(bad_elements(got, ref, bound)) == [i]
    got[i] = ref[i] + 0.9 * bound[i]
    assert bad_elements(got, ref, bound).size == 0


@pytest.mark.parametrize("beta_nonzero", [False, True])
def test_comparator_rejects_a_nan_moved_and_an_inf_flipped(beta_nonzero):
    M, alpha, beta, x, y0, ref, bound = _case("nonfinite", beta_nonzero=beta_nonzero)
    i = int(np.flatnonzero(np.isnan(ref[:-1]) & np.isfinite(ref[1:]))[0])
    got = ref.copy()
    got[i], got[i + 1] = ref[i + 1], np.nan
    assert list(bad_elements(got, ref, bound)) == [i, i + 1]
    k = int(np.flatnonzero(np.isinf(ref))[0])
    got = ref.copy()
    got[k] = -got[k]
    assert list(bad_elements(got, ref, bound)) == [k]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("G", GUARDS)
def test_guard_band_detects_one_changed_bit(dtype, G):
    y = np.arange(10, dtype=dtype)
    buf = guarded(y, G, "sentinel")
    assert np.array_equal(buf[G:G + 10], y) and bands_intact(buf, G, 10)
    for pos in (0, G - 1, G + 10, 2 * G + 9):
        b = buf.copy()
        bits = b.view(np.uint32 if dtype == np.float32 else np.uint64)
        bits[pos] ^= bits.dtype.type(1) << bits.dtype.type(7)
        assert not bands_intact(b, G, 10)


def spmm_row_emulation(M, B, skip_tail):
    """spmm_csr.cu's spmm_row restated in numpy: the row is walked in 32-entry batches, each in steps of 4 slots; a slot past
    the row's end carries c = 0, v = 0.  skip_tail=False adds v * B(0, j) for those slots (the defect), True skips them."""
    C_ = np.zeros((M.shape[0], B.shape[1]))
    with np.errstate(all="ignore"):
        for i in range(M.shape[0]):
            b, e = M.indptr[i], M.indptr[i + 1]
            acc = np.zeros(B.shape[1])
            for p in range(b, e, 32):
                cnt = min(32, e - p)
                for t in range(0, cnt, 4):
                    for u in range(4):
                        live = t + u < cnt
                        c, v = (M.indices[p + t + u], M.data[p + t + u]) if live else (0, 0.0)
                        if live or not skip_tail:
                            acc += v * B[c]
            C_[i] = acc
    return C_


def test_comparator_catches_the_spmm_tail_lane_defect():
    M0 = structure()
    M0 = csr_of(M0.indptr, M0.indices, np.ones(M0.nnz), M0.shape)
    n = 5
    lens = np.diff(M0.indptr)
    avoid0 = np.array([0 not in M0.indices[M0.indptr[i]:M0.indptr[i + 1]] for i in range(M0.shape[0])])
    assert np.any(avoid0 & (lens % 4 != 0))
    val, B, C0 = values("nonfinite", M0.nnz, (M0.shape[1], n), (M0.shape[0], n), np.float64, np.float64, 3)
    M = csr_of(M0.indptr, M0.indices, val, M0.shape)
    ref = reference(M, B, C0, 1.0, 0.0)
    bound = row_bound(M, B, C0, 1.0, 0.0, F64)
    assert_elementwise(spmm_row_emulation(M, B, skip_tail=True), ref, bound, "tail lanes skipped")
    bad = bad_elements(spmm_row_emulation(M, B, skip_tail=False), ref, bound)
    rows = np.unique(bad // n)
    assert rows.size and np.all(lens[rows] % 4 != 0)
    assert np.any(avoid0[rows])                      # rows that never reference column 0 go wrong too


def test_sell_oracle_skips_padding_whatever_its_value():
    M0 = structure()
    val = values("uniform", M0.nnz, (M0.shape[1],), (M0.shape[0],), F64, F64, 2)[0]
    x = values("uniform", 0, (M0.shape[1],), (M0.shape[0],), F64, F64, 4)[1]
    so, sc, sv = O.csr_to_sell(M0.indptr.astype(np.int32), M0.indices.astype(np.int32), val, 7)
    sv[sc < 0] = np.nan
    assert np.isnan(sv).any()
    M = csr_of(M0.indptr, M0.indices, val, M0.shape)
    assert_elementwise(O.spmv_sell(M.shape[0], 7, so, sc, sv, x), reference(M, x, x[:M.shape[0]], 1.0, 0.0),
                       row_bound(M, x, None, 1.0, 0.0, F64), "oracle, NaN padding")


# ------------------------------------------------------------------------------------------------------------------------------
# The generic kernels' own source on the host, every regime, both guard offsets
# ------------------------------------------------------------------------------------------------------------------------------
NPI = {0: np.int32, 1: np.int64}
NPF = {0: np.float32, 1: np.float64}
CTF = {0: C.c_float, 1: C.c_double}
COMBOS = [(0, 0, 0, 0), (0, 0, 0, 1), (0, 0, 1, 1), (1, 0, 0, 0), (1, 0, 0, 1), (1, 0, 1, 1), (1, 1, 0, 0), (1, 1, 0, 1), (1, 1, 1, 1)]
ROWS, COLS, BASE = 203, 150, 1          # partial last Sliced-ELL slice; base 1: the padding column is 0


@pytest.fixture(scope="module")
def emu():
    return generic_emu.load()


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def emu_structure(seed):
    off, col, _ = O.rmat_csr(ROWS, cols=COLS, avg_nnz=5, seed=seed, val_seed=seed + 1)
    return csr_of(off, col, np.ones(col.size), (ROWS, COLS))


def run_guarded(call, x, y0, beta, G, what):
    """call(xp, yp) on guarded x / y; returns y, and checks y's bands."""
    xb = guarded(x, G, np.nan)
    yb = guarded(start_y(y0, beta), G, "sentinel")
    assert call(_p(xb[G:]), _p(yb[G:])) == 0
    assert bands_intact(yb, G, y0.size), f"{what}: y guard band overwritten"
    return yb[G:G + y0.size]


def _check_all(M, transpose, a_dt, xy_dt, seed, launch, regimes=None):
    """launch(val, G, alpha, beta, xp, yp) runs one product on op(A) = M^T if transpose else M; val in M's storage order."""
    opM, perm = transpose_csr(M) if transpose else (M, None)
    kw = {} if regimes is None else dict(regimes=regimes)
    for regime, alpha, beta, val, x, y0, ref, bound in cases(opM, (opM.shape[1],), (opM.shape[0],), NPF[a_dt], NPF[xy_dt], seed, **kw):
        if transpose:                       # cases() draws the values in A^T's storage order
            val_a = np.empty_like(val)
            val_a[perm] = val
            val = val_a
        for G in GUARDS:
            what = f"{regime} alpha={alpha} beta={beta} G={G}"
            got = run_guarded(lambda xp, yp: launch(val, G, alpha, beta, xp, yp), x, y0, beta, G, what)
            assert_elementwise(got, ref, bound, what)


@pytest.mark.parametrize("off64,col64,a_dt,xy_dt", COMBOS)
@pytest.mark.parametrize("transpose", [0, 1])
def test_csr_generic_elementwise(emu, off64, col64, a_dt, xy_dt, transpose):
    M = emu_structure(40)
    ct = CTF[xy_dt]

    def launch(val, G, alpha, beta, xp, yp):
        o = (M.indptr + BASE).astype(NPI[off64])
        cb = guarded((M.indices + BASE).astype(NPI[col64]), G, BASE)
        vb = guarded(val, G, np.nan)
        lanes = 2 + (G + transpose) % 4
        return emu.emu_csr_generic(off64, col64, a_dt, xy_dt, transpose, lanes, 1, C.c_longlong(ROWS), C.c_longlong(COLS),
                                   C.c_longlong(M.nnz), _p(o), _p(cb[G:]), _p(vb[G:]), C.c_longlong(BASE), C.byref(ct(alpha)),
                                   C.byref(ct(beta)), xp, yp)
    _check_all(M, transpose, a_dt, xy_dt, 7, launch)


@pytest.mark.parametrize("idx64,a_dt,xy_dt", [(0, 0, 0), (0, 0, 1), (0, 1, 1), (1, 0, 0), (1, 0, 1), (1, 1, 1)])
@pytest.mark.parametrize("transpose", [0, 1])
def test_coo_generic_elementwise(emu, idx64, a_dt, xy_dt, transpose):
    """Entries in random order; A^T is the same kernel with the index arrays and the shape swapped (the shim's generic_mv)."""
    M = emu_structure(60)
    row = np.repeat(np.arange(ROWS), np.diff(M.indptr))
    perm = np.random.default_rng(1).permutation(M.nnz)
    ct = CTF[xy_dt]

    def launch(val, G, alpha, beta, xp, yp):
        r, c = (row[perm] + BASE).astype(NPI[idx64]), (M.indices[perm] + BASE).astype(NPI[idx64])
        rb, cb, vb = guarded(r, G, BASE), guarded(c, G, BASE), guarded(val[perm], G, np.nan)
        shape = (ROWS, COLS, rb, cb) if not transpose else (COLS, ROWS, cb, rb)
        return emu.emu_coo_generic(idx64, a_dt, xy_dt, 1, C.c_longlong(shape[0]), C.c_longlong(shape[1]), C.c_longlong(M.nnz),
                                   _p(shape[2][G:]), _p(shape[3][G:]), _p(vb[G:]), C.c_longlong(BASE), C.byref(ct(alpha)),
                                   C.byref(ct(beta)), xp, yp)
    _check_all(M, transpose, a_dt, xy_dt, 8, launch)


@pytest.mark.parametrize("off64,col64,a_dt,xy_dt", COMBOS)
@pytest.mark.parametrize("transpose,S", [(0, 32), (0, 7), (1, 32), (1, 2)])
@pytest.mark.parametrize("nan_padding", [False, True])
def test_sell_generic_elementwise(emu, off64, col64, a_dt, xy_dt, transpose, S, nan_padding):
    M = emu_structure(80 + S)
    ct = CTF[xy_dt]

    def launch(val, G, alpha, beta, xp, yp):
        so, sc, sv = O.csr_to_sell((M.indptr + BASE).astype(np.int32), (M.indices + BASE).astype(np.int32), val, S, base=BASE)
        if nan_padding:
            sv[sc == BASE - 1] = np.nan
        cb, vb = guarded(sc.astype(NPI[col64]), G, BASE), guarded(sv, G, np.nan)
        return emu.emu_sell_generic(off64, col64, a_dt, xy_dt, transpose, 1, C.c_longlong(ROWS), C.c_longlong(COLS), C.c_longlong(S),
                                    _p(so.astype(NPI[off64])), _p(cb[G:]), _p(vb[G:]), C.c_longlong(BASE), C.byref(ct(alpha)),
                                    C.byref(ct(beta)), xp, yp)
    _check_all(M, transpose, a_dt, xy_dt, 9, launch, regimes=("uniform", "nonfinite") if nan_padding else None)
