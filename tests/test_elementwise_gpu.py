"""Element-wise GPU checks (tests/elementwise_check.py) of every kernel that serves a cusparseSpMV / cusparseSpMM call: per-element
bound valid for any summation order, exact non-finite classification, guard bands around every operand (two offsets: a
multiple of 4 elements and an odd count), value regimes uniform / cancel / wide / nonfinite, plus NaN padding values for
Sliced-ELL.  Every call goes through the C ABI and must be served by our kernels (forwarded unchanged, native + 1); where the
closed library takes the input it runs on the same guarded buffers and meets the same comparator.  Matrices are small: the
oracle runs on the host.
"""
import numpy as np
import pytest
import torch

from elementwise_check import (EDGE, GUARDS, assert_elementwise, bad_elements, bands_intact, cases, csr_of, guarded, lens_to_csr, start_y,
                               transpose_csr)
from oracle import oracle as O

pytestmark = pytest.mark.gpu

SHAPES = ["single_huge_row", "huge_then_tiny", "alternating", "leading_empty", "trailing_empty", "all_empty",
          "many_rows_end_in_one_step", "rows_of_32", "tile_sized_rows", "one_by_one", "rmat_prime", "rmat_rect"]
EDGE_COLS = 120000
NPI = {32: np.int32, 64: np.int64}


@pytest.fixture(scope="module")
def cs():
    from cudalibrarysamples_b200 import cusparse_api
    return cusparse_api


@pytest.fixture(scope="module")
def b200(cs):
    return cs.Api("b200")


@pytest.fixture(scope="module")
def closed(cs):
    return cs.Api("cusparse")


@pytest.fixture(scope="module")
def handle(b200):
    """One cuSPARSE handle for every call (handles always belong to the closed library, for both implementations)."""
    h = b200.cusparseCreate()
    yield h
    b200.cusparseDestroy(h)


# base 0 with the guard offset that keeps 16-byte alignment, base 1 with the odd one
BASE_GUARD = ((0, GUARDS[0]), (1, GUARDS[1]))
# The closed library's COO kernel needs 16-byte-aligned index / value arrays (misaligned-address fault otherwise): it runs on the
# aligned guard offset only, and so does its Sliced-ELL kernel.
ALIGNED = GUARDS[0]
_SHAPE_CACHE = {}


def shape(name):
    """The matrix structure of a case as CSR (values replaced per regime)."""
    if name not in _SHAPE_CACHE:
        if name == "rmat_prime":                    # prime row count: no slice, tile or warp count divides it
            off, col, _ = O.rmat_csr(20011, avg_nnz=12, seed=301, val_seed=302)
            rows, cols = 20011, 20011
        elif name == "rmat_rect":
            rows, cols = 9001, 4099
            off, col, _ = O.rmat_csr(rows, cols=cols, avg_nnz=9, seed=303, val_seed=304)
        else:
            lens = EDGE[name]
            rows, cols = lens.size, EDGE_COLS
            off, col = lens_to_csr(lens, cols, 3)
        _SHAPE_CACHE[name] = csr_of(off, col, np.ones(col.size), (rows, cols))
    return _SHAPE_CACHE[name]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def counted(api, fn):
    """fn() with our library's call counters checked: our kernels served it (nothing forwarded)."""
    before = api.stats() if api.impl == "b200" else None
    out = fn()
    if before is not None:
        after = api.stats()
        assert after["forwarded"] == before["forwarded"], "the call was forwarded to the closed library"
        assert after["native"] == before["native"] + 1
    return out


def spmv_guarded(cs, api, h, fmt, rows, cols, arrays, x, y0, alpha, beta, base, G, transpose=False, xy_dtype=None, preprocess=True):
    """One cusparseSpMV with x / y as views at offset G into guarded buffers (x: NaN bands, y: sentinel bands); `arrays`
    holds device views into guarded index / value buffers.  Returns y (host) after checking y's bands."""
    xb, yb = dev(guarded(x, G, np.nan)), dev(guarded(start_y(y0, beta), G, "sentinel"))
    xv, yv = xb[G:G + x.size], yb[G:G + y0.size]
    op = cs.SpMVOperator(api, fmt, rows, cols, arrays, base=base, preprocess=preprocess, xy_dtype=xy_dtype, handle=h,
                         op=cs.CUSPARSE_OPERATION_TRANSPOSE if transpose else cs.CUSPARSE_OPERATION_NON_TRANSPOSE)

    def call():
        op(xv, yv, alpha, beta)
        torch.cuda.synchronize()
    try:
        counted(api, call)
    finally:
        op.close()
    out = yb.cpu().numpy()
    assert bands_intact(out, G, y0.size), "y guard band overwritten"
    return out[G:G + y0.size]


def guarded_dev(a, G, band):
    return dev(guarded(a, G, band))[G:G + a.size]


def csr_arrays(M, val, base, G, off_bits=32, col_bits=32):
    return dict(off=dev((M.indptr + base).astype(NPI[off_bits])), col=guarded_dev((M.indices + base).astype(NPI[col_bits]), G, base),
                val=guarded_dev(val, G, np.nan))


def each_case(M, transpose, a_dt, xy_dt, seed, regimes=None):
    """(regime, alpha, beta, A's values in M's storage order, x, y0, ref, bound) for op(A) = M^T if transpose else M."""
    opM, perm = transpose_csr(M) if transpose else (M, None)
    kw = {} if regimes is None else dict(regimes=regimes)
    for regime, alpha, beta, val, x, y0, ref, bound in cases(opM, (opM.shape[1],), (opM.shape[0],), a_dt, xy_dt, seed, **kw):
        if transpose:
            val_a = np.empty_like(val)
            val_a[perm] = val
            val = val_a
        yield regime, alpha, beta, val, x, y0, ref, bound


# ------------------------------------------------------------------------------------------------------------------ CSR
@pytest.fixture(params=["tile", "pipe", "ws", "rowwise", "seg", "seg:1", "seg:1000000", "flat", "short"])
def csr_kernel(request, b200):
    """Every CSR kernel variant (as in test_parity_gpu.py): "seg:N" = csr_seg_kernel with the row-sparse threshold N, "flat" /
    "short" = csr_flat_kernel / csr_short_kernel forced for every preprocessed matrix."""
    name, _, dense = request.param.partition(":")
    b200.set_option("B200SPMV_FLAT", "on" if name == "flat" else "off")
    b200.set_option("B200SPMV_SHORT", "on" if name == "short" else "off")
    b200.set_option("B200SPMV_CSR_KERNEL", "auto" if name in ("flat", "short") else name)
    b200.set_option("B200SPMV_SEG_DENSE", dense or "24")
    yield request.param
    b200.set_option("B200SPMV_CSR_KERNEL", "auto")
    b200.set_option("B200SPMV_SEG_DENSE", "24")
    b200.set_option("B200SPMV_FLAT", "auto")
    b200.set_option("B200SPMV_SHORT", "auto")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", SHAPES)
def test_csr_variants_elementwise(cs, b200, handle, csr_kernel, name, dtype):
    M = shape(name)
    for regime, alpha, beta, val, x, y0, ref, bound in each_case(M, False, dtype, dtype, 11):
        for base, G in BASE_GUARD:
            arrays = csr_arrays(M, val, base, G)
            for pre in (True, False):
                got = spmv_guarded(cs, b200, handle, "csr", *M.shape, arrays, x, y0, alpha, beta, base, G, preprocess=pre)
                assert_elementwise(got, ref, bound, f"{csr_kernel} {regime} a={alpha} b={beta} base={base} G={G} pre={pre}")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", SHAPES)
def test_csr_closed_library_elementwise(cs, handle, closed, name, dtype):
    """The closed library on the same guarded buffers, same comparator (as a check of the checks)."""
    M = shape(name)
    if M.nnz == 0:
        pytest.skip("no non-zeros")
    for regime, alpha, beta, val, x, y0, ref, bound in each_case(M, False, dtype, dtype, 11):
        for base, G in BASE_GUARD:
            got = spmv_guarded(cs, closed, handle, "csr", *M.shape, csr_arrays(M, val, base, G), x, y0, alpha, beta, base, G)
            assert_elementwise(got, ref, bound, f"closed {regime} a={alpha} b={beta} base={base} G={G}")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("base", [0, 1])
@pytest.mark.parametrize("name", SHAPES)
def test_csr_transpose_elementwise(cs, b200, closed, handle, name, base, dtype):
    """csr_transpose_kernel (opA = TRANSPOSE, y[cols] = alpha * A^T x[rows] + beta * y)."""
    M = shape(name)
    for regime, alpha, beta, val, x, y0, ref, bound in each_case(M, True, dtype, dtype, 12):
        for G in GUARDS:
            arrays = csr_arrays(M, val, base, G)
            got = spmv_guarded(cs, b200, handle, "csr", *M.shape, arrays, x, y0, alpha, beta, base, G, transpose=True)
            assert_elementwise(got, ref, bound, f"{regime} a={alpha} b={beta} G={G}")
            if M.nnz and G == GUARDS[base]:
                got = spmv_guarded(cs, closed, handle, "csr", *M.shape, arrays, x, y0, alpha, beta, base, G, transpose=True)
                assert_elementwise(got, ref, bound, f"closed {regime} a={alpha} b={beta} G={G}")


# ------------------------------------------------------------------------------------------------------------------ COO
@pytest.fixture(params=["tile", "seg"])
def coo_kernel(request, b200):
    b200.set_option("B200SPMV_COO_KERNEL", request.param)
    yield request.param
    b200.set_option("B200SPMV_COO_KERNEL", "auto")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("name", SHAPES)
def test_coo_elementwise(cs, b200, closed, handle, coo_kernel, name, transpose, dtype):
    """coo_tile_kernel (both sides of its 16-byte vec_ok test: the odd guard offset misaligns row / col / val) and
    coo_seg_kernel; row-sorted entries; A and A^T."""
    M = shape(name)
    row = np.repeat(np.arange(M.shape[0]), np.diff(M.indptr))
    for regime, alpha, beta, val, x, y0, ref, bound in each_case(M, transpose, dtype, dtype, 13):
        for base, G in BASE_GUARD:
            arrays = dict(row=guarded_dev((row + base).astype(np.int32), G, base),
                          col=guarded_dev((M.indices + base).astype(np.int32), G, base), val=guarded_dev(val, G, np.nan))
            what = f"{coo_kernel} {regime} a={alpha} b={beta} base={base} G={G}"
            got = spmv_guarded(cs, b200, handle, "coo", *M.shape, arrays, x, y0, alpha, beta, base, G, transpose=transpose)
            assert_elementwise(got, ref, bound, what)
            if coo_kernel == "tile" and M.nnz and G == ALIGNED:
                got = spmv_guarded(cs, closed, handle, "coo", *M.shape, arrays, x, y0, alpha, beta, base, G, transpose=transpose)
                assert_elementwise(got, ref, bound, "closed " + what)


# ------------------------------------------------------------------------------------------------------------------ Sliced-ELL
SELL_SHAPES = [s for s in SHAPES if s != "single_huge_row"]      # one 100000-entry row pads a 64-row slice to 6.4 M slots


def sell_case(M, val, S, base, G, nan_padding):
    so, sc, sv = O.csr_to_sell((M.indptr + base).astype(np.int32), (M.indices + base).astype(np.int32), val, S, base=base)
    if nan_padding:
        sv[sc == base - 1] = np.nan
    return dict(off=dev(so), col=guarded_dev(sc, G, base), val=guarded_dev(sv, G, np.nan), slice_size=S, nnz=M.nnz), sv


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("S,kernel", [(1, "sell_row"), (7, "sell_row"), (32, "sell32"), (32, "sell_row"), (33, "sell_row"),
                                      (64, "sell_row")])
@pytest.mark.parametrize("name", SELL_SHAPES)
def test_sell_elementwise(cs, b200, closed, handle, request, name, S, kernel, dtype):
    """Sliced-ELL, base 0 and 1, every regime plus `nan_padding` (every padding slot holds NaN: padding is marked by its column
    index, so its stored value must not matter -- the oracle and the generic kernel skip it).  The closed library's results on
    NaN padding and in the nonfinite regime are recorded in the test report, not asserted: it returns NaN where the oracle has
    +-Inf for a few rows of the rectangular matrix."""
    b200.set_option("B200SPMV_SELL_GENERIC", "1" if kernel == "sell_row" and S == 32 else "0")
    try:
        M = shape(name)
        seen = []
        for regime, alpha, beta, val, x, y0, ref, bound in each_case(M, False, dtype, dtype, 14, regimes=("uniform", "cancel", "wide",
                                                                                                          "nonfinite", "nan_padding")):
            for base, G in BASE_GUARD:
                arrays, sv = sell_case(M, val, S, base, G, regime == "nan_padding")
                what = f"{kernel} S={S} {regime} a={alpha} b={beta} base={base} G={G}"
                got = spmv_guarded(cs, b200, handle, "sell", *M.shape, arrays, x, y0, alpha, beta, base, G)
                assert_elementwise(got, ref, bound, what)
                if kernel == "sell_row" and M.nnz and G == ALIGNED:
                    lib = spmv_guarded(cs, closed, handle, "sell", *M.shape, arrays, x, y0, alpha, beta, base, G)
                    if regime in ("nan_padding", "nonfinite"):
                        seen.append(f"{what}: closed library {int(bad_elements(lib, ref, bound).size)} elements off the oracle, NaN in {int(np.count_nonzero(np.isnan(lib)))} of {lib.size} rows "
                                    f"(oracle: {int(np.count_nonzero(np.isnan(ref)))}; {int(np.count_nonzero(np.isnan(sv)))} padding slots)")
                    else:
                        assert_elementwise(lib, ref, bound, "closed " + what)
        if seen:
            request.node.user_properties.append(("closed_library_nan_padding", seen))
            print("\n".join(seen))
    finally:
        b200.set_option("B200SPMV_SELL_GENERIC", "0")


# ------------------------------------------------------------------------------------------------------------------ generic CSR
CSR_GENERIC = [(o, c, t) for (o, c) in ((64, 64), (64, 32)) for t in ("f64", "f32", "f32_f64")] + [(32, 32, "f32_f64")]
TYPES = {"f64": (np.float64, torch.float64), "f32": (np.float32, torch.float32), "f32_f64": (np.float32, torch.float64)}


@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("off_bits,col_bits,types", CSR_GENERIC)
@pytest.mark.parametrize("name", ["huge_then_tiny", "many_rows_end_in_one_step", "alternating", "leading_empty", "one_by_one",
                                  "rmat_prime", "rmat_rect"])
def test_csr_generic_elementwise(cs, b200, closed, handle, name, off_bits, col_bits, types, transpose):
    """csr_generic_kernel / csr_generic_transpose_kernel (64-bit indices, fp32 A with fp64 x / y), base 1."""
    b200.set_option("B200SPMV_GENERIC", "csr")      # the library default
    a_dt, xy = TYPES[types]
    xy_dt = np.float64 if xy == torch.float64 else np.float32
    M = shape(name)
    for regime, alpha, beta, val, x, y0, ref, bound in each_case(M, transpose, a_dt, xy_dt, 15):
        for G in GUARDS:
            arrays = csr_arrays(M, val, 1, G, off_bits, col_bits)
            what = f"{regime} a={alpha} b={beta} G={G}"
            try:
                got = spmv_guarded(cs, b200, handle, "csr", *M.shape, arrays, x, y0, alpha, beta, 1, G, transpose=transpose, xy_dtype=xy)
            except cs.CuSparseError as e:
                # 64-bit offsets with 32-bit columns: the closed library refuses the descriptor, and the shim keeps its verdict
                with pytest.raises(cs.CuSparseError) as theirs:
                    spmv_guarded(cs, closed, handle, "csr", *M.shape, arrays, x, y0, alpha, beta, 1, G, transpose=transpose, xy_dtype=xy)
                assert theirs.value.status == e.status
                continue
            assert_elementwise(got, ref, bound, what)
            if M.nnz and G == ALIGNED:
                try:
                    lib = spmv_guarded(cs, closed, handle, "csr", *M.shape, arrays, x, y0, alpha, beta, 1, G, transpose=transpose, xy_dtype=xy)
                except cs.CuSparseError:            # not a combination the closed library takes
                    continue
                assert_elementwise(lib, ref, bound, "closed " + what)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", ["huge_then_tiny", "alternating", "rmat_prime"])
def test_csr_without_a_buffer_elementwise(cs, b200, name, dtype):
    """externalBuffer = NULL: the plan-free csr_generic_kernel serves the call."""
    M = shape(name)
    for regime, alpha, beta, val, x, y0, ref, bound in each_case(M, False, dtype, dtype, 16):
        for G in GUARDS:
            arrays = csr_arrays(M, val, 0, G)
            xb, yb = dev(guarded(x, G, np.nan)), dev(guarded(start_y(y0, beta), G, "sentinel"))
            h = b200.cusparseCreate()
            m = b200.cusparseCreateCsr(*M.shape, M.nnz, arrays["off"], arrays["col"], arrays["val"])
            vx, vy = b200.cusparseCreateDnVec(x.size, xb[G:G + x.size]), b200.cusparseCreateDnVec(y0.size, yb[G:G + y0.size])
            ct = cs.CUDA_R_64F if dtype == np.float64 else cs.CUDA_R_32F

            def call():
                b200.cusparseSpMV(h, cs.CUSPARSE_OPERATION_NON_TRANSPOSE, alpha, m, vx, beta, vy, ct, 0, None)
                torch.cuda.synchronize()
            try:
                counted(b200, call)
                assert "csr_generic_kernel" in b200.last_csr_kernel()
            finally:
                b200.cusparseDestroySpMat(m); b200.cusparseDestroyDnVec(vx); b200.cusparseDestroyDnVec(vy); b200.cusparseDestroy(h)
            out = yb.cpu().numpy()
            assert bands_intact(out, G, y0.size)
            assert_elementwise(out[G:G + y0.size], ref, bound, f"{regime} a={alpha} b={beta} G={G}")


# ------------------------------------------------------------------------------------------------------------------ SpMM
# every row length mod 4, rows that avoid column 0, empty rows, rows longer than one 32-entry batch
SPMM_LENS = np.concatenate([[0, 1, 2, 3, 4, 5, 6, 7, 0, 31, 33, 34, 35, 64, 9, 10, 11], np.tile([1, 2, 3, 4, 13, 45, 70, 0], 40)])


def spmm_guarded(cs, api, M, val, B, C0, alpha, beta, order_b, order_c, G):
    """cuSPARSE's SpMM call sequence (spmm_csr_example.c:86-132) with B / C as views at offset G into guarded buffers (B: NaN
    bands, C: sentinel bands).  Returns C (host, 2-D)."""
    rows, cols = M.shape
    n = B.shape[1]
    lay = lambda a, o: (np.ascontiguousarray(a) if o == cs.CUSPARSE_ORDER_ROW else np.asfortranarray(a)).ravel(order="K")
    Bb = dev(guarded(lay(B, order_b), G, np.nan))
    Cb = dev(guarded(lay(start_y(C0, beta), order_c), G, "sentinel"))
    arrays = csr_arrays(M, val, 0, G)
    ct = cs.CUDA_R_64F if val.dtype == np.float64 else cs.CUDA_R_32F
    h = api.cusparseCreate()
    matA = api.cusparseCreateCsr(rows, cols, M.nnz, arrays["off"], arrays["col"], arrays["val"])
    matB = api.cusparseCreateDnMat(cols, n, cols if order_b == cs.CUSPARSE_ORDER_COL else n, Bb[G:G + B.size], order_b)
    matC = api.cusparseCreateDnMat(rows, n, rows if order_c == cs.CUSPARSE_ORDER_COL else n, Cb[G:G + C0.size], order_c)
    op = cs.CUSPARSE_OPERATION_NON_TRANSPOSE
    try:
        size = api.cusparseSpMM_bufferSize(h, op, op, alpha, matA, matB, beta, matC, ct)
        buf = torch.empty(max(size, 16), dtype=torch.uint8, device="cuda")
        api.cusparseSpMM_preprocess(h, op, op, alpha, matA, matB, beta, matC, ct, cs.CUSPARSE_SPMM_ALG_DEFAULT, buf)

        def call():
            api.cusparseSpMM(h, op, op, alpha, matA, matB, beta, matC, ct, cs.CUSPARSE_SPMM_ALG_DEFAULT, buf)
            torch.cuda.synchronize()
        counted(api, call)
    finally:
        api.cusparseDestroySpMat(matA); api.cusparseDestroyDnMat(matB); api.cusparseDestroyDnMat(matC); api.cusparseDestroy(h)
    out = Cb.cpu().numpy()
    assert bands_intact(out, G, C0.size), "C guard band overwritten"
    return out[G:G + C0.size].reshape((rows, n), order="C" if order_c == cs.CUSPARSE_ORDER_ROW else "F")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("n", [1, 3, 4, 5, 64, 67])
@pytest.mark.parametrize("order_b,order_c", [(1, 1), (2, 2), (2, 1), (1, 2)])
def test_spmm_elementwise(cs, b200, closed, order_b, order_c, n, dtype):
    """spmm_csr_kernel / spmm_csr_ctile_kernel (with column-major B transposed into the buffer for n >= 4, walked in place
    below).  In the nonfinite regime row 0 of B holds NaN / +Inf / -Inf: rows that never reference column 0 must stay finite,
    whatever their length mod 4."""
    cols = 900
    off, col = lens_to_csr(SPMM_LENS, cols, 21)
    M = csr_of(off, col, np.ones(col.size), (SPMM_LENS.size, cols))
    avoid0 = np.array([0 not in col[off[i]:off[i + 1]] for i in range(M.shape[0])])
    assert np.all([np.any(avoid0 & (SPMM_LENS % 4 == r)) for r in range(4)])
    for regime, alpha, beta, val, B, C0, ref, bound in cases(M, (cols, n), (M.shape[0], n), dtype, dtype, 17):
        for G in GUARDS:
            what = f"order_b={order_b} order_c={order_c} n={n} {regime} a={alpha} b={beta} G={G}"
            got = spmm_guarded(cs, b200, M, val, B, C0, alpha, beta, order_b, order_c, G)
            assert_elementwise(got, ref, bound, what)
            if order_b == order_c and G == ALIGNED:    # the closed library wants B and C in the same order
                lib = spmm_guarded(cs, closed, M, val, B, C0, alpha, beta, order_b, order_c, G)
                assert_elementwise(lib, ref, bound, "closed " + what)
