"""GPU parity tests: the sm_100a path, called through the C ABI (the cusparse* symbols exported by libb200spmv.so),
against (i) the reference's golden vectors, (ii) the CPU oracle, (iii) the closed cusparseSpMV on the same device
buffers, and (iv) size-independent properties at BASELINE.json's full sizes.

Tolerances (north_star): fp64 ||y - y_ref|| / ||y_ref|| < 1e-12, fp32 < 1e-5; integer preprocessing bit-exact.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import oracle as O
from oracle.partition_ref import check_partition, csr_partition

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {torch.float64: 1e-12, torch.float32: 1e-5}
NP = {torch.float64: np.float64, torch.float32: np.float32}


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


def dev(a):
    return torch.as_tensor(a).cuda()


def relerr(got, want):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    n = np.linalg.norm(want)
    return np.linalg.norm(got - want) / (n if n > 0 else 1.0)


def run(cs, api, fmt, rows, cols, arrays, x, y0, alpha, beta, base=0, preprocess=True, expect_forward=False):
    """One cusparseSpMV through the C ABI.  For the b200 library the call counters must show that OUR kernel served it
    (b200spmv_get_stats: forwarded == 0) -- a silent hand-over to the closed library would void the parity claim."""
    before = api.stats() if api.impl == "b200" else None
    op = cs.SpMVOperator(api, fmt, rows, cols, arrays, base=base, preprocess=preprocess)
    y = y0.clone()
    op(x, y, alpha, beta)
    torch.cuda.synchronize()
    op.close()
    if before is not None:
        after = api.stats()
        if expect_forward:
            assert after["forwarded"] == before["forwarded"] + 1 and after["native"] == before["native"]
        else:
            assert after["forwarded"] == before["forwarded"], "the call was forwarded to the closed library"
            assert after["native"] == before["native"] + 1
    return y


# ------------------------------------------------------------------------------------------ goldens
def toy_arrays(fmt):
    T = O.TOY
    if fmt == "csr":
        return dict(off=dev(T["csr_off"]), col=dev(T["csr_col"]), val=dev(T["val"]))
    if fmt == "coo":
        return dict(row=dev(T["coo_row"]), col=dev(T["csr_col"]), val=dev(T["val"]))
    return dict(off=dev(T["sell_off"]), col=dev(T["sell_col"]), val=dev(T["sell_val"]), slice_size=2, nnz=9)


@pytest.mark.parametrize("fmt", ["csr", "coo", "sell"])
@pytest.mark.parametrize("preprocess", [True, False])
def test_toy_golden_exact(cs, b200, fmt, preprocess):
    # spmv_csr_example.c:54,123-129 / spmv_coo_example.c:54 / spmv_sell_example.c:69 -- exact `!=` compare
    y = run(cs, b200, fmt, 4, 4, toy_arrays(fmt), dev(O.TOY["x"]), torch.zeros(4, device="cuda"), 1.0, 0.0,
            preprocess=preprocess)
    assert np.array_equal(y.cpu().numpy(), O.TOY["y_result"])


def test_spmvop_alpha_beta_golden(cs, b200):
    # spmv_csr_op_example.c:169-173,288-289,307-326: fp64, alpha 1, beta 3, tol 1e-14
    T = O.TOY
    arrays = dict(off=dev(T["csr_off"]), col=dev(T["csr_col"]), val=dev(T["val"].astype(np.float64)))
    y = run(cs, b200, "csr", 4, 4, arrays, dev(T["x"].astype(np.float64)), dev(np.array([5.0, 6, 7, 8])), 1.0, 3.0)
    assert np.max(np.abs(y.cpu().numpy() - np.array([34.0, 26, 72, 76]))) <= 1e-14


@pytest.mark.parametrize("name", ["spmv_csr", "spmv_coo", "spmv_sell"])
def test_reference_sample_passes_through_the_shim(name):
    """The unmodified reference sample, linked -lb200spmv -lcusparse (oracle/Makefile), must print PASSED."""
    exe = os.path.join(ROOT, "oracle", "_ref", f"{name}_example.b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref not built")
    p = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=clean_env(B200SPMV_LOG="1"))
    assert p.returncode == 0, p.stdout + p.stderr
    assert f"{name}_example test PASSED" in p.stdout
    assert "[b200spmv] SpMV" in p.stderr and "forwarded" not in p.stderr   # our kernel ran, not the closed one


def clean_env(**extra):
    """Environment for the C sample binaries: they must dlopen the libcusparse they are linked against, not the one
    this Python process picked (cudalibrarysamples_b200.lib sets B200SPMV_CUSPARSE for in-process use)."""
    env = {k: v for k, v in os.environ.items() if k != "B200SPMV_CUSPARSE"}
    env.update(extra)
    return env


def _trace(out):
    return [l for l in out.splitlines() if "rror" in l or "teration" in l]


@pytest.mark.parametrize("name,iters", [("cg", 39), ("bicgstab", 13)])
def test_solver_samples_reproduce_the_readme_trace(name, iters):
    """cuSPARSE/cg/README.md:78-99 (39 iterations, final 4.39e-07) and bicgstab/README.md:77-93 (13 iterations):
    the samples only print; the shim-linked binary must converge like the closed library does.  What the closed library
    printed is stored in tests/golden/<name>_example.cusparse.out (the same sample linked against the closed cuSPARSE of
    CUDA 12.9, run on one B200)."""
    ours = os.path.join(ROOT, "oracle", "_ref", f"{name}_example.b200")
    if not os.path.exists(ours):
        pytest.skip("oracle/_ref not built")
    a = subprocess.run([ours], capture_output=True, text=True, timeout=300, env=clean_env())
    theirs = open(os.path.join(ROOT, "tests", "golden", f"{name}_example.cusparse.out")).read()
    assert a.returncode == 0, a.stdout[-2000:] + a.stderr[-2000:]
    ta, tb = _trace(a.stdout), _trace(theirs)
    na = sum("teration =" in l or "=== ITERATION" in l.upper() for l in ta)
    nb = sum("teration =" in l or "=== ITERATION" in l.upper() for l in tb)
    assert na == nb == iters, (na, nb, ta[-3:], tb[-3:])
    # final residual lines agree to the printed precision's leading digits
    fa = [l for l in a.stdout.splitlines() if "Final error norm" in l]
    fb = [l for l in theirs.splitlines() if "Final error norm" in l]
    assert fa and fb
    va, vb = float(fa[0].split("=")[-1]), float(fb[0].split("=")[-1])
    assert abs(va - vb) <= 0.1 * abs(vb) + 1e-12, (fa, fb)


# ---------------------------------------------------------------------------- oracle + closed library
_RMAT_CACHE = {}


def rmat_case(rows, avg, dtype, seed):
    key = (rows, avg, dtype, seed)
    if key not in _RMAT_CACHE:
        off, col, val = O.rmat_csr(rows, avg_nnz=avg, seed=seed, val_seed=seed + 1, dtype=NP[dtype])
        x = O.uniform(seed + 2, rows, NP[dtype])
        y0 = O.uniform(seed + 3, rows, NP[dtype])
        _RMAT_CACHE[key] = (off, col, val, x, y0)
    return _RMAT_CACHE[key]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("alpha,beta", [(1.0, 0.0), (-1.0, 1.0), (0.75, 0.0), (2.5, -0.5)])
def test_csr_rmat_vs_oracle_and_cusparse(cs, b200, closed, dtype, alpha, beta):
    rows = 60000
    off, col, val, x, y0 = rmat_case(rows, 16, dtype, 21)
    assert np.diff(off).max() >= 2048, "case must contain rows that get split between tiles"
    want = O.spmv_csr(off, col, val, x, y0, alpha, beta)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    got = run(cs, b200, "csr", rows, rows, arrays, dev(x), dev(y0), alpha, beta)
    lib = run(cs, closed, "csr", rows, rows, arrays, dev(x), dev(y0), alpha, beta)
    assert relerr(got.cpu().numpy(), want) < TOL[dtype]
    assert relerr(got.cpu().numpy(), lib.cpu().numpy()) < TOL[dtype]
    # bit-reproducible: same plan, same summation order
    again = run(cs, b200, "csr", rows, rows, arrays, dev(x), dev(y0), alpha, beta)
    assert torch.equal(got, again)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_csr_without_preprocess_and_buffer_reuse(cs, b200, dtype):
    """cg_example.c:409-418 -> 156-160,220-224: no _preprocess call, one buffer, different x / y / alpha / beta."""
    rows = 30000
    off, col, val, x, y0 = rmat_case(rows, 8, dtype, 31)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    op = cs.SpMVOperator(b200, "csr", rows, rows, arrays, preprocess=False)
    for (alpha, beta, sx) in [(0.75, 0.0, 1), (-1.0, 1.0, 2), (1.0, 0.0, 3)]:
        xs = O.uniform(100 + sx, rows, NP[dtype])
        y = dev(y0)
        op(dev(xs), y, alpha, beta)
        torch.cuda.synchronize()
        assert relerr(y.cpu().numpy(), O.spmv_csr(off, col, val, xs, y0, alpha, beta)) < TOL[dtype]
    op.close()


def test_plan_is_trusted_only_after_preprocess(cs, b200):
    """Without cusparseSpMV_preprocess the external buffer is plain scratch (the caller may share it with SpSV / SpMM or
    get the address back from a caching allocator with other contents): the plan must be rebuilt on every call.  After
    preprocess the buffer is the caller's promise, and no further analysis runs."""
    rows = 30000
    off, col, val, x, y0 = rmat_case(rows, 8, torch.float64, 31)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    want = O.spmv_csr(off, col, val, x, y0, 1.0, 0.0)
    op = cs.SpMVOperator(b200, "csr", rows, rows, arrays, preprocess=False)
    a0 = b200.stats()["analyze"]
    for _ in range(3):
        op.buffer.fill_(0xA5)                      # somebody else used the scratch buffer in between
        y = dev(y0)
        op(dev(x), y, 1.0, 0.0)
        torch.cuda.synchronize()
        assert relerr(y.cpu().numpy(), want) < 1e-12
    assert b200.stats()["analyze"] == a0 + 3
    op.close()
    op = cs.SpMVOperator(b200, "csr", rows, rows, arrays, preprocess=True)
    a1 = b200.stats()["analyze"]
    for _ in range(3):
        y = dev(y0)
        op(dev(x), y, 1.0, 0.0)
    torch.cuda.synchronize()
    assert relerr(y.cpu().numpy(), want) < 1e-12
    assert b200.stats()["analyze"] == a1
    op.close()


def test_csr_in_place_residual_update(cs, b200):
    # cg_example.c:153-160: R = B; R = -A*X + R with y aliased in/out
    off, col, val = O.gen_stencil5(150)
    n = 150 * 150
    x = O.uniform(5, n)
    b = O.spmv_csr(off, col, val, np.ones(n), alpha=0.75)
    want = O.spmv_csr(off, col, val, x, b, -1.0, 1.0)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    got = run(cs, b200, "csr", n, n, arrays, dev(x), dev(b), -1.0, 1.0, preprocess=False)
    assert relerr(got.cpu().numpy(), want) < 1e-13


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_csr_base_one(cs, b200, closed, dtype):
    # cuSOLVERSp2cuDSS/csreigvsi2cuDSS_double.cpp:139-141,319 creates base-1 CSR descriptors
    rows = 20000
    off, col, val, x, y0 = rmat_case(rows, 12, dtype, 41)
    arrays = dict(off=dev(off + 1), col=dev(col + 1), val=dev(val))
    want = O.spmv_csr(off, col, val, x, y0, 1.5, 0.25)
    got = run(cs, b200, "csr", rows, rows, arrays, dev(x), dev(y0), 1.5, 0.25, base=1)
    lib = run(cs, closed, "csr", rows, rows, arrays, dev(x), dev(y0), 1.5, 0.25, base=1)
    assert relerr(got.cpu().numpy(), want) < TOL[dtype]
    assert relerr(got.cpu().numpy(), lib.cpu().numpy()) < TOL[dtype]


@pytest.fixture(params=["tile", "pipe", "ws", "rowwise", "seg", "seg:1", "seg:1000000", "flat", "short"])
def csr_kernel(request, b200):
    """Every CSR kernel variant of the library must give the same answers (b200spmv_set_option picks one).
    "seg:N" = csr_seg_kernel with the row-sparse threshold N: 1 sends every tile that has non-zeros down the register
    path (multi-row steps, > 32 row ends per step), 1000000 sends every tile down the staged-product path.
    "flat" = csr_flat_kernel on the preprocess-built flat plan, forced for every matrix with non-zeros (calls without
    cusparseSpMV_preprocess still take the tile kernels: the flat plan is only ever built by preprocess).
    "short" = csr_short_kernel (a warp per 32 rows) forced for every preprocessed matrix, whatever its row lengths: rows
    longer than the warp's product buffer go through its multi-pass path."""
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


@pytest.fixture(params=["tile", "seg"])
def coo_kernel(request, b200):
    b200.set_option("B200SPMV_COO_KERNEL", request.param)
    yield request.param
    b200.set_option("B200SPMV_COO_KERNEL", "auto")


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_every_csr_kernel_variant(cs, b200, csr_kernel, dtype):
    rows = 50000
    off, col, val, x, y0 = rmat_case(rows, 16, dtype, 121)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    for alpha, beta in [(1.0, 0.0), (-1.0, 1.0)]:
        want = O.spmv_csr(off, col, val, x, y0, alpha, beta)
        got = run(cs, b200, "csr", rows, rows, arrays, dev(x), dev(y0), alpha, beta)
        assert relerr(got.cpu().numpy(), want) < TOL[dtype], (csr_kernel, alpha, beta)
        again = run(cs, b200, "csr", rows, rows, arrays, dev(x), dev(y0), alpha, beta)
        assert torch.equal(got, again)
    # short rows + base 1 + no preprocess
    off, col, val = O.gen_stencil5(200)
    n = 200 * 200
    xs, ys = O.uniform(5, n), O.uniform(6, n)
    arrays = dict(off=dev(off + 1), col=dev(col + 1), val=dev(val))
    got = run(cs, b200, "csr", n, n, arrays, dev(xs), dev(ys), 0.75, 0.5, base=1, preprocess=False)
    assert relerr(got.cpu().numpy(), O.spmv_csr(off, col, val, xs, ys, 0.75, 0.5)) < 1e-12


@pytest.mark.parametrize("name", ["single_huge_row", "huge_then_tiny", "alternating", "all_empty", "trailing_empty", "leading_empty",
                                  "rmat_like_block", "many_rows_end_in_one_step", "rows_of_32", "tile_sized_rows", "exactly_long"])
def test_every_csr_kernel_variant_edge_profiles(cs, b200, csr_kernel, name):
    lens = EDGE[name]
    rows, cols = lens.size, 120000
    off, col, val = lens_to_csr(lens, cols, 3)
    x, y0 = O.uniform(1, cols), O.uniform(2, rows)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    want = O.spmv_csr(off, col, val, x, y0, -2.0, 0.5)
    got = run(cs, b200, "csr", rows, cols, arrays, dev(x), dev(y0), -2.0, 0.5).cpu().numpy()
    assert relerr(got, want) < 1e-12, (csr_kernel, name)


_CSR_CACHE = {}


def lens_to_csr(lens, cols, seed, dtype=np.float64):
    """Random CSR with the given row lengths (distinct sorted columns per row); cached: several tests share profiles."""
    key = (lens.tobytes(), cols, seed, np.dtype(dtype).str)
    if key in _CSR_CACHE:
        return _CSR_CACHE[key]
    rng = np.random.default_rng(seed)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    parts = []
    for l in lens:
        l = int(l)
        if l == 0:
            continue
        if l > cols // 8:
            c = rng.choice(cols, size=l, replace=False)
        else:                       # cheap rejection sampling for short rows
            c = np.unique(rng.integers(0, cols, size=2 * l + 8))
            while c.size < l:
                c = np.unique(np.concatenate([c, rng.integers(0, cols, size=2 * l + 8)]))
            c = rng.permutation(c)[:l]
        parts.append(np.sort(c))
    col = (np.concatenate(parts) if parts else np.zeros(0, int)).astype(np.int32)
    val = rng.uniform(-1, 1, off[-1]).astype(dtype)
    _CSR_CACHE[key] = (off, col, val)
    return off, col, val


EDGE = {
    "all_empty": np.zeros(5000, int),
    "single_huge_row": np.array([100000]),
    "huge_then_tiny": np.concatenate([[50000], np.ones(3000, int), [0] * 500, [700], [511], [512], [513]]),
    "exactly_long": np.full(100, 512),
    "just_below_long": np.full(100, 511),
    "tile_sized_rows": np.full(20, 2048),
    "alternating": np.tile([0, 1, 4095, 0, 0, 3], 50),
    "one_by_one": np.array([1]),
    "trailing_empty": np.concatenate([np.full(10, 40), np.zeros(9000, int)]),
    "leading_empty": np.concatenate([np.zeros(9000, int), np.full(10, 40)]),
    "rmat_like_block": np.tile([500, 158, 158, 50, 158, 50, 50, 16, 158, 50, 50, 16, 50, 16, 16, 5], 12),
    "many_rows_end_in_one_step": np.concatenate([[1800], np.ones(40, int), np.zeros(50, int), np.full(30, 2), [1900, 0, 0, 0, 1, 1, 1],
                                                 [2500], np.zeros(40, int), [1500], np.zeros(70, int), [30, 2000]]),
    "rows_of_32": np.full(300, 32),
}


@pytest.mark.parametrize("name", list(EDGE))
def test_csr_edge_profiles(cs, b200, closed, name):
    lens = EDGE[name]
    rows, cols = lens.size, 120000
    off, col, val = lens_to_csr(lens, cols, 3)
    x = O.uniform(1, cols)
    y0 = O.uniform(2, rows)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    for alpha, beta in [(1.0, 0.0), (-2.0, 0.5)]:
        want = O.spmv_csr(off, col, val, x, y0, alpha, beta)
        got = run(cs, b200, "csr", rows, cols, arrays, dev(x), dev(y0), alpha, beta).cpu().numpy()
        assert relerr(got, want) < 1e-12, (name, alpha, beta)
        if off[-1] > 0:
            lib = run(cs, closed, "csr", rows, cols, arrays, dev(x), dev(y0), alpha, beta).cpu().numpy()
            assert relerr(got, lib) < 1e-12


def test_beta_zero_does_not_read_y(cs, b200):
    # spmv_csr_example.c:61-78 copies hY = 0 but a caller may pass uninitialised / NaN y with beta = 0
    off, col, val = O.gen_stencil5(64)
    n = 64 * 64
    x = O.uniform(8, n)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    y0 = torch.full((n,), float("nan"), dtype=torch.float64, device="cuda")
    got = run(cs, b200, "csr", n, n, arrays, dev(x), y0, 1.0, 0.0)
    assert relerr(got.cpu().numpy(), O.spmv_csr(off, col, val, x)) < 1e-13


def test_device_pointer_mode(cs, b200):
    # cusparse.h:275-278: alpha / beta may live in device memory
    rows = 10000
    off, col, val, x, y0 = rmat_case(rows, 10, torch.float64, 51)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    op = cs.SpMVOperator(b200, "csr", rows, rows, arrays)
    b200.cusparseSetPointerMode(op.handle, cs.CUSPARSE_POINTER_MODE_DEVICE)
    y = dev(y0)
    op(dev(x), y, dev(np.array([-0.5])), dev(np.array([2.0])))
    torch.cuda.synchronize()
    b200.cusparseSetPointerMode(op.handle, cs.CUSPARSE_POINTER_MODE_HOST)
    op.close()
    assert relerr(y.cpu().numpy(), O.spmv_csr(off, col, val, x, y0, -0.5, 2.0)) < 1e-12


def test_non_default_stream_and_graph_capture(cs, b200):
    """cuSPARSE/graph_capture/graph_capture_example.c:118-135 pattern: the call must be capturable (no sync / alloc)."""
    rows = 20000
    off, col, val, x, y0 = rmat_case(rows, 16, torch.float64, 61)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    xs, y = dev(x), dev(y0)
    want = O.spmv_csr(off, col, val, x, y0, 1.0, 0.0)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        op = cs.SpMVOperator(b200, "csr", rows, rows, arrays)   # handle bound to stream s
        op(xs, y, 1.0, 0.0)                                     # warm-up outside capture
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        y.zero_()
        with torch.cuda.graph(g, stream=s):
            op(xs, y, 1.0, 0.0)
        y.zero_()
        g.replay()
        g.replay()
    torch.cuda.synchronize()
    assert relerr(y.cpu().numpy(), want) < 1e-12
    op.close()


def test_unsupported_combinations_are_forwarded_not_broken(cs, b200, closed):
    """What our kernels do not take, the shim must hand to the closed library unchanged -- and count it.  64-bit indices with
    the generic kernels switched off (B200SPMV_GENERIC=off; with them on, the default: tests/test_generic_gpu.py) stand for that set
    (complex / 16-bit value types, CSC / BSR / Blocked-ELL)."""
    rows = 5000
    off, col, val, x, y0 = rmat_case(rows, 8, torch.float64, 71)
    arrays = dict(off=dev(off.astype(np.int64)), col=dev(col.astype(np.int64)), val=dev(val))
    b200.set_option("B200SPMV_GENERIC", "off")
    try:
        got = run(cs, b200, "csr", rows, rows, arrays, dev(x), dev(y0), 1.0, 0.0, expect_forward=True)
    finally:
        b200.set_option("B200SPMV_GENERIC", "csr")      # the library default
    assert relerr(got.cpu().numpy(), O.spmv_csr(off, col, val, x)) < 1e-12


def test_shape_mismatch_is_an_error(cs, b200):
    T = O.TOY
    h = b200.cusparseCreate()
    m = b200.cusparseCreateCsr(4, 4, 9, dev(T["csr_off"]), dev(T["csr_col"]), dev(T["val"]))
    xv = torch.zeros(3, device="cuda")
    yv = torch.zeros(4, device="cuda")
    vx, vy = b200.cusparseCreateDnVec(3, xv), b200.cusparseCreateDnVec(4, yv)
    buf = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    with pytest.raises(cs.CuSparseError):
        b200.cusparseSpMV(h, cs.CUSPARSE_OPERATION_NON_TRANSPOSE, 1.0, m, vx, 0.0, vy, cs.CUDA_R_32F, 0, buf)
    b200.cusparseDestroySpMat(m); b200.cusparseDestroyDnVec(vx); b200.cusparseDestroyDnVec(vy); b200.cusparseDestroy(h)


# ------------------------------------------------------------------------------------------ COO / SELL
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("alpha,beta", [(1.0, 0.0), (-1.0, 1.0)])
def test_coo_vs_oracle_and_cusparse(cs, b200, closed, coo_kernel, dtype, alpha, beta):
    rows = 40000
    off, col, val, x, y0 = rmat_case(rows, 16, dtype, 81)
    row = O.csr_to_coo_rows(off)
    want = O.spmv_coo(rows, row, col, val, x, y0, alpha, beta)
    arrays = dict(row=dev(row), col=dev(col), val=dev(val))
    got = run(cs, b200, "coo", rows, rows, arrays, dev(x), dev(y0), alpha, beta).cpu().numpy()
    lib = run(cs, closed, "coo", rows, rows, arrays, dev(x), dev(y0), alpha, beta).cpu().numpy()
    assert relerr(got, want) < TOL[dtype]
    assert relerr(got, lib) < TOL[dtype]


def test_coo_unsorted_and_tiny(cs, b200, coo_kernel):
    rows = 3000
    off, col, val, x, y0 = rmat_case(rows, 8, torch.float64, 91)
    row = O.csr_to_coo_rows(off)
    p = np.random.default_rng(0).permutation(row.size)
    arrays = dict(row=dev(row[p]), col=dev(col[p]), val=dev(val[p]))
    got = run(cs, b200, "coo", rows, rows, arrays, dev(x), dev(y0), 2.0, 0.5).cpu().numpy()
    assert relerr(got, O.spmv_coo(rows, row, col, val, x, y0, 2.0, 0.5)) < 1e-12
    # nnz = 0: y = beta*y
    arrays = dict(row=torch.zeros(0, dtype=torch.int32, device="cuda"), col=torch.zeros(0, dtype=torch.int32, device="cuda"),
                  val=torch.zeros(0, dtype=torch.float64, device="cuda"))
    got = run(cs, b200, "coo", rows, rows, arrays, dev(x), dev(y0), 2.0, 0.5).cpu().numpy()
    assert np.array_equal(got, 0.5 * y0)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("slice_size", [32, 2, 7, 64])
def test_sell_vs_oracle_and_cusparse(cs, b200, closed, dtype, slice_size):
    # config 3's matrix family: 7-pt Laplacian (laplace_generator.hxx:34-107) in Sliced-ELL, padding col -1
    nx = 24
    off, col, val = O.gen_laplace7(nx)
    val = val.astype(NP[dtype])
    n = nx ** 3
    so, sc, sv = O.csr_to_sell(off, col, val, slice_size)
    x = O.uniform(3, n, NP[dtype])
    y0 = O.uniform(4, n, NP[dtype])
    arrays = dict(off=dev(so), col=dev(sc), val=dev(sv), slice_size=slice_size, nnz=int(col.size))
    for alpha, beta in [(1.0, 0.0), (-1.0, 1.0)]:
        want = O.spmv_sell(n, slice_size, so, sc, sv, x, y0, alpha, beta)
        got = run(cs, b200, "sell", n, n, arrays, dev(x), dev(y0), alpha, beta).cpu().numpy()
        lib = run(cs, closed, "sell", n, n, arrays, dev(x), dev(y0), alpha, beta).cpu().numpy()
        assert relerr(got, want) < TOL[dtype]
        assert relerr(got, lib) < TOL[dtype]


def test_sell_ragged_rmat(cs, b200):
    rows = 10000 + 13   # last slice is partial
    off, col, val, x, y0 = rmat_case(rows, 6, torch.float64, 95)
    so, sc, sv = O.csr_to_sell(off, col, val, 32)
    arrays = dict(off=dev(so), col=dev(sc), val=dev(sv), slice_size=32, nnz=int(col.size))
    got = run(cs, b200, "sell", rows, rows, arrays, dev(x), dev(y0), 1.0, 2.0).cpu().numpy()
    assert relerr(got, O.spmv_csr(off, col, val, x, y0, 1.0, 2.0)) < 1e-12


# ------------------------------------------------------------------------------------------ fused CG step (8(f)-2)
@pytest.mark.parametrize("fuse_dot", [False, True])
@pytest.mark.parametrize("graph", [False, True])
def test_fused_cg_matches_the_sample_loop(cs, b200, graph, fuse_dot):
    """The fused device-scalar CG driver (csrc/cg_fused.cu) against a plain numpy restatement of cg_example.c:215-287
    (no preconditioner) on the sample's own matrix family; with and without CUDA-graph replay."""
    from cudalibrarysamples_b200.cg import CgSolver, FusedCgSolver
    from cudalibrarysamples_b200.sharded import ShardedCsr
    grid = 96
    off, col, val = O.gen_stencil5(grid)
    n = grid * grid
    b = O.spmv_csr(off, col, val, np.ones(n), alpha=0.75)            # cg_example.c:405-418
    # reference loop on the CPU with the oracle SpMV
    x = np.zeros(n); r = b.copy(); p = r.copy(); delta = r @ r
    iters = 25
    for _ in range(iters):
        t = O.spmv_csr(off, col, val, p)
        alpha = delta / (t @ p)
        x += alpha * p; r -= alpha * t
        dn = r @ r
        p = r + (dn / delta) * p
        delta = dn

    def make_local(rr, cc, arrays):
        return cs.SpMVOperator(b200, "csr", rr, cc, arrays, preprocess=True)
    sh = ShardedCsr(dev(off), dev(col), dev(val), 0, 1, make_local, balance="rows")
    solver = FusedCgSolver(sh, dev(b), use_graph=graph)
    solver.fuse_dot = fuse_dot and sh.can_fuse_dot()          # T = A*P with T.P in its epilogue (opt-in: B200CG_FUSE_DOT=1)
    assert solver.fuse_dot == fuse_dot
    xs, norms = solver.run(iters)
    torch.cuda.synchronize()
    assert solver.graph_error is None, solver.graph_error
    assert abs(norms[0] - np.sqrt(b @ b)) <= 1e-12 * np.sqrt(b @ b)
    assert abs(norms[-1] - np.sqrt(delta)) <= 1e-6 * np.sqrt(delta)          # 25 iterations of rounding differences
    assert relerr(xs.cpu().numpy(), x) < 1e-9
    # a second run on the same solver (bench: warm-up run, then the timed run) gives the same answer
    xs2, norms2 = solver.run(iters)
    assert torch.equal(xs, xs2) and norms2 == norms
    # and the torch-op driver agrees
    xt, nt = CgSolver(sh, dev(b)).run(iters)
    assert relerr(xt.cpu().numpy(), x) < 1e-9
    sh.close()


# ------------------------------------------------------------------------------------------ Matrix Market input
@pytest.mark.parametrize("name", ["toy_4x4.mtx", "rmat_300.mtx", "sym_lower_5.mtx"])
def test_matrix_market_files_through_the_spmv_path(cs, b200, closed, name):
    """SURVEY.md 8(f)-4: matrices read the way cuDSS/simple_matrix_market/matrix_market_reader.h reads them, then the
    sample's cusparseCreateCsr / cusparseSpMV sequence; checked against the oracle and the closed library."""
    from cudalibrarysamples_b200.mtx import read_matrix_market
    n, m, off, col, val = read_matrix_market(os.path.join(ROOT, "tests", "golden", name))
    x, y0 = O.uniform(1, m), O.uniform(2, n)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    want = O.spmv_csr(off, col, val, x, y0, 2.0, -1.0)
    got = run(cs, b200, "csr", n, m, arrays, dev(x), dev(y0), 2.0, -1.0).cpu().numpy()
    lib = run(cs, closed, "csr", n, m, arrays, dev(x), dev(y0), 2.0, -1.0).cpu().numpy()
    assert relerr(got, want) < 1e-13 and relerr(got, lib) < 1e-13


# ------------------------------------------------------------------------------------------ SpMM (CSR x dense)
def _dense(buf2d, order, dtype):
    """2-D numpy matrix -> 1-D device buffer in the given cuSPARSE order with the tight leading dimension"""
    a = np.ascontiguousarray(buf2d, NP[dtype]) if order == 2 else np.asfortranarray(buf2d, NP[dtype])
    return dev(a.reshape(-1, order="C" if order == 2 else "F").copy())


def _undense(t, shape, order):
    return t.cpu().numpy().reshape(shape, order="C" if order == 2 else "F")


def test_spmm_reference_golden(cs, b200):
    # spmm_csr_example.c:50-66,143-151: fp32, column-major, exact compare
    T = O.TOY
    arrays = dict(off=dev(T["csr_off"]), col=dev(T["csr_col"]), val=dev(T["val"]))
    before = b200.stats()
    C = cs.spmm(b200, 4, 4, arrays, _dense(T["spmm_B"], 1, torch.float32), torch.zeros(12, device="cuda"), 1.0, 0.0)
    assert np.array_equal(C.cpu().numpy(), np.array([19, 8, 51, 52, 43, 24, 123, 120, 67, 40, 195, 188], np.float32))
    after = b200.stats()
    assert after["native"] == before["native"] + 1 and after["forwarded"] == before["forwarded"]


def test_spmm_sample_passes_through_the_shim():
    exe = os.path.join(ROOT, "oracle", "_ref", "spmm_csr_example.b200")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref not built")
    p = subprocess.run([exe], capture_output=True, text=True, timeout=120, env=clean_env(B200SPMV_LOG="1"))
    assert p.returncode == 0, p.stdout + p.stderr
    assert "spmm_csr_example test PASSED" in p.stdout
    assert "[b200spmv] SpMM spmm_csr_kernel" in p.stderr and "forwarded" not in p.stderr


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("order_b,order_c", [(1, 1), (2, 2), (2, 1), (1, 2)])
@pytest.mark.parametrize("n", [1, 64, 70])
def test_spmm_vs_oracle_and_cusparse(cs, b200, closed, dtype, order_b, order_c, n):
    rows = 3000
    off, col, val, _, _ = rmat_case(rows, 12, dtype, 131)
    rng = np.random.default_rng(n)
    B = rng.uniform(-1, 1, (rows, n)).astype(NP[dtype])
    C0 = rng.uniform(-1, 1, (rows, n)).astype(NP[dtype])
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    ob, oc = ("row" if order_b == 2 else "col"), ("row" if order_c == 2 else "col")
    for alpha, beta in [(1.0, 0.0), (-0.5, 2.0)]:
        want = O.spmm_csr(off, col, val, B, C0, alpha, beta, order_b=ob, order_c=oc, threads=4)
        got = _undense(cs.spmm(b200, rows, rows, arrays, _dense(B, order_b, dtype), _dense(C0, order_c, dtype), alpha, beta,
                               order_b, order_c), (rows, n), order_c)
        assert relerr(got, want) < TOL[dtype], (order_b, order_c, n, alpha, beta)
        if order_b == order_c:      # the closed library wants B and C in the same order
            lib = _undense(cs.spmm(closed, rows, rows, arrays, _dense(B, order_b, dtype), _dense(C0, order_c, dtype), alpha, beta,
                                   order_b, order_c), (rows, n), order_c)
            assert relerr(got, lib) < TOL[dtype]


def test_spmm_edge_rows_and_base_one(cs, b200):
    lens = np.concatenate([[0, 0, 700, 1, 0, 33, 32, 31], np.zeros(40, int), [5, 64, 0]])
    off, col, val = lens_to_csr(lens, 900, 5)
    rng = np.random.default_rng(1)
    B, C0 = rng.uniform(-1, 1, (900, 9)), rng.uniform(-1, 1, (lens.size, 9))
    want = O.spmm_csr(off, col, val, B, C0, 1.5, -1.0, order_b="row", order_c="row")
    arrays = dict(off=dev(off + 1), col=dev(col + 1), val=dev(val))
    got = _undense(cs.spmm(b200, lens.size, 900, arrays, _dense(B, 2, torch.float64), _dense(C0, 2, torch.float64), 1.5, -1.0, 2, 2,
                           base=1), (lens.size, 9), 2)
    assert relerr(got, want) < 1e-12
    # beta == 0 must not read C (NaN in, finite out)
    nanC = torch.full((lens.size * 9,), float("nan"), dtype=torch.float64, device="cuda")
    got = _undense(cs.spmm(b200, lens.size, 900, arrays, _dense(B, 2, torch.float64), nanC, 1.0, 0.0, 2, 2, base=1), (lens.size, 9), 2)
    assert relerr(got, O.spmm_csr(off, col, val, B, None, 1.0, 0.0, order_b="row", order_c="row")) < 1e-12


# ------------------------------------------------------------------ bit-exact integer work on the device
def read_plan(buffer, num_tiles):
    from cudalibrarysamples_b200 import lib
    o = lib.shim().b200spmv_csr_plan_tiles_offset()
    raw = buffer[o:o + (num_tiles + 1) * 8].view(torch.int32).view(-1, 2)
    return raw.cpu().numpy()


@pytest.mark.parametrize("case", ["rmat", "stencil", "huge_then_tiny", "empty"])
@pytest.mark.parametrize("base", [0, 1])
def test_partition_is_bit_exact(cs, b200, case, base):
    from cudalibrarysamples_b200 import lib
    L = lib.shim()
    t, l, b = C.c_int32(), C.c_int32(), C.c_int32()
    L.b200spmv_csr_plan_params(C.byref(t), C.byref(l), C.byref(b))
    if case == "rmat":
        off = O.rmat_csr(200000, avg_nnz=16, seed=5, val_seed=6)[0]
    elif case == "stencil":
        off = O.gen_stencil5(300)[0]
    elif case == "empty":
        off = np.zeros(30001, np.int32)
    else:
        off = np.concatenate([[0], np.cumsum(EDGE["huge_then_tiny"])]).astype(np.int32)
    off = off + base
    rows, nnz = off.size - 1, int(off[-1]) - base
    nt = L.b200spmv_csr_num_tiles(C.c_int64(rows), C.c_int64(nnz))
    ws = torch.zeros(L.b200spmv_csr_workspace_bytes(C.c_int64(rows), C.c_int64(nnz)), dtype=torch.uint8, device="cuda")
    d_off = dev(off)
    rc = L.b200spmv_csr_analyze(C.c_void_p(torch.cuda.current_stream().cuda_stream), C.c_int64(rows), C.c_int64(nnz),
                                C.c_void_p(d_off.data_ptr()), C.c_int32(base), C.c_void_p(ws.data_ptr()))
    assert rc == 0
    torch.cuda.synchronize()
    got = read_plan(ws, nt)
    want = csr_partition(off, base, t.value, l.value)
    assert np.array_equal(got, want)
    assert check_partition(got, off, base, t.value, l.value)
    # the split-row list (order of registration is free, content is not)
    from oracle.partition_ref import split_rows
    oc = L.b200spmv_csr_plan_ctl_offset(C.c_int64(rows), C.c_int64(nnz))
    osp = L.b200spmv_csr_plan_split_offset(C.c_int64(rows), C.c_int64(nnz))
    ctl = ws[oc:oc + 8].view(torch.int32).cpu().numpy()
    nsplit = int(ctl[1])
    assert ctl[0] == 0
    lst = ws[osp:osp + 16 * nsplit].view(torch.int32).view(-1, 4).cpu().numpy()
    assert sorted((int(a), int(b), int(c)) for a, b, c, _ in lst) == split_rows(want, off, base, t.value)


@pytest.mark.parametrize("case", ["rmat", "stencil", "huge_then_tiny", "many_rows_end_in_one_step", "leading_empty"])
@pytest.mark.parametrize("base", [0, 1])
def test_flat_plan_is_bit_exact(case, base):
    """The flat CSR plan of cusparseSpMV_preprocess (end-lane bitmask, run counters, non-empty-row table) against its numpy
    restatement oracle/partition_ref.py::flat_plan -- integer work, bit for bit."""
    from cudalibrarysamples_b200 import lib
    from oracle.partition_ref import flat_plan
    L = lib.shim()
    L.b200spmv_csr_flat_workspace_bytes.restype = C.c_size_t
    if case == "rmat":
        off = O.rmat_csr(200000, avg_nnz=16, seed=5, val_seed=6)[0]
    elif case == "stencil":
        off = O.gen_stencil5(300)[0]
    else:
        off = np.concatenate([[0], np.cumsum(EDGE[case])]).astype(np.int32)
    off = off + base
    rows, nnz = off.size - 1, int(off[-1]) - base
    ws = torch.full((L.b200spmv_csr_flat_workspace_bytes(C.c_int64(rows), C.c_int64(nnz)),), 0xA5, dtype=torch.uint8, device="cuda")
    d_off = dev(off)
    rc = L.b200spmv_csr_flat_analyze(C.c_void_p(torch.cuda.current_stream().cuda_stream), C.c_int64(rows), C.c_int64(nnz),
                                     C.c_void_p(d_off.data_ptr()), C.c_int32(base), C.c_void_p(ws.data_ptr()))
    assert rc == 0
    torch.cuda.synchronize()
    om, oc, on, ol = C.c_size_t(), C.c_size_t(), C.c_size_t(), C.c_size_t()
    L.b200spmv_csr_flat_plan_offsets(C.c_int64(rows), C.c_int64(nnz), C.byref(om), C.byref(oc), C.byref(on), C.byref(ol))
    mask, chunk_run, nzrow, (nruns, quiet, steps) = flat_plan(off, base)
    got_mask = ws[om.value:om.value + 4 * mask.size].view(torch.int32).cpu().numpy().view(np.uint32)
    got_run = ws[oc.value:oc.value + 4 * chunk_run.size].view(torch.int32).cpu().numpy()
    got_nzrow = ws[on.value:on.value + 4 * nzrow.size].view(torch.int32).cpu().numpy()
    ctl = ws[ol.value:ol.value + 16].view(torch.int32).cpu().numpy()
    assert np.array_equal(got_mask, mask)
    assert np.array_equal(got_run, chunk_run)
    assert np.array_equal(got_nzrow, nzrow)
    assert (int(ctl[0]), int(ctl[1]), int(ctl[2])) == (nruns, quiet, steps) and int(ctl[3]) == nruns


def test_flat_kernel_is_chosen_for_skewed_rows_only(cs, b200):
    """auto: preprocess reads the row statistic back and picks csr_flat_kernel for R-MAT, the tile kernels for a stencil."""
    off, col, val, x, y0 = rmat_case(60000, 16, torch.float64, 21)
    run(cs, b200, "csr", 60000, 60000, dict(off=dev(off), col=dev(col), val=dev(val)), dev(x), dev(y0), 1.0, 0.0)
    assert "csr_flat_kernel" in b200.last_csr_kernel()
    run(cs, b200, "csr", 60000, 60000, dict(off=dev(off), col=dev(col), val=dev(val)), dev(x), dev(y0), 1.0, 0.0, preprocess=False)
    assert "csr_flat_kernel" not in b200.last_csr_kernel()
    rows = 40000
    col16 = np.sort(np.random.default_rng(0).integers(0, rows, (rows, 16)), axis=1).astype(np.int32).reshape(-1)
    off16 = (np.arange(rows + 1) * 16).astype(np.int32)
    val16 = O.uniform(3, rows * 16)
    run(cs, b200, "csr", rows, rows, dict(off=dev(off16), col=dev(col16), val=dev(val16)), dev(O.uniform(4, rows)), dev(O.uniform(5, rows)), 1.0, 0.0)
    assert "csr_flat_kernel" not in b200.last_csr_kernel()


def test_short_kernel_is_chosen_when_every_row_is_short(cs, b200):
    """auto: preprocess reads the longest row back; stencils (cg_example.c:71-128) go to csr_short_kernel, R-MAT never does,
    and a call without cusparseSpMV_preprocess (cg_example.c itself) stays on the plan-per-call tile kernels."""
    off, col, val = O.gen_stencil5(300)
    n = 300 * 300
    xs, ys = O.uniform(5, n), O.uniform(6, n)
    arrays = dict(off=dev(off), col=dev(col), val=dev(val))
    want = O.spmv_csr(off, col, val, xs, ys, 0.75, 0.5)
    got = run(cs, b200, "csr", n, n, arrays, dev(xs), dev(ys), 0.75, 0.5)
    assert "csr_short_kernel" in b200.last_csr_kernel()
    assert relerr(got.cpu().numpy(), want) < 1e-13
    got = run(cs, b200, "csr", n, n, arrays, dev(xs), dev(ys), 0.75, 0.5, preprocess=False)
    assert "csr_short_kernel" not in b200.last_csr_kernel()
    assert relerr(got.cpu().numpy(), want) < 1e-12
    # one row of 33 non-zeros among the short ones: not eligible any more
    lens = np.full(5000, 5); lens[1234] = 33
    off, col, val = lens_to_csr(lens, 20000, 9)
    x, y0 = O.uniform(1, 20000), O.uniform(2, 5000)
    got = run(cs, b200, "csr", 5000, 20000, dict(off=dev(off), col=dev(col), val=dev(val)), dev(x), dev(y0), 1.0, 0.0)
    assert "csr_short_kernel" not in b200.last_csr_kernel()
    assert relerr(got.cpu().numpy(), O.spmv_csr(off, col, val, x, y0, 1.0, 0.0)) < 1e-12
    lens[1234] = 32
    off, col, val = lens_to_csr(lens, 20000, 9)
    got = run(cs, b200, "csr", 5000, 20000, dict(off=dev(off), col=dev(col), val=dev(val)), dev(x), dev(y0), 1.0, 0.0)
    assert "csr_short_kernel" in b200.last_csr_kernel()
    assert relerr(got.cpu().numpy(), O.spmv_csr(off, col, val, x, y0, 1.0, 0.0)) < 1e-12


def test_device_generators_are_bit_identical_to_the_oracle():
    from cudalibrarysamples_b200 import workloads as W
    off, col, val = W.rmat_csr(30000, avg_nnz=16, seed=42, val_seed=43)
    o2, c2, v2 = O.rmat_csr(30000, avg_nnz=16, seed=42, val_seed=43)
    assert np.array_equal(off.cpu().numpy(), o2) and np.array_equal(col.cpu().numpy(), c2)
    assert np.array_equal(val.cpu().numpy(), v2)
    assert np.array_equal(W.uniform(44, 1000, torch.float32).cpu().numpy(), O.uniform(44, 1000, np.float32))
    for a, b in zip(W.stencil5_csr(97), O.gen_stencil5(97)):
        assert np.array_equal(a.cpu().numpy(), b)
    for a, b in zip(W.stencil5_csr(31, 0.3, 0.3, 0.2), O.gen_stencil5(31, 0.3, 0.3, 0.2)):
        assert np.array_equal(a.cpu().numpy(), b)
    for a, b in zip(W.laplace7_csr(13), O.gen_laplace7(13)):
        assert np.array_equal(a.cpu().numpy(), b)
    off, col, val = O.gen_laplace7(9)
    for ss in (32, 5):
        for a, b in zip(W.csr_to_sell(dev(off), dev(col), dev(val), ss), O.csr_to_sell(off, col, val, ss)):
            assert np.array_equal(a.cpu().numpy(), b)
    assert np.array_equal(W.csr_to_coo_rows(dev(off)).cpu().numpy(), O.csr_to_coo_rows(off))


def test_coo_alg2_keeps_its_reproducibility_promise(cs, b200):
    """CUSPARSE_SPMV_COO_ALG2 = "provides deterministic (bit-wise) results for each run" (cusparse.h, cusparseSpMVAlg_t):
    our COO kernels use floating-point atomics, so that request is handed to the closed library -- counted as a forward."""
    off, col, val, x, y0 = rmat_case(30000, 16, torch.float64, 77)
    row = np.repeat(np.arange(30000, dtype=np.int32), np.diff(off))
    arrays = dict(row=dev(row), col=dev(col), val=dev(val))
    want = O.spmv_csr(off, col, val, x, y0, 1.0, 0.5)
    outs = []
    for _ in range(2):
        before = b200.stats()
        op = cs.SpMVOperator(b200, "coo", 30000, 30000, arrays, alg=4)          # CUSPARSE_SPMV_COO_ALG2
        y = dev(y0).clone()
        op(dev(x), y, 1.0, 0.5)
        torch.cuda.synchronize()
        op.close()
        after = b200.stats()
        assert after["forwarded"] == before["forwarded"] + 1 and after["native"] == before["native"]
        outs.append(y)
    assert torch.equal(outs[0], outs[1])
    assert relerr(outs[0].cpu().numpy(), want) < 1e-12


@pytest.mark.parametrize("fmt", ["csr", "coo"])
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_transposed_spmv_is_native(cs, b200, closed, fmt, dtype):
    """opA = CUSPARSE_OPERATION_TRANSPOSE (cusparse.h cusparseOperation_t): y[cols] = alpha * A^T x[rows] + beta * y on a
    rectangular matrix with empty rows, base 1; against the oracle run on the explicitly transposed matrix and against the
    closed library; served by our kernels (no forward)."""
    import scipy.sparse as sp
    rows, cols = 30000, 21000
    off, col, val, _, _ = rmat_case(rows, 12, dtype, 55)
    col = (col % cols).astype(np.int32)                          # rectangular: fold the columns (duplicates inside a row are fine)
    x, y0 = O.uniform(7, rows).astype(val.dtype), O.uniform(8, cols).astype(val.dtype)
    A = sp.csr_matrix((val.astype(np.float64), col, off), shape=(rows, cols))
    want = -1.5 * (A.T @ x.astype(np.float64)) + 0.5 * y0.astype(np.float64)
    if fmt == "csr":
        arrays = dict(off=dev(off + 1), col=dev(col + 1), val=dev(val))
    else:
        row = np.repeat(np.arange(rows, dtype=np.int32), np.diff(off))
        arrays = dict(row=dev(row + 1), col=dev(col + 1), val=dev(val))
    outs = {}
    for name, api in (("ours", b200), ("closed", closed)):
        before = api.stats() if api.impl == "b200" else None
        op = cs.SpMVOperator(api, fmt, rows, cols, arrays, base=1, op=cs.CUSPARSE_OPERATION_TRANSPOSE)
        y = dev(y0).clone()
        op(dev(x), y, -1.5, 0.5)
        torch.cuda.synchronize()
        op.close()
        if before is not None:
            after = api.stats()
            assert after["forwarded"] == before["forwarded"] and after["native"] == before["native"] + 1
        outs[name] = y.cpu().numpy()
    assert relerr(outs["ours"], want) < TOL[dtype]
    assert relerr(outs["ours"], outs["closed"]) < TOL[dtype]
    # beta = 0 must not read y (NaN-filled), alpha = 1
    op = cs.SpMVOperator(b200, fmt, rows, cols, arrays, base=1, op=cs.CUSPARSE_OPERATION_TRANSPOSE, preprocess=False)
    y = torch.full((cols,), float("nan"), dtype=dtype, device="cuda")
    op(dev(x), y, 1.0, 0.0)
    torch.cuda.synchronize()
    op.close()
    assert relerr(y.cpu().numpy(), A.T @ x.astype(np.float64)) < TOL[dtype]


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
def test_short_kernel_with_the_dot_product_in_its_epilogue(b200, dtype):
    """b200spmv_csr_short_mv_dot: T = A*P and T . P of a CG iteration (cg_example.c:220-227) in one launch; the dot is
    accumulated in fp64, deterministic, and the arrival counter of its workspace is left at zero (second call = same bits)."""
    import ctypes as C
    L = b200.lib
    L.b200spmv_csr_short_dot_workspace_bytes.restype = C.c_size_t
    off, col, val = O.gen_stencil5(257)
    n = 257 * 257
    val = val.astype(NP[dtype])
    x = O.uniform(5, n).astype(NP[dtype])
    want_y = O.spmv_csr(off, col, val, x, np.zeros(n, NP[dtype]), 1.0, 0.0)
    want_dot = float(np.dot(want_y.astype(np.float64), x.astype(np.float64)))
    d_off, d_col, d_val, d_x = dev(off), dev(col), dev(val), dev(x)
    y = torch.full((n,), float("nan"), dtype=dtype, device="cuda")
    out = torch.zeros(2, dtype=torch.float64, device="cuda")
    ws = torch.zeros(int(L.b200spmv_csr_short_dot_workspace_bytes()), dtype=torch.uint8, device="cuda")
    ct = C.c_double if dtype == torch.float64 else C.c_float
    one, zero = ct(1.0), ct(0.0)
    got = []
    for k in range(2):
        rc = L.b200spmv_csr_short_mv_dot(C.c_void_p(torch.cuda.current_stream().cuda_stream), C.c_int(1 if dtype == torch.float64 else 0),
                                         C.c_int64(n), C.c_int64(n), C.c_int64(int(col.size)), C.c_void_p(d_off.data_ptr()),
                                         C.c_void_p(d_col.data_ptr()), C.c_void_p(d_val.data_ptr()), C.c_int32(0), C.byref(one), C.byref(zero),
                                         C.c_int(0), C.c_void_p(d_x.data_ptr()), C.c_void_p(y.data_ptr()), C.c_void_p(d_x.data_ptr()),
                                         C.c_void_p(out[k:k + 1].data_ptr()), C.c_void_p(ws.data_ptr()))
        assert rc == 0
        torch.cuda.synchronize()
        got.append(float(out[k].item()))
    assert relerr(y.cpu().numpy(), want_y) < TOL[dtype]
    assert abs(got[0] - want_dot) <= (1e-12 if dtype == torch.float64 else 1e-5) * abs(want_dot)
    assert got[0] == got[1]
