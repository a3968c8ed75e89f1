"""Element-wise checking of y = alpha * op(A) * x + beta * y and C = alpha * A * B + beta * C: the comparator, the guard bands
and the value regimes shared by tests/test_elementwise_cpu.py and tests/test_elementwise_gpu.py.

A norm-wise relative error (||y - y_ref|| / ||y_ref||) misses kernels that are wrong in a few elements, in rows whose result
is small next to ||y||, or only for non-finite inputs.  This module checks every output element on its own:

  * per-element bound, valid for any summation order.  For output element i with L_i stored entries
        |got_i - ref_i| <= (gamma_T(L_i + 2) + gamma_64(L_i + 2)) * (|alpha| * sum_j |a_ij| |x_j| + |beta| |y0_i|) + (L_i + 2) * eta_T
    gamma_T(n) = n u / (1 - n u) with u the unit roundoff of the arithmetic type T (2^-24 for fp32; 2^-53 for fp64 and for fp32
    A with fp64 x / y), eta_T the smallest positive subnormal of T.  ref is the CPU oracle's result, accumulated in fp64 on
    the inputs widened exactly to fp64; gamma_64 covers the oracle's own rounding.  For SpMM the bound holds per element of C;
    for op(A) = A^T, L_i counts the entries of column i.
  * non-finite classification: where ref_i is NaN, +Inf or -Inf, got_i must be the same class; where ref_i is finite, got_i
    must be finite and meet the bound.  The class does not depend on the summation order (a sum holding +Inf and -Inf is NaN
    in any order), and none of the value regimes below can overflow or underflow in correct arithmetic.
  * guard bands: every operand is a view into a larger buffer.  x / B and the stored values are surrounded by NaN, the column
    (and COO row) indices by the valid index `base`, so a stray read shows up as NaN in the result instead of as a fault; y / C
    are surrounded by a sentinel bit pattern that must be bit-identical after the call.
"""
import numpy as np
import scipy.sparse as sp

from oracle import oracle as O

F32, F64 = np.dtype(np.float32), np.dtype(np.float64)
UNIT_ROUNDOFF = {F32: 2.0 ** -24, F64: 2.0 ** -53}
TINY = {F32: 2.0 ** -149, F64: 2.0 ** -1074}

# a multiple of 4 elements and an odd count: both sides of every 16-byte alignment test a kernel makes on its operands
GUARDS = (8, 3)
# signalling-NaN bit patterns: a kernel that reads the band gets a NaN, one that writes it changes the bits
SENTINEL = {F32: np.uint32(0x7FA5A5A5), F64: np.uint64(0x7FF5A5A5A5A5A5A5)}
UINT = {F32: np.uint32, F64: np.uint64}

REGIMES = ("uniform", "cancel", "wide", "nonfinite")
# (alpha, beta) per regime; with beta == 0 y starts NaN-filled (beta == 0 must not read y).  alpha == 0 is left out: cuSPARSE
# does not document whether it still forms A * x then.
SCALARS = {
    "uniform": ((1.0, 0.0), (-2.0, 0.5)),
    "cancel": ((-1.0, 1.0),),                 # y0 = A * x: the exact result is close to 0 in every row
    "wide": ((0.75, -1.5),),
    "nonfinite": ((1.0, 0.0), (-1.5, 0.5)),
    "nan_padding": ((1.0, 0.0), (-2.0, 0.5)),     # Sliced-ELL only: uniform values, NaN stored in every padding slot
}


def gamma(n, u):
    n = np.asarray(n, np.float64)
    return n * u / (1.0 - n * u)


def arith_type(a_dt, xy_dt):
    """The type the arithmetic runs in: that of x / y (fp32 A with fp64 x / y computes in fp64)."""
    return np.dtype(xy_dt)


def csr_of(off, col, val, shape):
    """scipy CSR over float64 values that keeps every stored entry (duplicates are not merged: each one is a term of the sum)."""
    return sp.csr_matrix((np.asarray(val, np.float64), np.asarray(col, np.int64), np.asarray(off, np.int64)), shape=shape)


def transpose_csr(M):
    """(A^T in CSR with one stored entry per stored entry of A, perm): entry k of A^T is entry perm[k] of A (scipy's
    conversions may merge duplicates)."""
    rows, cols = M.shape
    r = np.repeat(np.arange(rows, dtype=np.int64), np.diff(M.indptr))
    perm = np.argsort(M.indices, kind="stable")
    off = np.concatenate([[0], np.cumsum(np.bincount(M.indices, minlength=cols))])
    return csr_of(off, r[perm], M.data[perm], (cols, rows)), perm


def reference(M, x, y0, alpha, beta):
    """The oracle's y = alpha * M * x + beta * y0 (M = op(A) as CSR; fp64 accumulation on inputs widened exactly to fp64).
    x may be 2-D (SpMM: B, then y0 is C0); beta == 0 never reads y0."""
    off, col, val = M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data.astype(np.float64)
    x = np.asarray(x, np.float64)
    y0 = np.asarray(y0, np.float64)
    if x.ndim == 2:
        return O.spmm_csr(off, col, val, x, y0, alpha, beta, order_b="row", order_c="row")
    return O.spmv_csr(off, col, val, x, y0, alpha, beta)


def row_bound(M, x, y0, alpha, beta, arith):
    """The per-element bound above (M = op(A) as CSR, x 1-D or 2-D, arith = numpy type of the arithmetic)."""
    arith = np.dtype(arith)
    n = (np.diff(M.indptr) + 2).astype(np.float64)
    x = np.asarray(x, np.float64)
    if x.ndim == 2:
        n = n[:, None]
    absM = csr_of(M.indptr, M.indices, np.abs(M.data), M.shape)
    with np.errstate(invalid="ignore", over="ignore"):
        mag = abs(alpha) * (absM @ np.abs(x))
        if beta != 0:
            mag = mag + abs(beta) * np.abs(np.asarray(y0, np.float64))
    return (gamma(n, UNIT_ROUNDOFF[arith]) + gamma(n, UNIT_ROUNDOFF[F64])) * mag + n * TINY[arith]


def _cls(v):
    """0 finite, 1 NaN, 2 +Inf, 3 -Inf"""
    return np.where(np.isnan(v), 1, np.where(v == np.inf, 2, np.where(v == -np.inf, 3, 0)))


def bad_elements(got, ref, bound):
    """Flat indices of the elements that fail the classification or the bound."""
    ref = np.asarray(ref, np.float64)
    bound = np.broadcast_to(np.asarray(bound, np.float64), ref.shape).ravel()
    got = np.asarray(got, np.float64).ravel()
    ref = ref.ravel()
    cg, cr = _cls(got), _cls(ref)
    with np.errstate(invalid="ignore", over="ignore"):
        off = (cr == 0) & ~(np.abs(got - ref) <= bound)
    return np.flatnonzero((cg != cr) | off)


def assert_elementwise(got, ref, bound, what=""):
    bad = bad_elements(got, ref, bound)
    if bad.size:
        g, r = np.asarray(got, np.float64).ravel(), np.asarray(ref, np.float64).ravel()
        b = np.broadcast_to(np.asarray(bound, np.float64), np.shape(ref)).ravel()
        first = ", ".join(f"[{i}] got {g[i]!r} want {r[i]!r} (bound {b[i]:.3g})" for i in bad[:5])
        raise AssertionError(f"{what}: {bad.size} of {r.size} elements wrong; first: {first}")


# ------------------------------------------------------------------------------------------------ guard bands
def guarded(a, G, band):
    """A buffer of a.size + 2G elements holding `a` at offset G; both bands hold `band` (a value, or "sentinel")."""
    a = np.ascontiguousarray(a)
    buf = np.empty(a.size + 2 * G, a.dtype)
    if isinstance(band, str):
        buf.view(UINT[a.dtype])[:] = SENTINEL[a.dtype]
    else:
        buf[:] = band
    buf[G:G + a.size] = a
    return buf


def bands_intact(buf, G, n):
    """Both bands of a guarded("sentinel") output buffer still hold the sentinel, bit for bit."""
    bits = np.asarray(buf).view(UINT[np.asarray(buf).dtype])
    s = SENTINEL[np.asarray(buf).dtype]
    return bool(np.all(bits[:G] == s) and np.all(bits[G + n:] == s))


# ------------------------------------------------------------------------------------------------ value regimes
def _wide_k(a_dt, xy_dt):
    """Exponent ranges (A, x) of the `wide` regime: any fp32 intermediate on an fp64 path overflows or underflows."""
    if np.dtype(xy_dt) == F32:
        return 25, 25
    return (25, 200) if np.dtype(a_dt) == F32 else (100, 100)


def _wide(rng, size, k):
    return np.ldexp(rng.choice([-1.0, 1.0], size), rng.integers(-k, k + 1, size))


def values(regime, nnz, x_shape, y_shape, a_dt, xy_dt, seed):
    """Stored values of A, x (or B) and y0 (or C0) for a regime.  `cancel` uses the uniform values; its y0 = A * x is set by
    the caller (cancel_y0).  `nonfinite` puts NaN at x[0] (the index masked lanes default to), -Inf at x[-1], +Inf / -Inf /
    NaN at a few random positions, one Inf among the stored values and one in y0 (read only when beta != 0).  For a 2-D x
    (SpMM's B) the non-finite values go into row 0 of B."""
    rng = np.random.default_rng(seed)
    if regime == "wide":
        ka, kx = _wide_k(a_dt, xy_dt)
        val, x, y0 = _wide(rng, nnz, ka), _wide(rng, int(np.prod(x_shape)), kx), _wide(rng, int(np.prod(y_shape)), kx)
    else:
        val = rng.uniform(-1, 1, nnz)
        x, y0 = rng.uniform(-1, 1, int(np.prod(x_shape))), rng.uniform(-1, 1, int(np.prod(y_shape)))
    x, y0 = x.reshape(x_shape), y0.reshape(y_shape)
    if regime == "nonfinite":
        if x.ndim == 2:
            n = x.shape[1]
            x[0, :] = np.resize([np.nan, np.inf, -np.inf], n)
        elif x.size:
            x[rng.integers(0, x.size, 3)] = [np.inf, -np.inf, np.nan]
            x[0], x[-1] = np.nan, -np.inf
        if nnz:
            val[rng.integers(nnz)] = np.inf
        if y0.size:
            y0.flat[rng.integers(y0.size)] = np.inf
    return val.astype(a_dt), x.astype(xy_dt), y0.astype(xy_dt)


def cancel_y0(M, x, xy_dt):
    """y0 = oracle(op(A) * x), rounded to the type of y: with alpha = -1, beta = 1 every row of the result nearly cancels."""
    x = np.asarray(x, np.float64)
    zeros = np.zeros((M.shape[0],) + x.shape[1:])
    return reference(M, x, zeros, 1.0, 0.0).astype(xy_dt)


def start_y(y0, beta):
    """What y holds before the call: y0, or NaN everywhere when beta == 0."""
    return y0.copy() if beta != 0 else np.full_like(y0, np.nan)


def cases(M, x_shape, y_shape, a_dt, xy_dt, seed, regimes=REGIMES):
    """(regime, alpha, beta, val, x, y0, ref, bound) for every regime and scalar pair; val in the storage order of M's entries
    (the caller maps it onto its format).  M's own values are replaced."""
    arith = arith_type(a_dt, xy_dt)
    for regime in regimes:
        val, x, y0 = values(regime, M.nnz, x_shape, y_shape, a_dt, xy_dt, seed)
        Mv = csr_of(M.indptr, M.indices, val, M.shape)
        if regime == "cancel":
            y0 = cancel_y0(Mv, x, xy_dt)
        for alpha, beta in SCALARS[regime]:
            yield regime, alpha, beta, val, x, y0, reference(Mv, x, y0, alpha, beta), row_bound(Mv, x, y0, alpha, beta, arith)


# ------------------------------------------------------------------------------------------------ shapes
def lens_to_csr(lens, cols, seed):
    """Random CSR structure with the given row lengths (distinct sorted columns per row)."""
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
    return off, col


# Row-length profiles where kernels go wrong first (split rows, many row ends in one step, empty runs, tile-sized rows).
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
