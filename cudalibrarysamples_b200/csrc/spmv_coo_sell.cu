// spmv_coo_sell.cu -- COO and Sliced-ELL  y = alpha*A*x + beta*y  for B200 (sm_100a), fp32 / fp64, int32 indices.
//
// COO replaces cusparse::coomv_kernel behind cusparseSpMV for cusparseCreateCoo descriptors
//   (cuSPARSE/spmv_coo/spmv_coo_example.c:86-104): SoA row/col/val arrays, usually row-sorted
//   (spmv_coo_example.c:48-49) but any order is accepted.
// SELL replaces cusparse::sellmv_v1_kernel behind cusparseSpMV for cusparseCreateSlicedEll descriptors
//   (cuSPARSE/spmv_sell/spmv_sell_example.c:103-122): column-major inside each slice, padding col = -1.
#include "spmv_common.cuh"
#include "config.h"
#include "../../include/b200spmv.h"
#include <cstdlib>
#include <mutex>

#ifndef B200_SELL_UNROLL
#define B200_SELL_UNROLL 8
#endif
#ifndef B200_SELL_MIN_CTAS
#define B200_SELL_MIN_CTAS 4
#endif
#ifndef B200_SELL32_MIN_CTAS
#define B200_SELL32_MIN_CTAS 8   // 32 registers, 2048 threads/SM: measured 174 us vs 195 us at 40 registers (config 3)
#endif
#ifndef B200_SELL_WAVES      // persistent grid = SMs x resident CTAs x this
#define B200_SELL_WAVES 1
#endif

namespace b200 {

// ================================================================================================
// COO
//   pass 1: y = beta*y (or 0)                       -- rows without entries must still be scaled
//   pass 2: tiles of COO_TILE non-zeros; each thread owns COO_PER_THREAD consecutive entries (from
//           shared memory, after a coalesced 128-bit streaming load), folds runs of equal row index
//           and issues one fp atomic per run (RED.ADD at L2).  Runs that continue in the neighbouring
//           thread / tile simply produce one more atomic, so unsorted input stays correct.
// ================================================================================================
constexpr int COO_BLOCK = 256;
constexpr int COO_PER_THREAD = 8;
constexpr int COO_TILE = COO_BLOCK * COO_PER_THREAD;  // 2048, multiple of 4 -> tile starts stay 16B aligned

template <typename T>
__global__ void scale_y_kernel(T* __restrict__ y, int64_t rows, Scalars<T> s) {
    const T beta = s.b();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += (int64_t)gridDim.x * blockDim.x)
        y[i] = beta == T(0) ? T(0) : beta * y[i];
}

template <typename T>
struct CooArgs {
    const int* row;
    const int* col;
    const T*   val;
    const T*   x;
    T*         y;
    int        base;
    int        nnz;
    int        vec_ok;
    Scalars<T> s;
};

template <typename T>
__global__ void __launch_bounds__(COO_BLOCK) coo_tile_kernel(const CooArgs<T> a) {
    __shared__ T   sP[COO_TILE + COO_BLOCK / 4];  // padded: index i lives at i + i/32 -> conflict-free strided walk
    __shared__ int sR[COO_TILE + COO_BLOCK / 4];
    const int n0 = blockIdx.x * COO_TILE;
    const int n1 = min(n0 + COO_TILE, a.nnz);
    const T   alpha = a.s.a();
    constexpr int ITERS = COO_TILE / (COO_BLOCK * 4);
    const int nnz_vec_end = a.vec_ok ? (a.nnz & ~3) : 0;

    int r[ITERS][4], c[ITERS][4];
    T   v[ITERS][4];
#pragma unroll
    for (int it = 0; it < ITERS; it++) {
        const int i0 = n0 + (it * COO_BLOCK + (int)threadIdx.x) * 4;
        if (i0 < n1) {
            if (i0 + 4 <= nnz_vec_end) {
                const int4 rr = ldg_stream_int4(a.row + i0), cc = ldg_stream_int4(a.col + i0);
                r[it][0] = rr.x; r[it][1] = rr.y; r[it][2] = rr.z; r[it][3] = rr.w;
                c[it][0] = cc.x; c[it][1] = cc.y; c[it][2] = cc.z; c[it][3] = cc.w;
                load4_stream(a.val + i0, v[it]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const bool ok = i0 + j < n1;
                    r[it][j] = ok ? ldg_stream(a.row + i0 + j) : a.base;
                    c[it][j] = ok ? ldg_stream(a.col + i0 + j) : a.base;
                    v[it][j] = ok ? ldg_stream(a.val + i0 + j) : T(0);
                }
            }
        }
    }
#pragma unroll
    for (int it = 0; it < ITERS; it++) {
        const int i0 = n0 + (it * COO_BLOCK + (int)threadIdx.x) * 4;
        if (i0 < n1) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int i = i0 + j - n0;
                if (i0 + j < n1) {
                    const T xv = __ldg(a.x + (c[it][j] - a.base));
                    sP[i + (i >> 5)] = v[it][j] * xv;
                    sR[i + (i >> 5)] = r[it][j] - a.base;
                }
            }
        }
    }
    __syncthreads();

    const int cnt = n1 - n0;
    const int k0 = (int)threadIdx.x * COO_PER_THREAD;
    if (k0 < cnt) {
        const int k1 = min(k0 + COO_PER_THREAD, cnt);
        int cur = sR[k0 + (k0 >> 5)];
        T   sum = sP[k0 + (k0 >> 5)];
        for (int k = k0 + 1; k < k1; k++) {
            const int rr = sR[k + (k >> 5)];
            const T   p  = sP[k + (k >> 5)];
            if (rr != cur) {
                atomicAdd(a.y + cur, alpha * sum);
                cur = rr; sum = p;
            } else {
                sum += p;
            }
        }
        atomicAdd(a.y + cur, alpha * sum);
    }
}

// ------------------------------------------------------------------------------------------------
// coo_seg_kernel (default): no shared memory, no barriers -- every warp owns a contiguous chunk of COO_SEG_STEPS x 32
// entries and walks it with a per-lane accumulator, exactly like csr_seg_kernel, except that the row boundaries come
// straight from the row indices: lane l ends a run iff row[l] != row[l + 1].  A 32-entry step inside one row costs
// nothing (acc += product); a step with run ends costs one butterfly for the first run (accumulator + head of the
// step) plus a segmented shuffle scan with as many levels as the longest remaining run needs, and ONE atomic (RED.ADD
// at L2) per run end.  For row-sorted input (spmv_coo_example.c:48-49) that is one atomic per row and chunk instead of
// one per 8 entries; unsorted input stays correct (every run of equal row indices is just added where it belongs).
// Measured motivation: round 1's coo_tile_kernel was 0.66x the closed library on R-MAT 1M (125.8 vs 82.8 us).
// ------------------------------------------------------------------------------------------------
#ifndef B200_COO_SEG_STEPS
#define B200_COO_SEG_STEPS 8
#endif
#ifndef B200_COO_SEG_BATCH
#define B200_COO_SEG_BATCH 4
#endif
#ifndef B200_COO_SEG_MIN_CTAS
#define B200_COO_SEG_MIN_CTAS 4
#endif
constexpr int COO_SEG_STEPS = B200_COO_SEG_STEPS, COO_SEG_BATCH = B200_COO_SEG_BATCH;
constexpr int COO_SEG_CHUNK = 32 * COO_SEG_STEPS;
static_assert(COO_SEG_STEPS % COO_SEG_BATCH == 0, "steps per chunk must be a multiple of the batch");

template <typename T>
__device__ __forceinline__ T coo_warp_allsum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

template <typename T>
__global__ void __launch_bounds__(COO_BLOCK, B200_COO_SEG_MIN_CTAS) coo_seg_kernel(const CooArgs<T> a) {
    const int lane = (int)threadIdx.x & 31;
    const long long wid = (long long)blockIdx.x * (COO_BLOCK / 32) + ((int)threadIdx.x >> 5);
    const long long c0 = wid * COO_SEG_CHUNK;
    if (c0 >= a.nnz) return;                                  // warp-uniform
    const int n0 = (int)c0;
    const int n1 = min(n0 + COO_SEG_CHUNK, a.nnz);            // this warp's entries [n0, n1)
    const T alpha = a.s.a();
    T acc = T(0);

    int r[COO_SEG_BATCH], rn[COO_SEG_BATCH], c[COO_SEG_BATCH];
    T   v[COO_SEG_BATCH];
    auto issue = [&](int kb) {
#pragma unroll
        for (int k = 0; k < COO_SEG_BATCH; k++) {
            const int e = n0 + (kb + k) * 32 + lane;
            const bool live = e < n1;
            r[k]  = live ? ldg_stream(a.row + e) : -1;
            rn[k] = (live && e + 1 < n1) ? ldg_stream(a.row + e + 1) : -2;    // the chunk's last entry always ends a run
            c[k]  = live ? ldg_stream(a.col + e) : a.base;
            v[k]  = live ? ldg_stream(a.val + e) : T(0);
        }
    };
    issue(0);
    // Fully unrolled over the 8 steps of a chunk (47 KB of SASS for fp64): measured 79.0 us on R-MAT 1M against 83.1 us
    // with run-time step loops (5 KB) -- unlike csr_seg_kernel (159 KB unrolled) this one still fits the instruction cache.
#pragma unroll
    for (int kb = 0; kb < COO_SEG_STEPS; kb += COO_SEG_BATCH) {
        if (n0 + kb * 32 >= n1) break;                        // warp-uniform
        T   p[COO_SEG_BATCH];
        int rr[COO_SEG_BATCH];
        unsigned mm[COO_SEG_BATCH];
#pragma unroll
        for (int k = 0; k < COO_SEG_BATCH; k++) {
            const bool live = n0 + (kb + k) * 32 + lane < n1;
            p[k]  = live ? v[k] * __ldg(a.x + (c[k] - a.base)) : T(0);
            rr[k] = r[k];
            mm[k] = __ballot_sync(0xffffffffu, live && r[k] != rn[k]);
        }
        if (kb + COO_SEG_BATCH < COO_SEG_STEPS && n0 + (kb + COO_SEG_BATCH) * 32 < n1) issue(kb + COO_SEG_BATCH);
#pragma unroll
        for (int k = 0; k < COO_SEG_BATCH; k++) {
            const T pk = p[k]; const int rk = rr[k]; const unsigned m = mm[k];
            if (m == 0u) { acc += pk; continue; }             // the whole step lies inside one run
            const int e1 = __ffs(m) - 1, ek = 31 - __clz(m);
            const T t1 = coo_warp_allsum(acc + (lane <= e1 ? pk : T(0)));
            T q = (lane > e1 && lane <= ek) ? pk : T(0);
            if (m & (m - 1u)) {                               // more runs end: segmented inclusive scan
                const unsigned below = m & ((1u << lane) - 1u);
                const int dist = (lane > e1 && lane <= ek) ? lane - (32 - __clz(below)) : 0;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    if (__ballot_sync(0xffffffffu, dist >= d) == 0u) break;
                    const T t = __shfl_up_sync(0xffffffffu, q, d);
                    if (dist >= d) q += t;
                }
            }
            if ((m >> lane) & 1u) atomicAdd(a.y + (rk - a.base), alpha * (lane == e1 ? t1 : q));
            acc = lane > ek ? pk : T(0);
        }
    }
}

template <typename T>
static int launch_coo(cudaStream_t stream, int64_t rows, int64_t nnz, const void* row, const void* col, const void* val,
                      int base, const void* alpha, const void* beta, int on_device, const void* x, void* y) {
    Scalars<T> s;
    if (on_device) { s.alpha = T(0); s.beta = T(0); s.alpha_dev = (const T*)alpha; s.beta_dev = (const T*)beta; }
    else { s.alpha = *(const T*)alpha; s.beta = *(const T*)beta; s.alpha_dev = nullptr; s.beta_dev = nullptr; }
    {
        const int threads = 256;
        int64_t blocks = (rows + threads - 1) / threads;
        if (blocks > 148 * 16) blocks = 148 * 16;
        scale_y_kernel<T><<<(unsigned)blocks, threads, 0, stream>>>((T*)y, rows, s);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
    }
    if (nnz > 0) {
        CooArgs<T> a;
        a.row = (const int*)row; a.col = (const int*)col; a.val = (const T*)val; a.x = (const T*)x; a.y = (T*)y;
        a.base = base; a.nnz = (int)nnz; a.s = s;
        a.vec_ok = (((uintptr_t)row | (uintptr_t)col | (uintptr_t)val) & 15) == 0;
        if (config().coo_kernel == 0) {
            const unsigned blocks = (unsigned)((nnz + COO_TILE - 1) / COO_TILE);
            coo_tile_kernel<T><<<blocks, COO_BLOCK, 0, stream>>>(a);
        } else {
            const int64_t per_cta = (int64_t)COO_SEG_CHUNK * (COO_BLOCK / 32);
            const unsigned blocks = (unsigned)((nnz + per_cta - 1) / per_cta);
            coo_seg_kernel<T><<<blocks, COO_BLOCK, 0, stream>>>(a);
        }
    }
    return (int)cudaGetLastError();
}

// ================================================================================================
// Sliced-ELL: one thread per row; slice-column-major storage makes the 32 lanes of a warp read 32
// consecutive values / column indices for every k (fully coalesced when sliceSize is a multiple of 32).
// A thread's whole lifetime on one row would be three dependent memory round trips (slice offsets -> val/col
// -> x) with nothing to overlap them, so the kernel is persistent and software-pipelined: every thread walks
// rows r, r + stride, r + 2*stride, ... and the slice offsets and the first SELL_UNROLL val/col entries of the
// NEXT row are already in flight into registers while the current row gathers x and accumulates.
// ================================================================================================
constexpr int SELL_BLOCK = 256;
constexpr int SELL_UNROLL = B200_SELL_UNROLL;

template <typename T>
struct SellArgs {
    const int* slice_off;
    const int* col;
    const T*   val;
    const T*   x;
    T*         y;
    int        base;
    int        rows;
    int        slice_size;
    Scalars<T> s;
};

template <typename T>
struct SellRow {
    int    width;          // entries per row in this row's slice
    size_t first;          // index of the row's k = 0 entry
    int    c[SELL_UNROLL];
    T      v[SELL_UNROLL];
};

// CS = compile-time slice size (0: use the run-time value).  With CS known the row -> slice division is a shift and
// every val/col load of a row is `base pointer + immediate`, which matters: profiled on B200 the generic version is
// bound by instruction issue (39 instructions per 32 non-zeros), not by memory.
template <typename T, int CS>
__device__ __forceinline__ void sell_issue(const SellArgs<T>& a, int row, SellRow<T>& r) {
    const int C = CS ? CS : a.slice_size;
    const int s = row / C, lane = row - s * C;
    const int beg = __ldg(a.slice_off + s) - a.base, end = __ldg(a.slice_off + s + 1) - a.base;
    r.width = (end - beg) / C;
    r.first = (size_t)beg + lane;
#pragma unroll
    for (int u = 0; u < SELL_UNROLL; u++) {
        const bool live = u < r.width;
        r.c[u] = live ? ldg_stream(a.col + r.first + (size_t)u * C) - a.base : -1;
        r.v[u] = live ? ldg_stream(a.val + r.first + (size_t)u * C) : T(0);
    }
}

template <typename T, int CS>
__global__ void __launch_bounds__(SELL_BLOCK, sizeof(T) == 4 ? B200_SELL_MIN_CTAS : (B200_SELL_MIN_CTAS > 3 ? 3 : B200_SELL_MIN_CTAS)) sell_row_kernel(const SellArgs<T> a) {
    const int stride = (int)(gridDim.x * SELL_BLOCK);
    int row = blockIdx.x * SELL_BLOCK + (int)threadIdx.x;
    if (row >= a.rows) return;
    const T alpha = a.s.a(), beta = a.s.b();
    const int C = CS ? CS : a.slice_size;
    SellRow<T> cur;
    sell_issue<T, CS>(a, row, cur);
    for (;;) {
        const int  next = row + stride;
        const bool has_next = next < a.rows;
        SellRow<T> nxt;
        T xx[SELL_UNROLL];
#pragma unroll
        for (int u = 0; u < SELL_UNROLL; u++) xx[u] = cur.c[u] >= 0 ? __ldg(a.x + cur.c[u]) : T(0);
        if (has_next) sell_issue<T, CS>(a, next, nxt);   // next row's stream in flight before this row's gathers land
        T sum = T(0);
#pragma unroll
        for (int u = 0; u < SELL_UNROLL; u++)          // padding (and slots past the width: c = -1) is skipped, not added as v * 0
            if (cur.c[u] >= 0) sum += cur.v[u] * xx[u];
        for (int k = SELL_UNROLL; k < cur.width; k += SELL_UNROLL) {      // slices wider than SELL_UNROLL
            int cc[SELL_UNROLL];
            T   vv[SELL_UNROLL], xv[SELL_UNROLL];
#pragma unroll
            for (int u = 0; u < SELL_UNROLL; u++) {
                const bool live = k + u < cur.width;
                cc[u] = live ? ldg_stream(a.col + cur.first + (size_t)(k + u) * C) - a.base : -1;
                vv[u] = live ? ldg_stream(a.val + cur.first + (size_t)(k + u) * C) : T(0);
            }
#pragma unroll
            for (int u = 0; u < SELL_UNROLL; u++) xv[u] = cc[u] >= 0 ? __ldg(a.x + cc[u]) : T(0);
#pragma unroll
            for (int u = 0; u < SELL_UNROLL; u++)
                if (cc[u] >= 0) sum += vv[u] * xv[u];
        }
        T* yp = a.y + row;
        *yp = axpby(alpha, sum, beta, yp);
        if (!has_next) break;
        row = next;
        cur = nxt;
    }
}

// Lean variant for sliceSize == 32 (one warp = one slice, so the slice width is warp-uniform): one thread per row, the
// row's W entries are loaded with immediate offsets and no predicates (switch on W for W <= 8, fully unrolled), x is
// gathered through a base pointer that already has the index base folded in.  ~10 instructions per non-zero instead
// of ~20: this kernel is bound by instruction issue, not by memory, until it is this lean (profiles/).
template <typename T, int W>
__device__ __forceinline__ T sell32_row(const int* __restrict__ cp, const T* __restrict__ vp, const T* __restrict__ xp, int base) {
    int c[W];
    T   v[W], x[W];
#pragma unroll
    for (int u = 0; u < W; u++) { c[u] = ldg_stream(cp + u * 32); v[u] = ldg_stream(vp + u * 32); }
#pragma unroll
    for (int u = 0; u < W; u++) x[u] = c[u] >= base ? __ldg(xp + c[u]) : T(0);     // padding: column -1 (+base)
    // padding contributes nothing, whatever value is stored in its slot (v * 0 would be NaN for an Inf / NaN there)
    T sum = T(0);
#pragma unroll
    for (int u = 0; u < W; u++)
        if (c[u] >= base) sum += v[u] * x[u];
    return sum;
}

template <typename T>
__global__ void __launch_bounds__(SELL_BLOCK, B200_SELL32_MIN_CTAS) sell32_kernel(const SellArgs<T> a) {
    const int row = blockIdx.x * SELL_BLOCK + (int)threadIdx.x;
    if (row >= a.rows) return;
    const int s = row >> 5, lane = row & 31;
    const int beg = __ldg(a.slice_off + s) - a.base, end = __ldg(a.slice_off + s + 1) - a.base;
    const int width = (end - beg) >> 5;
    const int* cp = a.col + beg + lane;
    const T*   vp = a.val + beg + lane;
    const T*   xp = a.x - a.base;
    T sum;
    switch (width) {                       // warp-uniform
        case 0: sum = T(0); break;
        case 1: sum = sell32_row<T, 1>(cp, vp, xp, a.base); break;
        case 2: sum = sell32_row<T, 2>(cp, vp, xp, a.base); break;
        case 3: sum = sell32_row<T, 3>(cp, vp, xp, a.base); break;
        case 4: sum = sell32_row<T, 4>(cp, vp, xp, a.base); break;
        case 5: sum = sell32_row<T, 5>(cp, vp, xp, a.base); break;
        case 6: sum = sell32_row<T, 6>(cp, vp, xp, a.base); break;
        case 7: sum = sell32_row<T, 7>(cp, vp, xp, a.base); break;
        case 8: sum = sell32_row<T, 8>(cp, vp, xp, a.base); break;
        default: {
            sum = T(0);
            int k = 0;
            for (; k + 8 <= width; k += 8) sum += sell32_row<T, 8>(cp + k * 32, vp + k * 32, xp, a.base);
            for (; k < width; k++) sum += sell32_row<T, 1>(cp + k * 32, vp + k * 32, xp, a.base);
        }
    }
    T* yp = a.y + row;
    *yp = axpby(a.s.a(), sum, a.s.b(), yp);
}

template <typename T>
static int launch_sell(cudaStream_t stream, int64_t rows, int64_t slice_size, const void* slice_off, const void* col,
                       const void* val, int base, const void* alpha, const void* beta, int on_device, const void* x,
                       void* y) {
    SellArgs<T> a;
    a.slice_off = (const int*)slice_off; a.col = (const int*)col; a.val = (const T*)val; a.x = (const T*)x; a.y = (T*)y;
    a.base = base; a.rows = (int)rows; a.slice_size = (int)slice_size;
    if (on_device) { a.s.alpha = T(0); a.s.beta = T(0); a.s.alpha_dev = (const T*)alpha; a.s.beta_dev = (const T*)beta; }
    else { a.s.alpha = *(const T*)alpha; a.s.beta = *(const T*)beta; a.s.alpha_dev = nullptr; a.s.beta_dev = nullptr; }
    // persistent grid of the generic kernel: SMs x resident CTAs, cached per (device, value type) under a lock
    static int grid_cache[64][2];
    static std::mutex mu;
    const int ti = sizeof(T) == 4 ? 0 : 1;
    int dev = 0;
    cudaGetDevice(&dev);
    int64_t persistent;
    {
        std::lock_guard<std::mutex> lk(mu);
        int& g = grid_cache[dev & 63][ti];
        if (!g) {
            int n = 1, sms = 148;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, (const void*)sell_row_kernel<T, 0>, SELL_BLOCK, 0);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            g = sms * (n < 1 ? 1 : n);
        }
        persistent = (int64_t)g * B200_SELL_WAVES;
    }
    int64_t blocks = (rows + SELL_BLOCK - 1) / SELL_BLOCK;
    if (blocks > persistent) blocks = persistent;
    if (slice_size == 32 && !config().sell_generic) {
        const int64_t all = (rows + SELL_BLOCK - 1) / SELL_BLOCK;
        sell32_kernel<T><<<(unsigned)all, SELL_BLOCK, 0, stream>>>(a);
    } else {
        sell_row_kernel<T, 0><<<(unsigned)blocks, SELL_BLOCK, 0, stream>>>(a);
    }
    return (int)cudaGetLastError();
}

}  // namespace b200

using namespace b200;

extern "C" {

size_t b200spmv_coo_workspace_bytes(int64_t, int64_t) { return 0; }

int b200spmv_coo_mv(void* stream, int dtype, int64_t rows, int64_t cols, int64_t nnz, const void* row_ind,
                    const void* col_ind, const void* values, int32_t base, const void* alpha, const void* beta,
                    int scalars_on_device, const void* x, void* y, void* /*workspace*/) {
    if (rows < 0 || cols < 0 || nnz < 0 || nnz > INT32_MAX - 4 || rows > INT32_MAX - 1 || !alpha || !beta) return -1;
    if (rows == 0) return 0;
    if (!y || (nnz > 0 && (!row_ind || !col_ind || !values || !x))) return -1;
    if (dtype == 0)
        return launch_coo<float>((cudaStream_t)stream, rows, nnz, row_ind, col_ind, values, base, alpha, beta,
                                 scalars_on_device, x, y);
    if (dtype == 1)
        return launch_coo<double>((cudaStream_t)stream, rows, nnz, row_ind, col_ind, values, base, alpha, beta,
                                  scalars_on_device, x, y);
    return -1;
}

size_t b200spmv_sell_workspace_bytes(int64_t, int64_t, int64_t) { return 0; }

int b200spmv_sell_mv(void* stream, int dtype, int64_t rows, int64_t cols, int64_t slice_size, const void* slice_offsets,
                     const void* col_ind, const void* values, int32_t base, const void* alpha, const void* beta,
                     int scalars_on_device, const void* x, void* y, void* /*workspace*/) {
    if (rows < 0 || cols < 0 || slice_size <= 0 || rows > INT32_MAX - 1 || !alpha || !beta) return -1;
    if (rows == 0) return 0;
    if (!y || !slice_offsets) return -1;
    if (dtype == 0)
        return launch_sell<float>((cudaStream_t)stream, rows, slice_size, slice_offsets, col_ind, values, base, alpha,
                                  beta, scalars_on_device, x, y);
    if (dtype == 1)
        return launch_sell<double>((cudaStream_t)stream, rows, slice_size, slice_offsets, col_ind, values, base, alpha,
                                   beta, scalars_on_device, x, y);
    return -1;
}

}  // extern "C"
