// spmm_csr.cu -- CSR x dense  C = alpha*A*B + beta*C  on B200 (sm_100a), fp32 / fp64, int32 indices (SURVEY.md 8(f)-1,
// BASELINE.json configs[4]).  Replaces cusparse::csrmm kernels behind cusparseSpMM for CSR descriptors with
// opA = opB = NON_TRANSPOSE (call site: cuSPARSE/spmm_csr/spmm_csr_example.c:105-132; golden C at :64-66).
//
// One warp per row of A and per panel of 64 columns of B / C.  The row's (col, val) pairs are loaded 32 at a time with
// one coalesced instruction each and broadcast with shuffles; for every non-zero the 32 lanes read 64 consecutive
// entries of row `col` of B.  With ROW-major B that is one contiguous 256 B (fp32) segment per non-zero -- the fast case
// SURVEY.md names; with COLUMN-major B (the sample's layout) the same code walks B with stride ldb: correct, one sector per
// element -- measured on BASELINE.json configs[4] (2M x 2M, 32 per row, n = 64, fp32): 72 ms, the closed library 32 ms,
// against 3.6 ms (closed: 5.3 ms) for the same product with row-major operands.  So the sample's layout takes two extra steps
// (round 2): B is transposed once per call into the caller's externalBuffer (cusparseSpMM_bufferSize asks for cols*n
// elements; +1 GB of traffic = 0.2 ms on that config) and read row-major from there, and a column-major C is produced by
// spmm_csr_ctile_kernel, which parks a 32-row x 64-column block of C in shared memory and writes it out as 128 B column
// segments.  C is written once, alpha / beta applied in the epilogue (beta == 0 never reads C).  No tensor cores:
// 2 flop per 4-byte B element fetched.  Bytes per product (row-major, fp32): nnz*8 (A) + nnz*n*4 (B rows, mostly L2 hits
// when B fits) + rows*n*4 (C).
#include "spmv_common.cuh"
#include "config.h"
#include "../../include/b200spmv.h"

namespace b200 {

constexpr int SPMM_WARPS = 8;       // rows per CTA
constexpr int SPMM_PANEL = 64;      // columns of B / C per warp pass (2 per lane)

template <typename T>
struct SpmmArgs {
    const int* off;
    const int* col;
    const T*   val;
    const T*   B;
    T*         C;
    int        base, rows, n;
    long long  sbk, sbj;            // B(k, j) = B[k * sbk + j * sbj]
    long long  sci, scj;            // C(i, j) = C[i * sci + j * scj]
    Scalars<T> s;
};

// One warp-row of the product: acc0 / acc1 = row `row` of A times columns ja / jb of B (B(k, j) = B[k * sbk + j * sbj]).
template <typename T>
__device__ __forceinline__ void spmm_row(const SpmmArgs<T>& a, int row, int lane, int ja, int jb, bool la, bool lb, T& acc0, T& acc1) {
    const int b = __ldg(a.off + row) - a.base, e = __ldg(a.off + row + 1) - a.base;
    const T* Ba = a.B + (long long)ja * a.sbj;
    const T* Bb = a.B + (long long)jb * a.sbj;
    for (int p = b; p < e; p += 32) {
        const int  i = p + lane;
        const int  c = i < e ? ldg_stream(a.col + i) - a.base : 0;
        const T    v = i < e ? ldg_stream(a.val + i) : T(0);
        const int  cnt = min(32, e - p);
        for (int t = 0; t < cnt; t += 4) {                       // four B rows in flight per lane
            int kk[4];
            T   vv[4], b0[4], b1[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                kk[u] = __shfl_sync(0xffffffffu, c, (t + u) & 31);
                vv[u] = __shfl_sync(0xffffffffu, v, (t + u) & 31);
            }
            // Slots t + u >= cnt lie past the row's end (c = 0, v = 0) and must not touch B: 0 * B(0, j) is NaN when row 0 of
            // B holds an Inf or a NaN.  The predicate is warp-uniform.
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const long long ro = (long long)kk[u] * a.sbk;
                const bool in_row = t + u < cnt;
                b0[u] = (la && in_row) ? __ldg(Ba + ro) : T(0);
                b1[u] = (lb && in_row) ? __ldg(Bb + ro) : T(0);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) { acc0 += vv[u] * b0[u]; acc1 += vv[u] * b1[u]; }
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(32 * SPMM_WARPS) spmm_csr_kernel(const SpmmArgs<T> a) {
    const int lane = (int)threadIdx.x & 31;
    const int row = blockIdx.x * SPMM_WARPS + ((int)threadIdx.x >> 5);
    if (row >= a.rows) return;                                   // warp-uniform
    const int j0 = blockIdx.y * SPMM_PANEL;
    const int ja = j0 + lane, jb = j0 + 32 + lane;               // my two columns
    const bool la = ja < a.n, lb = jb < a.n;
    T acc0 = T(0), acc1 = T(0);
    spmm_row(a, row, lane, ja, jb, la, lb, acc0, acc1);
    const T alpha = a.s.a(), beta = a.s.b();
    if (la) { T* cp = a.C + (long long)row * a.sci + (long long)ja * a.scj; *cp = axpby(alpha, acc0, beta, cp); }
    if (lb) { T* cp = a.C + (long long)row * a.sci + (long long)jb * a.scj; *cp = axpby(alpha, acc1, beta, cp); }
}

// Column-major C (sci == 1): a CTA computes 32 rows x 64 columns of C (each of its 8 warps 4 rows, one after the other),
// parks them transposed in shared memory, and writes every column's 32 consecutive rows as one coalesced 128 B / 256 B store.
constexpr int SPMM_TILE_ROWS = 32;
template <typename T>
__global__ void __launch_bounds__(32 * SPMM_WARPS) spmm_csr_ctile_kernel(const SpmmArgs<T> a) {
    __shared__ T tile[SPMM_PANEL][SPMM_TILE_ROWS + 1];
    const int lane = (int)threadIdx.x & 31, warp = (int)threadIdx.x >> 5;
    const int row0 = blockIdx.x * SPMM_TILE_ROWS;
    const int j0 = blockIdx.y * SPMM_PANEL;
    const int ja = j0 + lane, jb = j0 + 32 + lane;
    const bool la = ja < a.n, lb = jb < a.n;
    constexpr int PER_WARP = SPMM_TILE_ROWS / SPMM_WARPS;
#pragma unroll 1
    for (int rr = 0; rr < PER_WARP; rr++) {
        const int rl = warp * PER_WARP + rr, row = row0 + rl;
        T acc0 = T(0), acc1 = T(0);
        if (row < a.rows) spmm_row(a, row, lane, ja, jb, la, lb, acc0, acc1);       // warp-uniform
        tile[lane][rl] = acc0;                                                       // bank (lane + rl) % 32: conflict-free
        tile[32 + lane][rl] = acc1;
    }
    __syncthreads();
    const T alpha = a.s.a(), beta = a.s.b();
    const int row = row0 + lane;
    constexpr int COLS_PER_WARP = SPMM_PANEL / SPMM_WARPS;
#pragma unroll
    for (int q = 0; q < COLS_PER_WARP; q++) {
        const int jj = warp * COLS_PER_WARP + q, j = j0 + jj;
        if (j < a.n && row < a.rows) {
            T* cp = a.C + (long long)row * a.sci + (long long)j * a.scj;
            *cp = axpby(alpha, tile[jj][lane], beta, cp);
        }
    }
}

// B (cols x n, column-major, leading dimension ldb) -> Bt (cols x n, row-major, tight): 32 x 32 tiles through shared memory
template <typename T>
__global__ void __launch_bounds__(256) spmm_transpose_b_kernel(const T* __restrict__ B, long long ldb, T* __restrict__ Bt, int cols, int n) {
    __shared__ T tile[32][33];
    const int tx = (int)threadIdx.x & 31, ty = (int)threadIdx.x >> 5;
    const int k0 = blockIdx.x * 32, j0 = blockIdx.y * 32;
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
        const int k = k0 + tx, j = j0 + ty + i;
        if (k < cols && j < n) tile[ty + i][tx] = B[(long long)j * ldb + k];
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
        const int k = k0 + ty + i, j = j0 + tx;
        if (k < cols && j < n) Bt[(long long)k * n + j] = tile[tx][ty + i];
    }
}

constexpr int SPMM_MIN_N_FOR_TRANSPOSE = 4;      // below that a strided walk over column-major B costs less than the extra pass

template <typename T>
static int launch_spmm(cudaStream_t stream, int64_t rows, int64_t n, const void* off, const void* col, const void* val, int base,
                       const void* alpha, const void* beta, int on_device, const void* B, int64_t ldb, int b_row_major,
                       void* C, int64_t ldc, int c_row_major, int64_t cols, void* workspace) {
    SpmmArgs<T> a;
    a.off = (const int*)off; a.col = (const int*)col; a.val = (const T*)val; a.B = (const T*)B; a.C = (T*)C;
    a.base = base; a.rows = (int)rows; a.n = (int)n;
    if (!b_row_major && workspace && n >= SPMM_MIN_N_FOR_TRANSPOSE && cols > 0) {
        // the sample's layout: one pass turns B into a row-major copy in the caller's buffer
        const dim3 tg((unsigned)((cols + 31) / 32), (unsigned)((n + 31) / 32));
        spmm_transpose_b_kernel<T><<<tg, 256, 0, stream>>>((const T*)B, (long long)ldb, (T*)workspace, (int)cols, (int)n);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
        a.B = (const T*)workspace; b_row_major = 1; ldb = n;
    }
    a.sbk = b_row_major ? ldb : 1; a.sbj = b_row_major ? 1 : ldb;
    a.sci = c_row_major ? ldc : 1; a.scj = c_row_major ? 1 : ldc;
    if (on_device) { a.s.alpha = T(0); a.s.beta = T(0); a.s.alpha_dev = (const T*)alpha; a.s.beta_dev = (const T*)beta; }
    else { a.s.alpha = *(const T*)alpha; a.s.beta = *(const T*)beta; a.s.alpha_dev = nullptr; a.s.beta_dev = nullptr; }
    if (!c_row_major && b_row_major) {               // column-major C from row-major B: tiles of C transposed in shared memory
        const dim3 grid((unsigned)((rows + SPMM_TILE_ROWS - 1) / SPMM_TILE_ROWS), (unsigned)((n + SPMM_PANEL - 1) / SPMM_PANEL));
        spmm_csr_ctile_kernel<T><<<grid, 32 * SPMM_WARPS, 0, stream>>>(a);
        return (int)cudaGetLastError();
    }
    const dim3 grid((unsigned)((rows + SPMM_WARPS - 1) / SPMM_WARPS), (unsigned)((n + SPMM_PANEL - 1) / SPMM_PANEL));
    spmm_csr_kernel<T><<<grid, 32 * SPMM_WARPS, 0, stream>>>(a);
    return (int)cudaGetLastError();
}

}  // namespace b200

using namespace b200;

extern "C" {

size_t b200spmm_csr_workspace_bytes(int dtype, int64_t cols, int64_t n, int b_row_major) {
    if (b_row_major || n < SPMM_MIN_N_FOR_TRANSPOSE || cols <= 0 || n <= 0) return 0;
    return ((size_t)cols * (size_t)n * (dtype == 1 ? 8 : 4) + 255) / 256 * 256;
}

int b200spmm_csr_ws(void* stream, int dtype, int64_t rows, int64_t cols, int64_t n, int64_t nnz, const void* row_offsets,
                    const void* col_ind, const void* values, int32_t base, const void* alpha, const void* beta,
                    int scalars_on_device, const void* B, int64_t ldb, int b_row_major, void* C, int64_t ldc,
                    int c_row_major, void* workspace) {
    if (rows < 0 || cols < 0 || n < 0 || nnz < 0 || !alpha || !beta) return -1;
    if (rows == 0 || n == 0) return 0;
    if (rows > INT32_MAX - 64 || cols > INT32_MAX - 64 || n > INT32_MAX - 64 || nnz > INT32_MAX - 65536 || (n + SPMM_PANEL - 1) / SPMM_PANEL > 65535) return -1;
    if (!row_offsets || !C || (nnz > 0 && (!col_ind || !values || !B))) return -1;
    if (ldb < (b_row_major ? n : cols) || ldc < (c_row_major ? n : rows)) return -1;
    if (workspace && ((uintptr_t)workspace & 15)) workspace = nullptr;
    if (nnz == 0) workspace = nullptr;                       // B may be NULL then: nothing to transpose
    if (dtype == 0)
        return launch_spmm<float>((cudaStream_t)stream, rows, n, row_offsets, col_ind, values, base, alpha, beta, scalars_on_device,
                                  B, ldb, b_row_major, C, ldc, c_row_major, cols, workspace);
    if (dtype == 1)
        return launch_spmm<double>((cudaStream_t)stream, rows, n, row_offsets, col_ind, values, base, alpha, beta, scalars_on_device,
                                   B, ldb, b_row_major, C, ldc, c_row_major, cols, workspace);
    return -1;
}

int b200spmm_csr(void* stream, int dtype, int64_t rows, int64_t cols, int64_t n, int64_t nnz, const void* row_offsets,
                 const void* col_ind, const void* values, int32_t base, const void* alpha, const void* beta,
                 int scalars_on_device, const void* B, int64_t ldb, int b_row_major, void* C, int64_t ldc, int c_row_major) {
    return b200spmm_csr_ws(stream, dtype, rows, cols, n, nnz, row_offsets, col_ind, values, base, alpha, beta, scalars_on_device, B, ldb,
                           b_row_major, C, ldc, c_row_major, nullptr);
}

}  // extern "C"
