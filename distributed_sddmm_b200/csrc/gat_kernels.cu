// gat_kernels.cu -- the device operations the GAT (include/hnh/gat.hpp; reference gat.hpp:84-113) needs beyond the
// SDDMM / SpMM path.  Forward: LeakyReLU on an edge-value vector, ReLU of a head's output written into its column
// window of the layer output, and the dense projection X * W.  Backward: the ReLU-window and LeakyReLU derivatives and
// the two transposed products W_grad = X^T H_grad and X_grad (+)= H_grad W^T.
//
// The projection is this library's own fp64 GEMM (dgemm_dmma_kernel below): C = A B for a tall A (rows of the
// graph) and a small B (the head's weight matrix), on the fp64 tensor-core path (mma.sync m8n8k4, DMMA) with
// shared-memory tiles.  Blackwell's tcgen05 has no fp64 kind, so mma.sync IS the fp64 tensor path on sm_100a.
#include <algorithm>

#include "hnh_b200.h"
#include "launch.h"

namespace {

using hnh::check_cuda;
using hnh::count_launch;
using hnh::set_error;

constexpr int kThreads = 256;

// x -> max(x, 0) + alpha * min(x, 0)
__global__ void leaky_relu_kernel(double *__restrict__ dst, const double *__restrict__ src, int64_t n, double alpha) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const double x = src[i];
        dst[i] = fmax(x, 0.0) + fmin(x, 0.0) * alpha;
    }
}

// dst[i, col0 + j] = max(src[i, j], 0): dst has ld_dst columns, src is rows x cols, contiguous
__global__ void relu_cols_kernel(double *__restrict__ dst, int64_t ld_dst, int64_t col0, const double *__restrict__ src,
                                 int64_t rows, int64_t cols) {
    const int64_t n = rows * cols;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
        const int64_t i = t / cols, j = t - i * cols;
        dst[i * ld_dst + col0 + j] = fmax(src[t], 0.0);
    }
}

// dst[i, j] = grad[i, col0 + j] if out[i, col0 + j] > 0 else 0: grad and out have ld columns, dst is rows x cols
__global__ void relu_cols_backward_kernel(double *__restrict__ dst, const double *__restrict__ grad,
                                          const double *__restrict__ out, int64_t ld, int64_t col0, int64_t rows,
                                          int64_t cols) {
    const int64_t n = rows * cols;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) {
        const int64_t i = t / cols, j = t - i * cols;
        const int64_t at = i * ld + col0 + j;
        dst[t] = out[at] > 0.0 ? grad[at] : 0.0;
    }
}

// x -> 1 if x > 0 else alpha: the derivative of leaky_relu_kernel, with torch's value alpha at 0
__global__ void leaky_relu_slope_kernel(double *__restrict__ dst, const double *__restrict__ src, int64_t n, double alpha) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = src[i] > 0.0 ? 1.0 : alpha;
}

int grid_for_elements(int64_t n, int *grid) {
    int sms = 0;
    int rc = hnh::device_sm_count(&sms);
    if (rc) return rc;
    const int64_t want = (n + (int64_t)kThreads * 4 - 1) / ((int64_t)kThreads * 4);
    *grid = (int)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sms * 8));
    return HNH_OK;
}

// ---- fp64 GEMM on DMMA ---------------------------------------------------------------------------------
// C (m x n) = A (m x k) B (k x n), all row-major, contiguous.  CTA tile 64 x 64, 4 warps of 32 x 32 (4 x 4 DMMA tiles
// of 8 x 8), K in steps of 16 through shared memory.  Fragment layout of mma.m8n8k4.f64 (PTX ISA): with g = lane / 4,
// t = lane % 4:  A[g][t],  B[t][g],  C[g][2t], C[g][2t + 1].  The shared-memory row strides (20 and 68 doubles) put
// the 16 lanes of a half-warp on 16 different bank pairs for both fragment loads.  Edges are zero-filled on load and
// masked on store, so any m, n, k >= 1 works.
constexpr int GM = 64, GN = 64, GK = 16, GA_LD = GK + 4, GB_LD = GN + 4;

__device__ __forceinline__ void dmma_8x8x4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(128)
dgemm_dmma_kernel(double *__restrict__ C, const double *__restrict__ A, const double *__restrict__ B, int64_t m, int n, int k) {
    __shared__ double As[GM][GA_LD];
    __shared__ double Bs[GK][GB_LD];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wr = (warp >> 1) * 32, wc = (warp & 1) * 32;  // this warp's 32 x 32 corner inside the CTA tile
    const int col_tiles = (n + GN - 1) / GN;
    const int64_t row_tiles = (m + GM - 1) / GM;
    for (int64_t tile = blockIdx.x; tile < row_tiles * col_tiles; tile += gridDim.x) {
        const int64_t row0 = (tile / col_tiles) * GM;
        const int col0 = (int)(tile % col_tiles) * GN;
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
        for (int k0 = 0; k0 < k; k0 += GK) {
            __syncthreads();  // the previous K step has been consumed
            for (int e = threadIdx.x; e < GM * GK; e += 128) {
                const int r = e / GK, c = e % GK;
                const int64_t gr = row0 + r;
                As[r][c] = (gr < m && k0 + c < k) ? A[gr * k + k0 + c] : 0.0;
            }
            for (int e = threadIdx.x; e < GK * GN; e += 128) {
                const int r = e / GN, c = e % GN;
                Bs[r][c] = (k0 + r < k && col0 + c < n) ? B[(int64_t)(k0 + r) * n + col0 + c] : 0.0;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < GK; kk += 4) {
                double a[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; i++) a[i] = As[wr + i * 8 + g][kk + t];
#pragma unroll
                for (int j = 0; j < 4; j++) b[j] = Bs[kk + t][wc + j * 8 + g];
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) dmma_8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int64_t r = row0 + wr + i * 8 + g;
            if (r >= m) continue;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int c = col0 + wc + j * 8 + 2 * t;
                if (c < n) C[r * n + c] = acc[i][j][0];
                if (c + 1 < n) C[r * n + c + 1] = acc[i][j][1];
            }
        }
    }
}

// ---- transposed fp64 GEMMs of the backward pass, on the same DMMA fragments ------------------------------
// C (k x n) = A^T B for A (m x k), B (m x n), the reduction running over the long graph-row dimension m.  The CTA at
// (output tile, chunk) reduces rows [chunk * rows_per_chunk, ...) of A and B into one 64 x 64 output tile; both operands
// are staged as [row of the chunk][output index] (stride 68, as Bs above), so a[i] = As[kk + t][wr + i * 8 + g] is the
// A[g][t] fragment of A^T.  With one chunk the tile goes straight to C, otherwise to partials[chunk] for
// sum_partials_kernel.  No atomics: the result depends on (m, n, k) only, and repeated calls agree bit for bit.
__global__ void __launch_bounds__(128)
dgemm_tn_dmma_kernel(double *__restrict__ P, const double *__restrict__ A, const double *__restrict__ B, int64_t m, int n,
                     int k, int64_t rows_per_chunk) {
    __shared__ double As[GK][GB_LD];
    __shared__ double Bs[GK][GB_LD];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wr = (warp >> 1) * 32, wc = (warp & 1) * 32;
    const int col_tiles = (n + GN - 1) / GN;
    const int row0 = (int)(blockIdx.x / col_tiles) * GM;  // output rows: columns of A
    const int col0 = (int)(blockIdx.x % col_tiles) * GN;  // output columns: columns of B
    const int64_t r_lo = (int64_t)blockIdx.y * rows_per_chunk;
    const int64_t r_hi = min(m, r_lo + rows_per_chunk);
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
    for (int64_t r0 = r_lo; r0 < r_hi; r0 += GK) {
        __syncthreads();
        for (int e = threadIdx.x; e < GK * GM; e += 128) {
            const int r = e / GM, c = e % GM;
            const int64_t gr = r0 + r;
            As[r][c] = (gr < r_hi && row0 + c < k) ? A[gr * k + row0 + c] : 0.0;
        }
        for (int e = threadIdx.x; e < GK * GN; e += 128) {
            const int r = e / GN, c = e % GN;
            const int64_t gr = r0 + r;
            Bs[r][c] = (gr < r_hi && col0 + c < n) ? B[gr * n + col0 + c] : 0.0;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GK; kk += 4) {
            double a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; i++) a[i] = As[kk + t][wr + i * 8 + g];
#pragma unroll
            for (int j = 0; j < 4; j++) b[j] = Bs[kk + t][wc + j * 8 + g];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) dmma_8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
    double *out = P + (int64_t)blockIdx.y * k * n;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int r = row0 + wr + i * 8 + g;
        if (r >= k) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int c = col0 + wc + j * 8 + 2 * t;
            if (c < n) out[(int64_t)r * n + c] = acc[i][j][0];
            if (c + 1 < n) out[(int64_t)r * n + c + 1] = acc[i][j][1];
        }
    }
}

// C[i] = sum over chunks of P[chunk][i], chunks in ascending order
__global__ void sum_partials_kernel(double *__restrict__ C, const double *__restrict__ P, int64_t size, int chunks) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < size; i += stride) {
        double s = 0.0;
        for (int c = 0; c < chunks; c++) s += P[(int64_t)c * size + i];
        C[i] = s;
    }
}

// C (m x n) = A (m x k) B^T (+ C when accumulate) for B (n x k): dgemm_dmma_kernel with B staged as [column of C][K]
// (stride 20, as As), so b[j] = Bs[wc + j * 8 + g][kk + t] is the B[t][g] fragment of B^T.
__global__ void __launch_bounds__(128)
dgemm_nt_dmma_kernel(double *__restrict__ C, const double *__restrict__ A, const double *__restrict__ B, int64_t m, int n,
                     int k, int accumulate) {
    __shared__ double As[GM][GA_LD];
    __shared__ double Bs[GN][GA_LD];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int wr = (warp >> 1) * 32, wc = (warp & 1) * 32;
    const int col_tiles = (n + GN - 1) / GN;
    const int64_t row_tiles = (m + GM - 1) / GM;
    for (int64_t tile = blockIdx.x; tile < row_tiles * col_tiles; tile += gridDim.x) {
        const int64_t row0 = (tile / col_tiles) * GM;
        const int col0 = (int)(tile % col_tiles) * GN;
        double acc[4][4][2];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[i][j][0] = acc[i][j][1] = 0.0;
        for (int k0 = 0; k0 < k; k0 += GK) {
            __syncthreads();
            for (int e = threadIdx.x; e < GM * GK; e += 128) {
                const int r = e / GK, c = e % GK;
                const int64_t gr = row0 + r;
                As[r][c] = (gr < m && k0 + c < k) ? A[gr * k + k0 + c] : 0.0;
            }
            for (int e = threadIdx.x; e < GN * GK; e += 128) {
                const int r = e / GK, c = e % GK;
                Bs[r][c] = (col0 + r < n && k0 + c < k) ? B[(int64_t)(col0 + r) * k + k0 + c] : 0.0;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < GK; kk += 4) {
                double a[4], b[4];
#pragma unroll
                for (int i = 0; i < 4; i++) a[i] = As[wr + i * 8 + g][kk + t];
#pragma unroll
                for (int j = 0; j < 4; j++) b[j] = Bs[wc + j * 8 + g][kk + t];
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < 4; j++) dmma_8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const int64_t r = row0 + wr + i * 8 + g;
            if (r >= m) continue;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int c = col0 + wc + j * 8 + 2 * t;
                if (c < n) C[r * n + c] = accumulate ? C[r * n + c] + acc[i][j][0] : acc[i][j][0];
                if (c + 1 < n) C[r * n + c + 1] = accumulate ? C[r * n + c + 1] + acc[i][j][1] : acc[i][j][1];
            }
        }
    }
}

// Split of the TN reduction: about kTnCtas CTAs in all, at least kTnMinRows rows each.  A function of the shape only,
// so that the summation order (and with it every bit of the result) does not depend on the device.
constexpr int64_t kTnCtas = 1024, kTnMinRows = 256;

}  // namespace

extern "C" {

int hnh_leaky_relu_f64(double *dst, const double *src, int64_t n, double alpha, void *stream) {
    if (n < 0) return set_error(HNH_E_INVALID, "hnh_leaky_relu_f64: negative size");
    if (n == 0) return HNH_OK;
    if (!dst || !src) return set_error(HNH_E_INVALID, "hnh_leaky_relu_f64: null pointer");
    int grid;
    int rc = grid_for_elements(n, &grid);
    if (rc) return rc;
    leaky_relu_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(dst, src, n, alpha);
    count_launch(1);
    return check_cuda(cudaGetLastError(), "leaky_relu_kernel launch");
}

int hnh_relu_cols_f64(double *dst, int64_t ld_dst, int64_t col0, const double *src, int64_t rows, int64_t cols, void *stream) {
    if (rows < 0 || cols < 0 || col0 < 0 || ld_dst < col0 + cols)
        return set_error(HNH_E_INVALID, "hnh_relu_cols_f64: column window [%lld, %lld) outside a row of %lld",
                         (long long)col0, (long long)(col0 + cols), (long long)ld_dst);
    if (rows == 0 || cols == 0) return HNH_OK;
    if (!dst || !src) return set_error(HNH_E_INVALID, "hnh_relu_cols_f64: null pointer");
    int grid;
    int rc = grid_for_elements(rows * cols, &grid);
    if (rc) return rc;
    relu_cols_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(dst, ld_dst, col0, src, rows, cols);
    count_launch(1);
    return check_cuda(cudaGetLastError(), "relu_cols_kernel launch");
}

int hnh_dgemm_f64(double *C, const double *A, const double *B, int64_t m, int64_t n, int64_t k, void *stream) {
    if (m < 0 || n < 0 || k < 0 || m > INT32_MAX || n > INT32_MAX || k > INT32_MAX)
        return set_error(HNH_E_INVALID, "hnh_dgemm_f64: bad shape %lld x %lld x %lld", (long long)m, (long long)n, (long long)k);
    if (m == 0 || n == 0) return HNH_OK;
    if (!C || (k > 0 && (!A || !B))) return set_error(HNH_E_INVALID, "hnh_dgemm_f64: null pointer");
    if (k == 0)
        return check_cuda(cudaMemsetAsync(C, 0, sizeof(double) * (size_t)(m * n), (cudaStream_t)stream), "cudaMemsetAsync");
    int sms = 0;
    int rc = hnh::device_sm_count(&sms);
    if (rc) return rc;
    const int64_t tiles = ((m + GM - 1) / GM) * ((n + GN - 1) / GN);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, (int64_t)sms * 8));
    dgemm_dmma_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(C, A, B, m, (int)n, (int)k);
    rc = check_cuda(cudaGetLastError(), "dgemm_dmma_kernel launch");
    if (rc) return rc;
    count_launch(1);
    return HNH_OK;
}

int hnh_relu_cols_backward_f64(double *dst, const double *grad, const double *out, int64_t ld, int64_t col0, int64_t rows,
                               int64_t cols, void *stream) {
    if (rows < 0 || cols < 0 || col0 < 0 || ld < col0 + cols)
        return set_error(HNH_E_INVALID, "hnh_relu_cols_backward_f64: column window [%lld, %lld) outside a row of %lld",
                         (long long)col0, (long long)(col0 + cols), (long long)ld);
    if (rows == 0 || cols == 0) return HNH_OK;
    if (!dst || !grad || !out) return set_error(HNH_E_INVALID, "hnh_relu_cols_backward_f64: null pointer");
    int grid;
    int rc = grid_for_elements(rows * cols, &grid);
    if (rc) return rc;
    relu_cols_backward_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(dst, grad, out, ld, col0, rows, cols);
    count_launch(1);
    return check_cuda(cudaGetLastError(), "relu_cols_backward_kernel launch");
}

int hnh_leaky_relu_slope_f64(double *dst, const double *src, int64_t n, double alpha, void *stream) {
    if (n < 0) return set_error(HNH_E_INVALID, "hnh_leaky_relu_slope_f64: negative size");
    if (n == 0) return HNH_OK;
    if (!dst || !src) return set_error(HNH_E_INVALID, "hnh_leaky_relu_slope_f64: null pointer");
    int grid;
    int rc = grid_for_elements(n, &grid);
    if (rc) return rc;
    leaky_relu_slope_kernel<<<grid, kThreads, 0, (cudaStream_t)stream>>>(dst, src, n, alpha);
    count_launch(1);
    return check_cuda(cudaGetLastError(), "leaky_relu_slope_kernel launch");
}

int hnh_dgemm_tn_f64(double *C, const double *A, const double *B, int64_t m, int64_t n, int64_t k, void *stream) {
    if (m < 0 || n < 0 || k < 0 || n > INT32_MAX || k > INT32_MAX || n * k > INT32_MAX)
        return set_error(HNH_E_INVALID, "hnh_dgemm_tn_f64: bad shape %lld x %lld x %lld", (long long)m, (long long)n, (long long)k);
    if (n == 0 || k == 0) return HNH_OK;
    if (!C || (m > 0 && (!A || !B))) return set_error(HNH_E_INVALID, "hnh_dgemm_tn_f64: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (m == 0) return check_cuda(cudaMemsetAsync(C, 0, sizeof(double) * (size_t)(n * k), st), "cudaMemsetAsync");
    const int64_t tiles = ((k + GM - 1) / GM) * ((n + GN - 1) / GN);
    const int64_t want = std::max<int64_t>(1, std::min<int64_t>((m + kTnMinRows - 1) / kTnMinRows, kTnCtas / tiles));
    const int64_t rows_per_chunk = ((m + want - 1) / want + GK - 1) / GK * GK;
    const int chunks = (int)((m + rows_per_chunk - 1) / rows_per_chunk);
    double *partial = C;
    int rc;
    if (chunks > 1) {
        // per-call scratch, stream-ordered (as hnh_squared_norm_f64)
        rc = check_cuda(cudaMallocAsync((void **)&partial, sizeof(double) * (size_t)(chunks * n * k), st), "cudaMallocAsync");
        if (rc) return rc;
    }
    dgemm_tn_dmma_kernel<<<dim3((unsigned)tiles, (unsigned)chunks), 128, 0, st>>>(partial, A, B, m, (int)n, (int)k, rows_per_chunk);
    count_launch(1);
    rc = check_cuda(cudaGetLastError(), "dgemm_tn_dmma_kernel launch");
    if (chunks > 1) {
        if (!rc) {
            const int grid = (int)std::min<int64_t>((n * k + kThreads - 1) / kThreads, 1024);
            sum_partials_kernel<<<grid, kThreads, 0, st>>>(C, partial, n * k, chunks);
            count_launch(1);
            rc = check_cuda(cudaGetLastError(), "sum_partials_kernel launch");
        }
        cudaError_t e = cudaFreeAsync(partial, st);
        if (!rc) rc = check_cuda(e, "cudaFreeAsync");
    }
    return rc;
}

int hnh_dgemm_nt_f64(double *C, const double *A, const double *B, int64_t m, int64_t n, int64_t k, double beta,
                     void *stream) {
    if (m < 0 || n < 0 || k < 0 || n > INT32_MAX || k > INT32_MAX)
        return set_error(HNH_E_INVALID, "hnh_dgemm_nt_f64: bad shape %lld x %lld x %lld", (long long)m, (long long)n, (long long)k);
    if (beta != 0.0 && beta != 1.0) return set_error(HNH_E_INVALID, "hnh_dgemm_nt_f64: beta must be 0 or 1, not %g", beta);
    if (m == 0 || n == 0) return HNH_OK;
    if (!C || (k > 0 && (!A || !B))) return set_error(HNH_E_INVALID, "hnh_dgemm_nt_f64: null pointer");
    if (k == 0)
        return beta == 1.0 ? HNH_OK
                           : check_cuda(cudaMemsetAsync(C, 0, sizeof(double) * (size_t)(m * n), (cudaStream_t)stream), "cudaMemsetAsync");
    int sms = 0;
    int rc = hnh::device_sm_count(&sms);
    if (rc) return rc;
    const int64_t tiles = ((m + GM - 1) / GM) * ((n + GN - 1) / GN);
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, (int64_t)sms * 8));
    dgemm_nt_dmma_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(C, A, B, m, (int)n, (int)k, beta == 1.0);
    count_launch(1);
    return check_cuda(cudaGetLastError(), "dgemm_nt_dmma_kernel launch");
}

}  // extern "C"
