/*
 * hnh_b200.h -- C ABI of the B200-native local kernels (libhnh_b200.so).
 *
 * This is the drop-in boundary under the reference's C++ plugin interface
 * `KernelImplementation` (reference sparse_kernels.h:15-79).  Every entry point is
 * `extern "C"`, takes plain pointers and sizes (no torch / Eigen / MKL types), enqueues
 * its work on the CUDA stream passed as `void *stream` (NULL = legacy default stream) and
 * returns 0 on success or a negative HNH_E_* code -- it never prints-and-exits the way the
 * reference does (sparse_kernels.cpp:75-83).  `hnh_last_error_string()` describes the last
 * failure on the calling thread.
 *
 * Unless a name ends in `_host`, all data pointers are DEVICE pointers.
 * Dense operands are row-major, contiguous, leading dimension = r (reference common.h:13,
 * `DenseMatrix`), fp64.  Index arrays are int64 (MKL_INT under -DMKL_ILP64, reference
 * CMakeLists.txt:37).  CSR arrays are the four vectors of the reference's `CSRHandle`
 * (SpmatLocal.hpp:55-62): values, col_idx, rowStart (rows+1 entries), row_idx (expanded).
 *
 * There is no CPU fallback behind this ABI: without a CUDA device every compute entry
 * point fails with HNH_E_CUDA.
 */
#ifndef HNH_B200_H
#define HNH_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HNH_OK 0
#define HNH_E_INVALID (-1) /* bad argument (null pointer, negative size, r <= 0 ...)     */
#define HNH_E_CUDA (-2)    /* a CUDA runtime call or kernel launch failed                */
#define HNH_E_MODE (-3)    /* block transposition does not match the requested SpMM mode */
#define HNH_E_ALLOC (-4)   /* device or pinned-host allocation failed                    */
#define HNH_E_COMM (-5)    /* NCCL / transport failure                                   */

/* flags (bit set) */
#define HNH_FLAG_DEFAULT 0
#define HNH_FLAG_FORCE_GENERIC 1 /* use the any-r scalar kernel (testing)                  */
#define HNH_FLAG_FORCE_DIRECT 2  /* use the direct-load row kernels instead of TMA-staged */
/* BETA0: overwrite instead of accumulate -- sddmm: values = dot; spmm: Y = CSR*X;
 * fused: values = dot, Out = result (Out may then alias X).  Equivalent to zeroing the
 * output first (setValuesConstant(0) / setZero(), SpmatLocal.hpp:595-605,
 * distributed_sparse.h:275) but without the extra pass over memory. */
#define HNH_FLAG_BETA0 4
/* fused only: overwrite just the values (each block is visited once per FusedMM) or just Out */
#define HNH_FLAG_BETA0_VALUES 16
#define HNH_FLAG_BETA0_OUT 32
/* sddmm / fused, r in {128, 256}: stage the row-side factor tile with bulk asynchronous copies
 * (cp.async.bulk + mbarrier, SASS UBLKCP) instead of direct loads.  Without this flag the library picks
 * per kernel from measurements (TMA for SDDMM and for the r = 256 overwrite-fused kernel; direct loads
 * otherwise); HNH_FLAG_FORCE_DIRECT or env HNH_TMA=0 force the direct-load kernels, HNH_TMA=1 the
 * TMA-staged ones. */
#define HNH_FLAG_TMA_STAGE 64
/* experimental: per-warp TMA slots (no block barrier); never selected automatically */
#define HNH_FLAG_TMA_WARP 128
/* hnh_sddmm_scaled_f64 with scaled_out: the block's values receive scale * dot as well (default: the plain dot) */
#define HNH_FLAG_SCALE_VALUES 256

/* ABI / build identification. */
int hnh_abi_version(void);
const char *hnh_build_info(void);
const char *hnh_last_error_string(void);
/* Number of kernel launches issued through this library by the calling process so far
 * (bench.py reports the delta over its timed region as `gpu_launches`). */
uint64_t hnh_launch_count(void);

/* ---- K1: SDDMM -- replaces StandardKernel::sddmm_local (sparse_kernels.cpp:13-57) ------
 * values[i] += sum_k X[row(i), k] * Y[col_idx[i], k]   for every nonzero i of the block.
 * (X, Y) are already role-resolved: (A, B) for a non-transposed block, (B, A) for a
 * transposed one (sparse_kernels.cpp:29-38).  `rows` = number of CSR rows of the block,
 * rowStart[rows] == nnz.  Accumulates (+=), exactly like the reference; callers zero
 * `values` first (SpmatLocal::setValuesConstant, SpmatLocal.hpp:595-605).
 * nnz == 0 or rows == 0 is a successful no-op (sparse_kernels.cpp:25-27). */
int hnh_sddmm_f64(const int64_t *rowStart, const int64_t *col_idx, double *values,
                  int64_t rows, int64_t nnz, const double *X, const double *Y, int r,
                  int flags, void *stream);
/* The same with the Hadamard epilogue of the reference's `SValues.cwiseProduct(getCSRValues())`
 * (15D_dense_shift.hpp:364-368, SpmatLocal.hpp:571-593) folded in: `scale` is aligned with `values`
 * (scale[i] belongs to nonzero i of this block).  scaled_out != NULL: values[i] = dot (as above) and
 * scaled_out[i] = scale[i] * dot.  scaled_out == NULL: values[i] = scale[i] * dot.  scale == NULL is
 * hnh_sddmm_f64.  HNH_FLAG_SCALE_VALUES: with scaled_out, values[i] = scale[i] * dot too.  With accumulation
 * (no BETA0) the old value is added to the dot BEFORE scaling. */
int hnh_sddmm_scaled_f64(const int64_t *rowStart, const int64_t *col_idx, double *values, int64_t rows,
                         int64_t nnz, const double *X, const double *Y, int r, int flags, const double *scale,
                         double *scaled_out, void *stream);

/* Same operation driven by the expanded COO arrays the reference kernel actually reads
 * (`row_idx[i]`, `col_idx[i]`, sparse_kernels.cpp:45-47); needs no rowStart. */
int hnh_sddmm_coo_f64(const int64_t *row_idx, const int64_t *col_idx, double *values,
                      int64_t nnz, const double *X, const double *Y, int r, int flags,
                      void *stream);

/* ---- K2: SpMM -- replaces StandardKernel::spmm_local (sparse_kernels.cpp:59-127) -------
 * Y[rows x r] += CSR[rows x *] * X   (alpha = beta = 1, row-major, ld = r: the
 * mkl_sparse_d_mm call at sparse_kernels.cpp:95-120).  X is gathered by col_idx.  The
 * kernel never bounds-checks col_idx against a column count (the reference declares too few
 * columns in 15D_sparse_shift.hpp:132). */
int hnh_spmm_f64(const int64_t *rowStart, const int64_t *col_idx, const double *values,
                 int64_t rows, int64_t nnz, const double *X, double *Y, int r, int flags,
                 void *stream);

/* ---- K3: fused SDDMM -> SpMM on one block ------------------------------------------------
 * Replaces the two back-to-back triple_function calls of the fusion-2 loop body
 * (15D_dense_shift.hpp:203-217):  values[i] += X[row(i)] . Y[col(i)];  then
 * Out[row] += sum_{i in row} values[i] * Y[col(i)]   -- with ONE gather of each Y row. */
int hnh_fused_f64(const int64_t *rowStart, const int64_t *col_idx, double *values,
                  int64_t rows, int64_t nnz, const double *X, const double *Y, double *Out,
                  int r, int flags, void *stream);
/* The same with the caller's S values folded in (the Hadamard product the reference applies between its SDDMM and
 * SpMM passes, distributed_sparse.h:289-312): values[i] = scale[i] * dot, Out += sum_i values[i] * Y[col_i], and
 * scaled_out[i] (optional) = values[i] -- the user-visible SDDMM result.  Needs HNH_FLAG_BETA0_VALUES, a table width
 * and aligned operands (HNH_E_INVALID otherwise: use the separate calls). */
int hnh_fused_scaled_f64(const int64_t *rowStart, const int64_t *col_idx, double *values, int64_t rows,
                         int64_t nnz, const double *X, const double *Y, double *Out, int r, int flags,
                         const double *scale, double *scaled_out, void *stream);

/* ---- K4: value plumbing (SpmatLocal.hpp:571-605, 15D_dense_shift.hpp:366) -------------- */
int hnh_fill_f64(double *dst, int64_t n, double value, void *stream);
/* dst[i] = uniform(-1,1) from a counter-based hash of (seed, i) -- DenseMatrix::setRandom
 * (als_conjugate_gradients.cpp:143-146) */
int hnh_random_uniform_f64(double *dst, int64_t n, uint64_t seed, void *stream);
/* dst[i] = a[i] * b[i]  (VectorXd::cwiseProduct of SValues and getCSRValues()) */
int hnh_hadamard_f64(double *dst, const double *a, const double *b, int64_t n, void *stream);
/* row_idx[i] = CSR row of nonzero i (SpmatLocal.hpp:139-147,160-163) */
int hnh_expand_row_idx(const int64_t *rowStart, int64_t rows, int64_t nnz, int64_t *row_idx,
                       void *stream);

/* ---- dense row algebra used between fusedSpMM calls by the ALS-CG caller
 *      (als_conjugate_gradients.cpp:9-29,99-138) ------------------------------------------ */
/* out[i] = sum_k A[i,k] * B[i,k]   (batch_dot_product) */
int hnh_batch_dot_f64(double *out, const double *A, const double *B, int64_t rows, int r,
                      void *stream);
/* D[i,k] = C[i,k] + alpha * s[i] * M[i,k]   (X += scale_matrix_rows(s, M) and friends;
 * s may be NULL meaning all-ones; C may be NULL meaning zero; D may alias C or M) */
int hnh_row_axpy_f64(double *D, const double *C, double alpha, const double *s,
                     const double *M, int64_t rows, int r, void *stream);
/* elementwise vector helpers: out = (a + ca) / (b + cb); b == NULL: out = a + ca */
int hnh_vec_quotient_f64(double *out, const double *a, double ca, const double *b, double cb,
                         int64_t n, void *stream);
/* dst = alpha * x + beta * y elementwise (y may be NULL when beta == 0) */
int hnh_axpby_f64(double *dst, double alpha, const double *x, double beta, const double *y,
                  int64_t n, void *stream);
/* *out (device scalar) = sum x[i]^2 */
int hnh_squared_norm_f64(double *out, const double *x, int64_t n, void *stream);

/* ---- GAT forward pass helpers (reference gat.hpp:84-113; include/hnh/gat.hpp) --------------
 * dst[i] = max(src[i], 0) + alpha * min(src[i], 0)   (gat.hpp:98; dst may alias src) */
int hnh_leaky_relu_f64(double *dst, const double *src, int64_t n, double alpha, void *stream);
/* dst[i, col0 + j] = max(src[i, j], 0) for a rows x cols src and a dst with ld_dst columns
 * (buffers[i+1].middleCols(j * w, w) = A.array().max(0), gat.hpp:104) */
int hnh_relu_cols_f64(double *dst, int64_t ld_dst, int64_t col0, const double *src, int64_t rows,
                      int64_t cols, void *stream);
/* C (m x n) = A (m x k) * B (k x n), all row-major and contiguous (buffers[i] * wMats[j],
 * gat.hpp:90).  This library's own kernel: fp64 tensor-core MMA (mma.sync m8n8k4) over shared-memory tiles. */
int hnh_dgemm_f64(double *C, const double *A, const double *B, int64_t m, int64_t n, int64_t k,
                  void *stream);

/* ---- GAT backward pass helpers (include/hnh/gat.hpp, GAT::backwardPass) ----------------------
 * dst[i, j] = grad[i, col0 + j] if out[i, col0 + j] > 0, else 0 (ReLU'(0) = 0): the gradient of a head's
 * column window.  grad and out have ld columns, dst is rows x cols, contiguous. */
int hnh_relu_cols_backward_f64(double *dst, const double *grad, const double *out, int64_t ld, int64_t col0,
                               int64_t rows, int64_t cols, void *stream);
/* dst[i] = 1 if src[i] > 0, else alpha: the derivative of hnh_leaky_relu_f64 (alpha at 0; dst may alias src) */
int hnh_leaky_relu_slope_f64(double *dst, const double *src, int64_t n, double alpha, void *stream);
/* C (k x n) = A^T B for A (m x k) and B (m x n), row-major; m (the graph rows) is the long dimension.  DMMA tiles over
 * row chunks, partial tiles summed in a fixed order: deterministic, repeated calls agree bit for bit.  m == 0 gives
 * C = 0.  Allocates its scratch stream-ordered. */
int hnh_dgemm_tn_f64(double *C, const double *A, const double *B, int64_t m, int64_t n, int64_t k, void *stream);
/* C (m x n) = A B^T + beta * C for A (m x k) and B (n x k), row-major; beta is 0 or 1 (HNH_E_INVALID otherwise). */
int hnh_dgemm_nt_f64(double *C, const double *A, const double *B, int64_t m, int64_t n, int64_t k, double beta,
                     void *stream);

/* ---- host-side setup helpers (untimed; HOST pointers) --------------------------------------
 * hnh_er_generate_host replaces the CombBLAS Graph500 generator call of
 * SpmatLocal::loadTuples(false, logM, nnz_per_row) (SpmatLocal.hpp:499-516): rows
 * [row_lo,row_hi) of the seeded N x N Erdos-Renyi matrix, sorted (row, col), unique, values 1.
 * Returns the tuple count (>= 0) or a negative HNH_E_* code. */
int64_t hnh_er_generate_host(int logM, int nnz_per_row, uint64_t seed, int64_t row_lo,
                             int64_t row_hi, uint64_t *rows_out, uint64_t *cols_out,
                             double *vals_out, int64_t capacity);
/* hnh_coo_to_csr_host replaces the MKL inspector sequence of the CSRLocal constructor
 * (SpmatLocal.hpp:117-147): COO -> CSR, optional transpose, stable.  rowStart has
 * (transpose ? cols : rows) + 1 entries; row_idx (expanded stored-row index) may be NULL. */
int hnh_coo_to_csr_host(int64_t rows, int64_t cols, int64_t nnz, const uint64_t *r,
                        const uint64_t *c, const double *v, int transpose, int64_t *rowStart,
                        int64_t *col_idx, int64_t *row_idx, double *values);

/* Device versions of the two helpers above (DEVICE pointers; untimed setup; they synchronise `stream`
 * before returning).  Output is bit-identical with the host versions: the generator is a pure function
 * of (seed, row, k), the CSR order is a stable sort by stored row.  nnz_per_row <= 128; one block holds
 * fewer than 2^31 entries. */
int64_t hnh_er_generate_device(int logM, int nnz_per_row, uint64_t seed, int64_t row_lo,
                               int64_t row_hi, uint64_t *rows_out, uint64_t *cols_out,
                               double *vals_out, int64_t capacity, void *stream);
int hnh_coo_to_csr_device(int64_t rows, int64_t cols, int64_t nnz, const uint64_t *r,
                          const uint64_t *c, const double *v, int transpose, int64_t *rowStart,
                          int64_t *col_idx, int64_t *row_idx, double *values, void *stream);

/* Device-resident tuple pipeline of the setup path (SoA tuples r / c / v in HBM; reference: host vectors of
 * spcoord_t, SpmatLocal.hpp:389-462).  All synchronise `stream` before returning; fewer than 2^31 tuples per call.
 *  - bucket_by_owner: owner(i) = table[rb * table_cols + cb] with (rb, cb) = (r/rows_in_block, c/cols_in_block), or
 *    (c/rows_in_block, r/cols_in_block) when `transpose` (NonzeroDistribution::getOwner, SpmatLocal.hpp:45-52); the
 *    table is a HOST array filled from the distribution's blockOwner().  Output: the tuples grouped by owner in
 *    input order (stable), r and c exchanged when `transpose`; starts_host[nbuckets + 1] = segment offsets.
 *  - sort_colmajor: in place, ascending (c, r), ties in input order (the order redistribute_nonzeros leaves,
 *    SpmatLocal.hpp:458).  max_r / max_c bound the keys (number of radix bits).
 *  - mod: r %= mod_r, c %= mod_c (0 = leave).   - block_starts: first position with c >= k * block_width. */
int hnh_tuples_bucket_by_owner_device(const uint64_t *r, const uint64_t *c, const double *v, int64_t n, int transpose,
                                      int64_t rows_in_block, int64_t cols_in_block, const int *owner_table_host,
                                      int64_t table_rows, int64_t table_cols, int nbuckets, uint64_t *r_out,
                                      uint64_t *c_out, double *v_out, int64_t *starts_host, void *stream);
int hnh_tuples_sort_colmajor_device(uint64_t *r, uint64_t *c, double *v, int64_t n, uint64_t max_r, uint64_t max_c,
                                    void *stream);
int hnh_tuples_mod_device(uint64_t *r, uint64_t *c, int64_t n, uint64_t mod_r, uint64_t mod_c, void *stream);
int hnh_tuples_block_starts_device(const uint64_t *c_sorted, int64_t n, uint64_t block_width, int divisions,
                                   int64_t *starts_host, void *stream);

/* ---- host-buffer entry points (pinned or pageable HOST pointers) -------------------------
 * One call = H2D of the dense operands and values, the kernel(s), D2H of the results, all
 * inside the call; the block's CSR structure is taken from a resident handle made once with
 * hnh_block_create_host (the reference also builds its CSR once, SpmatLocal.hpp:78-188).
 * These are what bench.py's `e2e` leg times. */
typedef struct hnh_block hnh_block_t;
int hnh_block_create_host(const int64_t *rowStart, const int64_t *col_idx, int64_t rows,
                          int64_t cols, int64_t nnz, int r_max, hnh_block_t **out);
void hnh_block_destroy(hnh_block_t *blk);
/* op: 0 = sddmm (values_io += X.Y), 1 = spmm (Out += CSR*Y with values_io), 2 = fused.
 * X: rows x r, Y: cols x r, Out: rows x r (op 1, 2), values_io: nnz.
 * run_flags: HNH_RUN_ZERO_VALUES = start from values == 0 on the device instead of copying
 * values_io in (SpmatLocal::setValuesConstant(0), SpmatLocal.hpp:595-605);
 * HNH_RUN_ZERO_OUT = start from Out == 0 on the device instead of copying Out in
 * (`localA.setZero()`, distributed_sparse.h:275,304). */
#define HNH_RUN_ZERO_VALUES 1
#define HNH_RUN_ZERO_OUT 2
int hnh_block_run_host(hnh_block_t *blk, int op, const double *X, const double *Y,
                       double *values_io, double *Out, int r, int run_flags, void *stream);

/* One-shot forms with HOST pointers for a reference-side KernelImplementation that keeps the
 * reference's host data structures (include/hnh/reference_plugin/cuda_kernel.h): operands are
 * mirrored on the device for the call, the result is copied back, the call synchronises.
 * hnh_sddmm_coo_host: values[i] += X[row_idx[i]] . Y[col_idx[i]]  (StandardKernel::sddmm_local,
 * sparse_kernels.cpp:44-55; X has x_rows rows, Y has y_rows rows, both r wide).
 * hnh_spmm_host: Y[rows x r] += CSR * X  (the mkl_sparse_d_mm call, sparse_kernels.cpp:95-120;
 * X has x_rows rows). */
int hnh_sddmm_coo_host(const int64_t *row_idx, const int64_t *col_idx, double *values, int64_t nnz,
                       const double *X, int64_t x_rows, const double *Y, int64_t y_rows, int r);
int hnh_spmm_host(const int64_t *rowStart, const int64_t *col_idx, const double *values,
                  int64_t rows, int64_t nnz, const double *X, int64_t x_rows, double *Y, int r);

#ifdef __cplusplus
}
#endif
#endif /* HNH_B200_H */
