/*
 * hnh_b200_driver.h -- C ABI over the C++ host classes of libhnh_b200.so
 * (SpmatLocal, FlexibleGrid, Distributed_Sparse and its 1.5D / 2.5D subclasses,
 * benchmark_algorithm), for callers that are not C++: bench.py and the tests bind it with
 * ctypes.  C++ callers include the headers under include/hnh/ directly -- they carry the
 * reference's own class and method names (see INTEGRATION.md).
 *
 * All functions return 0 or a negative HNH_E_* code (hnh_b200.h); hnh_last_error_string()
 * describes the failure.  One process = one rank = one GPU.
 */
#ifndef HNH_B200_DRIVER_H
#define HNH_B200_DRIVER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HNHD_NCCL_ID_BYTES 128

/* Caller-supplied transport on HOST buffers (the "External" transport of hnh/comm.h).  Each
 * callback returns 0 on success.  `comm` is an integer handle; 0 is the world.  These map
 * one-to-one onto the MPI calls of the reference (MPI_Sendrecv distributed_sparse.h:351-361,
 * MPI_Allgather 15D_dense_shift.hpp:194, MPI_Reduce_scatter :240, MPI_Alltoallv
 * SpmatLocal.hpp:451, MPI_Barrier, MPI_Comm_split FlexibleGrid.hpp:80-88). */
typedef struct hnhd_external_transport {
    void *ctx;
    int (*sendrecv)(void *ctx, int comm, const void *sbuf, size_t sbytes, int dst, void *rbuf,
                    size_t rbytes, int src);
    int (*allgather)(void *ctx, int comm, const void *sbuf, void *rbuf, size_t bytes_each);
    int (*reduce_scatter_f64)(void *ctx, int comm, const double *sbuf, double *rbuf,
                              size_t count_each);
    int (*allreduce_f64)(void *ctx, int comm, double *buf, size_t count);
    int (*alltoallv)(void *ctx, int comm, const void *sbuf, const size_t *sbytes,
                     const size_t *sdispls, void *rbuf, const size_t *rbytes,
                     const size_t *rdispls);
    int (*barrier)(void *ctx, int comm);
    int (*split)(void *ctx, int comm, int color, int key, int *new_comm, int *new_rank,
                 int *new_size);
} hnhd_external_transport_t;

/* ---- world (replaces MPI_Init / MPI_Finalize, bench_erdos_renyi.cpp:20,120) ---------------- */
int hnhd_init_self(void);
int hnhd_nccl_unique_id(char out[HNHD_NCCL_ID_BYTES]);
int hnhd_init_nccl(int rank, int world_size, const char unique_id[HNHD_NCCL_ID_BYTES]);
int hnhd_init_external(int rank, int world_size, const hnhd_external_transport_t *cb);
int hnhd_finalize(void);
int hnhd_world_rank(void);
int hnhd_world_size(void);
int hnhd_barrier(void);
int hnhd_device_synchronize(void);

/* ---- SpmatLocal ----------------------------------------------------------------------------- */
typedef struct hnhd_spmat hnhd_spmat_t;
/* SpmatLocal::loadTuples(false, logM, nnz_per_row, "") (SpmatLocal.hpp:467-533) with the
 * repo's seeded Erdos-Renyi generator; every rank generates its 1-D row slice. */
int hnhd_spmat_load_er(int logM, int nnz_per_row, uint64_t seed, hnhd_spmat_t **out);
/* SpmatLocal::loadTuples(true, -1, -1, filename): MatrixMarket coordinate file (general / symmetric, real /
 * integer / pattern); every rank keeps a share of the entries (SpmatLocal.hpp:479-491 reads with CombBLAS). */
int hnhd_spmat_load_file(const char *filename, hnhd_spmat_t **out);
/* Arbitrary local tuples of a global M x N matrix (any distribution over the ranks). */
int hnhd_spmat_from_tuples(uint64_t M, uint64_t N, const uint64_t *rows, const uint64_t *cols,
                           const double *vals, int64_t n_local, hnhd_spmat_t **out);
int hnhd_spmat_info(const hnhd_spmat_t *S, uint64_t *M, uint64_t *N, uint64_t *dist_nnz,
                    int64_t *local_tuples);
int hnhd_spmat_tuples(const hnhd_spmat_t *S, uint64_t *rows, uint64_t *cols, double *vals,
                      int64_t capacity);
void hnhd_spmat_destroy(hnhd_spmat_t *S);

/* ---- Distributed_Sparse subclasses ---------------------------------------------------------- */
typedef struct hnhd_alg hnhd_alg_t;
/* name: "15d_fusion1" | "15d_fusion2" | "15d_sparse" | "25d_dense_replicate" |
 * "25d_sparse_replicate"  (the selectors of benchmark_dist.cpp:45-82).  The kernel plugged in
 * is the library's StandardKernel (CUDA). */
int hnhd_alg_create(const char *name, hnhd_spmat_t *S, int R, int c, hnhd_alg_t **out);
void hnhd_alg_destroy(hnhd_alg_t *alg);

typedef struct hnhd_alg_dims {
    int64_t M, N, R;
    int p, c;
    int localArows, localAcols, localBrows, localBcols;
    int64_t s_values, st_values; /* like_S_values / like_ST_values lengths */
    int r_split;
    int grid_i, grid_j, grid_k;
    int n_a_submatrices, n_b_submatrices;
} hnhd_alg_dims_t;
int hnhd_alg_dims(hnhd_alg_t *alg, hnhd_alg_dims_t *out);
/* aSubmatrices / bSubmatrices (distributed_sparse.h:57-58): 4 ints each
 * (topRow, leftCol, rowCount, colCount). which: 0 = A, 1 = B. */
int hnhd_alg_submatrices(hnhd_alg_t *alg, int which, int *out4, int capacity);
/* JSON text of json_algorithm_info() / json_perf_statistics() (distributed_sparse.h:131-179,
 * 245-261).  Collective.  Returns the length written (excluding NUL) or a negative code. */
/* Wall-clock seconds of the setup phases of this process so far (tuple generation, redistribution, COO -> CSR), as
 * a JSON object {phase: seconds}; reset != 0 clears the counters afterwards. */
int hnhd_setup_times_json(char *out, size_t capacity, int reset);
int hnhd_alg_info_json(hnhd_alg_t *alg, char *out, size_t capacity);
int hnhd_alg_perf_json(hnhd_alg_t *alg, char *out, size_t capacity);
int hnhd_alg_reset_timers(hnhd_alg_t *alg);

/* Local CSR blocks of S (which = 0) or ST (which = 1), copied to HOST arrays: for tests.
 * block_count -> number of blocks; for each block: rows, cols, nnz, transpose, is_null. */
int hnhd_alg_block_count(hnhd_alg_t *alg, int which);
int hnhd_alg_block_meta(hnhd_alg_t *alg, int which, int block, int64_t *rows, int64_t *cols,
                        int64_t *nnz, int *transpose, int *is_null);
int hnhd_alg_block_arrays(hnhd_alg_t *alg, int which, int block, int64_t *rowStart,
                          int64_t *col_idx, int64_t *row_idx, double *values);

/* ---- resident dense matrices / value vectors (DenseMatrix / VectorXd on the device) -------- */
typedef struct hnhd_dense hnhd_dense_t;
typedef struct hnhd_vec hnhd_vec_t;
int hnhd_dense_create(int64_t rows, int64_t cols, double value, hnhd_dense_t **out);
int hnhd_dense_like(hnhd_alg_t *alg, int which /*0=A,1=B*/, double value, hnhd_dense_t **out);
int hnhd_dense_fill(hnhd_dense_t *m, double value);
int hnhd_dense_dummy_initialize(hnhd_alg_t *alg, hnhd_dense_t *m, int which); /* :322-346 */
int hnhd_dense_from_host(hnhd_dense_t *m, const double *host); /* rows*cols doubles */
int hnhd_dense_to_host(const hnhd_dense_t *m, double *host);
int hnhd_dense_shape(const hnhd_dense_t *m, int64_t *rows, int64_t *cols);
/* Device pointer of the matrix storage.  NOT stable across operations: spmm / fusedSpMM / ring shifts may return
 * their result by swapping the matrix's storage with an internal buffer (instead of the reference's copy-back,
 * common.h:88-92), after which an earlier pointer refers to recycled memory.  Re-query after every operation. */
void *hnhd_dense_data(hnhd_dense_t *m);
void hnhd_dense_destroy(hnhd_dense_t *m);
int hnhd_vec_create(int64_t n, double value, hnhd_vec_t **out);
int hnhd_vec_like(hnhd_alg_t *alg, int which /*0=S,1=ST*/, double value, hnhd_vec_t **out);
int hnhd_vec_fill(hnhd_vec_t *v, double value);
int hnhd_vec_from_host(hnhd_vec_t *v, const double *host);
int hnhd_vec_to_host(const hnhd_vec_t *v, double *host);
int64_t hnhd_vec_size(const hnhd_vec_t *v);
void hnhd_vec_destroy(hnhd_vec_t *v);

/* ---- the public operations (distributed_sparse.h:266-320) ----------------------------------- */
#define HNHD_OP_SDDMM_A 0
#define HNHD_OP_SDDMM_B 1
#define HNHD_OP_SPMM_A 2
#define HNHD_OP_SPMM_B 3
#define HNHD_OP_FUSED_A 4 /* fusedSpMM(A, B, S, result, Amat) */
#define HNHD_OP_FUSED_B 5
#define HNHD_OP_INITIAL_SHIFT 6 /* aux = KernelMode (0 sddmmA,1 spmmA,2 spmmB,3 sddmmB) */
#define HNHD_OP_DE_SHIFT 7
/* Enqueues the operation (stream-ordered; returns before the GPU finishes).  svals / result
 * may be NULL where the operation does not use them (spmm: result unused). */
int hnhd_alg_op(hnhd_alg_t *alg, int op, hnhd_dense_t *A, hnhd_dense_t *B, hnhd_vec_t *svals,
                hnhd_vec_t *result, int aux);

/* fusedSpMM on HOST operands (Distributed_Sparse::fusedSpMM_host, include/hnh/distributed_sparse.h): hostA / hostB
 * are this rank's local shards in (preferably pinned) host memory, hostOut receives the SpMM result; A and B are
 * the device staging matrices.  mode: 0 = Amat, 1 = Bmat.  chunk_rows > 0 sets the row chunk of the upload /
 * kernel / download pipeline the 1.5D dense-shift algorithm runs on one rank, 0 keeps the default, < 0 turns the
 * pipeline off (copy in, fusedSpMM, copy out).  Returns after hostOut is complete. */
int hnhd_alg_fused_host(hnhd_alg_t *alg, hnhd_dense_t *A, hnhd_dense_t *B, hnhd_vec_t *svals, hnhd_vec_t *result,
                        const double *hostA, const double *hostB, double *hostOut, int mode, int64_t chunk_rows);

/* CUDA-event timing on the library's compute stream: start, ..., stop -> milliseconds. */
int hnhd_timer_start(void);
int hnhd_timer_stop(double *ms_out);

/* benchmark_algorithm (benchmark_dist.cpp:26-167): constructs the algorithm, runs
 * `trials` timed FusedMM (or SDDMM+SpMM when fused == 0) calls after `warmup` untimed ones,
 * appends the reference-schema JSON record to output_file on rank 0 (NULL = no file) and
 * returns the record in json_out. */
int hnhd_benchmark_algorithm(hnhd_spmat_t *S, const char *algorithm_name, const char *output_file,
                             int fused, int R, int c, const char *app, int trials, int warmup,
                             char *json_out, size_t capacity);

/* Distributed_ALS on `alg` (als_conjugate_gradients.cpp): artificial ground truth, initializeEmbeddings(),
 * residual, `steps` alternating cg_optimizer(Amat, 10) / cg_optimizer(Bmat, 10) rounds, residual again.
 * out2 = {residual before, residual after} (world-reduced, identical on every rank).  Collective. */
int hnhd_als_residuals(hnhd_alg_t *alg, int steps, double *out2);

/* The same alternating rounds on CALLER inputs, for parity tests against the reference's Distributed_ALS: ground
 * truth = SDDMM of the local shards hostAgt / hostBgt over the all-ones pattern (as the constructor builds it,
 * als_conjugate_gradients.cpp:166-186), embeddings = hostA0 / hostB0 (instead of initializeEmbeddings()'s random
 * draw), `steps` rounds of cg_optimizer(Amat, cg_iters); cg_optimizer(Bmat, cg_iters).  out2 = residual before /
 * after; hostA_out / hostB_out (may be NULL) receive the local embeddings.  Collective. */
int hnhd_als_run(hnhd_alg_t *alg, const double *hostAgt, const double *hostBgt, const double *hostA0,
                 const double *hostB0, int steps, int cg_iters, double *out2, double *hostA_out,
                 double *hostB_out);

/* ---- GAT (include/hnh/gat.hpp; reference gat.hpp:26-113) ------------------------------------
 * layers3: n_layers triples (input_features, features_per_head, num_heads).  The object keeps a
 * pointer to `alg`, which must outlive it.  buffer 0 is the network input, buffer i + 1 the output
 * of layer i; weights are input_width x head_width, row-major, as hnhd_gat_weight_shape reports. */
typedef struct hnhd_gat hnhd_gat_t;
int hnhd_gat_create(hnhd_alg_t *alg, int n_layers, const int *layers3, double leaky_relu_alpha,
                    hnhd_gat_t **out);
int hnhd_gat_weight_shape(hnhd_gat_t *g, int layer, int head, int64_t *rows, int64_t *cols);
int hnhd_gat_set_weight(hnhd_gat_t *g, int layer, int head, const double *host);
int hnhd_gat_buffer_shape(hnhd_gat_t *g, int buffer, int64_t *rows, int64_t *cols);
int hnhd_gat_set_input(hnhd_gat_t *g, const double *host);          /* buffer 0 */
int hnhd_gat_get_buffer(hnhd_gat_t *g, int buffer, double *host);   /* synchronises */
int hnhd_gat_forward(hnhd_gat_t *g);                                /* forwardPass(); stream-ordered */
/* Backward pass (GAT::backwardPass) from dL/d(last buffer) = host_output_grad (this rank's rows, the shape of the last
 * buffer).  Needs the forward pass of the current weights in the buffers; overwrites the gradients.  Collective: the
 * weight gradients are summed over all ranks.  HNH_E_INVALID, with nothing enqueued, where
 * hnhd_gat_supports_backward() is 0; the error string says why. */
int hnhd_gat_supports_backward(hnhd_gat_t *g);                      /* 1, 0, or a negative code */
int hnhd_gat_backward(hnhd_gat_t *g, const double *host_output_grad);
int hnhd_gat_get_weight_grad(hnhd_gat_t *g, int layer, int head, double *host); /* weight shape; synchronises */
int hnhd_gat_get_input_grad(hnhd_gat_t *g, double *host);           /* shape of buffer 0; synchronises */
int hnhd_gat_get_weight(hnhd_gat_t *g, int layer, int head, double *host);      /* synchronises */
int hnhd_gat_sgd_step(hnhd_gat_t *g, double lr);                    /* W -= lr * W_grad for every weight */
void hnhd_gat_destroy(hnhd_gat_t *g);

#ifdef __cplusplus
}
#endif
#endif /* HNH_B200_DRIVER_H */
