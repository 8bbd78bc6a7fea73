// driver.cpp -- extern "C" driver ABI (include/hnh_b200_driver.h) over the C++ host classes.
#include "hnh_b200_driver.h"

#include <cstring>
#include <memory>

#include "hnh/15D_dense_shift.hpp"
#include "hnh/15D_sparse_shift.hpp"
#include "hnh/25D_cannon_dense.hpp"
#include "hnh/25D_cannon_sparse.hpp"
#include "hnh/als_conjugate_gradients.h"
#include "hnh/benchmark_dist.hpp"
#include "hnh/distributed_sparse.h"
#include "hnh/gat.hpp"
#include "hnh_b200.h"
#include "launch.h"

Distributed_Sparse *hnh_make_algorithm(const string &name, SpmatLocal *spmat, int R, int c, KernelImplementation *k);

struct hnhd_spmat {
    SpmatLocal m;
};
struct hnhd_alg {
    StandardKernel kernel;
    std::unique_ptr<Distributed_Sparse> alg;
};
struct hnhd_dense {
    DenseMatrix m;
};
struct hnhd_vec {
    VectorXd v;
};
struct hnhd_gat {
    std::unique_ptr<GAT> g;
};

namespace {

// run f, translating C++ exceptions into error codes
template <class F>
int guarded(F f) {
    try {
        f();
        return HNH_OK;
    } catch (const hnh::Error &e) {
        return hnh::set_error(e.code, "%s", e.what());
    } catch (const std::bad_alloc &) {
        return hnh::set_error(HNH_E_ALLOC, "out of host memory");
    } catch (const std::exception &e) {
        return hnh::set_error(HNH_E_INVALID, "%s", e.what());
    }
}

int copy_json(const json &j, char *out, size_t capacity) {
    const string s = j.dump();
    if (!out || capacity < s.size() + 1)
        return hnh::set_error(HNH_E_INVALID, "json buffer too small (%zu needed)", s.size() + 1);
    std::memcpy(out, s.c_str(), s.size() + 1);
    return (int)s.size();
}

cudaEvent_t g_t0 = nullptr, g_t1 = nullptr;

}  // namespace

extern "C" {

int hnhd_init_self(void) { return guarded([] { hnh::Comm::init_self(); }); }
int hnhd_nccl_unique_id(char out[HNHD_NCCL_ID_BYTES]) { return guarded([&] { hnh::Comm::nccl_unique_id(out); }); }
int hnhd_init_nccl(int rank, int world_size, const char uid[HNHD_NCCL_ID_BYTES]) {
    return guarded([&] { hnh::Comm::init_nccl(rank, world_size, uid); });
}
int hnhd_init_external(int rank, int world_size, const hnhd_external_transport_t *cb) {
    return guarded([&] { hnh::Comm::init_external(rank, world_size, cb); });
}
int hnhd_finalize(void) {
    return guarded([] {
        if (hnh::Runtime::get().has_device()) hnh::Runtime::get().sync_all();
        hnh::Comm::finalize();
    });
}
int hnhd_world_rank(void) { return hnh::Comm::world_initialised() ? hnh::Comm::world()->rank() : -1; }
int hnhd_world_size(void) { return hnh::Comm::world_initialised() ? hnh::Comm::world()->size() : -1; }
int hnhd_barrier(void) { return guarded([] { hnh::Comm::world()->barrier(); }); }
int hnhd_device_synchronize(void) { return guarded([] { hnh::Runtime::get().sync_all(); }); }

int hnhd_setup_times_json(char *out, size_t capacity, int reset) {
    int n = 0;
    int rc = guarded([&] {
        json j = json::object();
        for (auto &kv : hnh::setup_times()) j[kv.first] = kv.second;
        n = copy_json(j, out, capacity);
        if (reset) hnh::setup_times_reset();
    });
    return rc ? rc : n;
}

// ---- SpmatLocal ---------------------------------------------------------------------------------
int hnhd_spmat_load_er(int logM, int nnz_per_row, uint64_t seed, hnhd_spmat_t **out) {
    return guarded([&] {
        if (!out) throw hnh::Error(HNH_E_INVALID, "null out");
        std::unique_ptr<hnhd_spmat> s(new hnhd_spmat);
        SpmatLocal::er_seed = seed;
        s->m.loadTuples(false, logM, nnz_per_row, "");
        *out = s.release();
    });
}
int hnhd_spmat_load_file(const char *filename, hnhd_spmat_t **out) {
    return guarded([&] {
        if (!filename || !out) throw hnh::Error(HNH_E_INVALID, "null argument");
        std::unique_ptr<hnhd_spmat> s(new hnhd_spmat);
        s->m.loadTuples(true, -1, -1, filename);
        *out = s.release();
    });
}
int hnhd_spmat_from_tuples(uint64_t M, uint64_t N, const uint64_t *rows, const uint64_t *cols, const double *vals,
                           int64_t n_local, hnhd_spmat_t **out) {
    return guarded([&] {
        if (!out || n_local < 0 || (n_local > 0 && (!rows || !cols || !vals))) throw hnh::Error(HNH_E_INVALID, "bad argument");
        std::unique_ptr<hnhd_spmat> s(new hnhd_spmat);
        s->m.setTuples(M, N, rows, cols, vals, n_local);
        *out = s.release();
    });
}
int hnhd_spmat_info(const hnhd_spmat_t *S, uint64_t *M, uint64_t *N, uint64_t *dist_nnz, int64_t *local_tuples) {
    if (!S) return hnh::set_error(HNH_E_INVALID, "null spmat");
    if (M) *M = S->m.M;
    if (N) *N = S->m.N;
    if (dist_nnz) *dist_nnz = S->m.dist_nnz;
    if (local_tuples) *local_tuples = S->m.local_tuple_count();
    return HNH_OK;
}
int hnhd_spmat_tuples(const hnhd_spmat_t *S, uint64_t *rows, uint64_t *cols, double *vals, int64_t capacity) {
    if (!S || S->m.local_tuple_count() > capacity) return hnh::set_error(HNH_E_INVALID, "bad argument / capacity");
    if (S->m.tuples_on_device()) {
        int rc = guarded([&] { const_cast<hnhd_spmat_t *>(S)->m.tuples_to_host(); });
        if (rc) return rc;
    }
    for (size_t i = 0; i < S->m.coords.size(); i++) {
        rows[i] = S->m.coords[i].r;
        cols[i] = S->m.coords[i].c;
        vals[i] = S->m.coords[i].value;
    }
    return HNH_OK;
}
void hnhd_spmat_destroy(hnhd_spmat_t *S) { delete S; }

// ---- algorithms ---------------------------------------------------------------------------------
int hnhd_alg_create(const char *name, hnhd_spmat_t *S, int R, int c, hnhd_alg_t **out) {
    return guarded([&] {
        if (!name || !S || !out) throw hnh::Error(HNH_E_INVALID, "null argument");
        std::unique_ptr<hnhd_alg> a(new hnhd_alg);
        a->alg.reset(hnh_make_algorithm(name, &S->m, R, c, &a->kernel));
        *out = a.release();
    });
}
void hnhd_alg_destroy(hnhd_alg_t *alg) { delete alg; }

int hnhd_alg_dims(hnhd_alg_t *a, hnhd_alg_dims_t *o) {
    return guarded([&] {
        if (!a || !o) throw hnh::Error(HNH_E_INVALID, "null argument");
        Distributed_Sparse &d = *a->alg;
        o->M = d.M; o->N = d.N; o->R = d.R; o->p = d.p; o->c = d.c;
        o->localArows = d.localArows; o->localAcols = d.localAcols;
        o->localBrows = d.localBrows; o->localBcols = d.localBcols;
        o->s_values = d.num_S_values();
        o->st_values = d.num_ST_values();
        o->r_split = d.r_split ? 1 : 0;
        o->grid_i = d.grid->i; o->grid_j = d.grid->j; o->grid_k = d.grid->k;
        o->n_a_submatrices = (int)d.aSubmatrices.size();
        o->n_b_submatrices = (int)d.bSubmatrices.size();
    });
}
int hnhd_alg_submatrices(hnhd_alg_t *a, int which, int *out4, int capacity) {
    if (!a || !out4) return hnh::set_error(HNH_E_INVALID, "null argument");
    const vector<DenseSubmatrix> &v = which == 0 ? a->alg->aSubmatrices : a->alg->bSubmatrices;
    if ((int)v.size() * 4 > capacity) return hnh::set_error(HNH_E_INVALID, "capacity too small");
    for (size_t i = 0; i < v.size(); i++) {
        out4[4 * i] = v[i].topRow; out4[4 * i + 1] = v[i].leftCol;
        out4[4 * i + 2] = v[i].rowCount; out4[4 * i + 3] = v[i].colCount;
    }
    return (int)v.size();
}
int hnhd_alg_info_json(hnhd_alg_t *a, char *out, size_t capacity) {
    int n = 0;
    int rc = guarded([&] { n = copy_json(a->alg->json_algorithm_info(), out, capacity); });
    return rc ? rc : n;
}
int hnhd_alg_perf_json(hnhd_alg_t *a, char *out, size_t capacity) {
    int n = 0;
    int rc = guarded([&] { n = copy_json(a->alg->json_perf_statistics(), out, capacity); });
    return rc ? rc : n;
}
int hnhd_alg_reset_timers(hnhd_alg_t *a) { return guarded([&] { a->alg->reset_performance_timers(); }); }

static SpmatLocal *pick(hnhd_alg_t *a, int which) { return which == 0 ? a->alg->S.get() : a->alg->ST.get(); }
int hnhd_alg_block_count(hnhd_alg_t *a, int which) { return a ? (int)pick(a, which)->csr_blocks.size() : -1; }
int hnhd_alg_block_meta(hnhd_alg_t *a, int which, int block, int64_t *rows, int64_t *cols, int64_t *nnz, int *transpose,
                        int *is_null) {
    if (!a) return hnh::set_error(HNH_E_INVALID, "null argument");
    SpmatLocal *m = pick(a, which);
    if (block < 0 || block >= (int)m->csr_blocks.size()) return hnh::set_error(HNH_E_INVALID, "block out of range");
    CSRLocal *b = m->csr_blocks[block];
    *is_null = b == nullptr;
    *rows = b ? b->rows : 0;
    *cols = b ? b->cols : 0;
    *nnz = b ? b->num_coords : 0;
    *transpose = b ? (int)b->transpose : 0;
    return HNH_OK;
}
int hnhd_alg_block_arrays(hnhd_alg_t *a, int which, int block, int64_t *rowStart, int64_t *col_idx, int64_t *row_idx,
                          double *values) {
    return guarded([&] {
        CSRLocal *b = pick(a, which)->csr_blocks.at((size_t)block);
        if (!b) throw hnh::Error(HNH_E_INVALID, "null block");
        CSRLocal::HostCSR h = b->to_host();
        std::memcpy(rowStart, h.rowStart.data(), sizeof(int64_t) * h.rowStart.size());
        std::memcpy(col_idx, h.col_idx.data(), sizeof(int64_t) * h.col_idx.size());
        std::memcpy(row_idx, h.row_idx.data(), sizeof(int64_t) * h.row_idx.size());
        std::memcpy(values, h.values.data(), sizeof(double) * h.values.size());
    });
}

// ---- dense / vectors ------------------------------------------------------------------------------
int hnhd_dense_create(int64_t rows, int64_t cols, double value, hnhd_dense_t **out) {
    return guarded([&] {
        std::unique_ptr<hnhd_dense> d(new hnhd_dense);
        d->m = DenseMatrix::Constant(rows, cols, value);
        *out = d.release();
    });
}
int hnhd_dense_like(hnhd_alg_t *a, int which, double value, hnhd_dense_t **out) {
    return guarded([&] {
        std::unique_ptr<hnhd_dense> d(new hnhd_dense);
        d->m = which == 0 ? a->alg->like_A_matrix(value) : a->alg->like_B_matrix(value);
        *out = d.release();
    });
}
int hnhd_dense_fill(hnhd_dense_t *m, double value) { return guarded([&] { m->m.setConstant(value); }); }
int hnhd_dense_dummy_initialize(hnhd_alg_t *a, hnhd_dense_t *m, int which) {
    return guarded([&] { a->alg->dummyInitialize(m->m, which == 0 ? Amat : Bmat); });
}
int hnhd_dense_from_host(hnhd_dense_t *m, const double *host) { return guarded([&] { m->m.copy_from_host(host); }); }
int hnhd_dense_to_host(const hnhd_dense_t *m, double *host) {
    return guarded([&] { m->m.copy_to_host(host); });
}
int hnhd_dense_shape(const hnhd_dense_t *m, int64_t *rows, int64_t *cols) {
    *rows = m->m.rows();
    *cols = m->m.cols();
    return HNH_OK;
}
void *hnhd_dense_data(hnhd_dense_t *m) { return m->m.data(); }
void hnhd_dense_destroy(hnhd_dense_t *m) { delete m; }

int hnhd_vec_create(int64_t n, double value, hnhd_vec_t **out) {
    return guarded([&] {
        std::unique_ptr<hnhd_vec> v(new hnhd_vec);
        v->v = VectorXd::Constant(n, value);
        *out = v.release();
    });
}
int hnhd_vec_like(hnhd_alg_t *a, int which, double value, hnhd_vec_t **out) {
    return guarded([&] {
        std::unique_ptr<hnhd_vec> v(new hnhd_vec);
        v->v = which == 0 ? a->alg->like_S_values(value) : a->alg->like_ST_values(value);
        *out = v.release();
    });
}
int hnhd_vec_fill(hnhd_vec_t *v, double value) { return guarded([&] { v->v.setConstant(value); }); }
int hnhd_vec_from_host(hnhd_vec_t *v, const double *host) { return guarded([&] { v->v.copy_from_host(host); }); }
int hnhd_vec_to_host(const hnhd_vec_t *v, double *host) {
    return guarded([&] {
        vector<double> h = v->v.to_host();
        std::memcpy(host, h.data(), sizeof(double) * h.size());
    });
}
int64_t hnhd_vec_size(const hnhd_vec_t *v) { return v ? v->v.size() : -1; }
void hnhd_vec_destroy(hnhd_vec_t *v) { delete v; }

// ---- operations -------------------------------------------------------------------------------------
int hnhd_alg_op(hnhd_alg_t *a, int op, hnhd_dense_t *A, hnhd_dense_t *B, hnhd_vec_t *svals, hnhd_vec_t *result, int aux) {
    return guarded([&] {
        if (!a) throw hnh::Error(HNH_E_INVALID, "null algorithm");
        Distributed_Sparse &d = *a->alg;
        auto needAB = [&] { if (!A || !B) throw hnh::Error(HNH_E_INVALID, "A and B are required"); };
        auto needS = [&] { if (!svals) throw hnh::Error(HNH_E_INVALID, "svals is required"); };
        auto needR = [&] { if (!result) throw hnh::Error(HNH_E_INVALID, "result is required"); };
        switch (op) {
            case HNHD_OP_SDDMM_A: needAB(); needS(); needR(); d.sddmmA(A->m, B->m, svals->v, result->v); break;
            case HNHD_OP_SDDMM_B: needAB(); needS(); needR(); d.sddmmB(A->m, B->m, svals->v, result->v); break;
            case HNHD_OP_SPMM_A: needAB(); needS(); d.spmmA(A->m, B->m, svals->v); break;
            case HNHD_OP_SPMM_B: needAB(); needS(); d.spmmB(A->m, B->m, svals->v); break;
            case HNHD_OP_FUSED_A: needAB(); needS(); needR(); d.fusedSpMM(A->m, B->m, svals->v, result->v, Amat); break;
            case HNHD_OP_FUSED_B: needAB(); needS(); needR(); d.fusedSpMM(A->m, B->m, svals->v, result->v, Bmat); break;
            case HNHD_OP_INITIAL_SHIFT: d.initial_shift(A ? &A->m : nullptr, B ? &B->m : nullptr, (KernelMode)aux); break;
            case HNHD_OP_DE_SHIFT: d.de_shift(A ? &A->m : nullptr, B ? &B->m : nullptr, (KernelMode)aux); break;
            default: throw hnh::Error(HNH_E_INVALID, "unknown op");
        }
    });
}

int hnhd_alg_fused_host(hnhd_alg_t *a, hnhd_dense_t *A, hnhd_dense_t *B, hnhd_vec_t *svals, hnhd_vec_t *result,
                        const double *hostA, const double *hostB, double *hostOut, int mode, int64_t chunk_rows) {
    return guarded([&] {
        if (!a || !A || !B || !svals || !result || !hostA || !hostB || !hostOut || (mode != 0 && mode != 1))
            throw hnh::Error(HNH_E_INVALID, "hnhd_alg_fused_host: bad argument");
        Distributed_Sparse &d = *a->alg;
        Sparse15D_Dense_Shift *ds = dynamic_cast<Sparse15D_Dense_Shift *>(&d);
        const int64_t keep = ds ? ds->host_pipeline_chunk_rows : 0;
        if (ds && chunk_rows != 0) ds->host_pipeline_chunk_rows = chunk_rows;
        try {
            d.fusedSpMM_host(hostA, hostB, hostOut, A->m, B->m, svals->v, result->v, mode == 0 ? Amat : Bmat);
        } catch (...) {
            if (ds) ds->host_pipeline_chunk_rows = keep;
            throw;
        }
        if (ds) ds->host_pipeline_chunk_rows = keep;
    });
}

int hnhd_timer_start(void) {
    return guarded([] {
        if (!g_t0) {
            hnh::cuda_check(cudaEventCreate(&g_t0), "cudaEventCreate");
            hnh::cuda_check(cudaEventCreate(&g_t1), "cudaEventCreate");
        }
        hnh::cuda_check(cudaEventRecord(g_t0, hnh::Runtime::get().compute_stream()), "cudaEventRecord");
    });
}
int hnhd_timer_stop(double *ms_out) {
    return guarded([&] {
        if (!g_t0) throw hnh::Error(HNH_E_INVALID, "hnhd_timer_stop without start");
        hnh::cuda_check(cudaEventRecord(g_t1, hnh::Runtime::get().compute_stream()), "cudaEventRecord");
        hnh::cuda_check(cudaEventSynchronize(g_t1), "cudaEventSynchronize");
        float ms = 0.f;
        hnh::cuda_check(cudaEventElapsedTime(&ms, g_t0, g_t1), "cudaEventElapsedTime");
        *ms_out = ms;
    });
}

int hnhd_benchmark_algorithm(hnhd_spmat_t *S, const char *algorithm_name, const char *output_file, int fused, int R, int c,
                             const char *app, int trials, int warmup, char *json_out, size_t capacity) {
    int n = 0;
    int rc = guarded([&] {
        json j = benchmark_algorithm_ex(&S->m, algorithm_name, output_file ? output_file : "", fused != 0, R, c,
                                        app ? app : "vanilla", trials, warmup);
        n = json_out ? copy_json(j, json_out, capacity) : 0;
    });
    return rc ? rc : n;
}

int hnhd_als_residuals(hnhd_alg_t *a, int steps, double *out2) {
    return guarded([&] {
        if (!a || !out2) throw hnh::Error(HNH_E_INVALID, "null argument");
        Distributed_ALS als(a->alg.get(), true);
        als.initializeEmbeddings();
        out2[0] = als.computeResidual();
        for (int i = 0; i < steps; i++) {
            als.cg_optimizer(Amat, 10);
            als.cg_optimizer(Bmat, 10);
        }
        out2[1] = als.computeResidual();
    });
}

int hnhd_als_run(hnhd_alg_t *a, const double *hostAgt, const double *hostBgt, const double *hostA0, const double *hostB0,
                 int steps, int cg_iters, double *out2, double *hostA_out, double *hostB_out) {
    return guarded([&] {
        if (!a || !hostAgt || !hostBgt || !hostA0 || !hostB0 || !out2 || steps < 0 || cg_iters < 0)
            throw hnh::Error(HNH_E_INVALID, "hnhd_als_run: bad argument");
        Distributed_Sparse *d = a->alg.get();
        Distributed_ALS als(d, false);
        DenseMatrix Agt = d->like_A_matrix(0.0), Bgt = d->like_B_matrix(0.0);
        Agt.copy_from_host(hostAgt);
        Bgt.copy_from_host(hostBgt);
        VectorXd ones = d->like_S_values(1.0);
        als.ground_truth = d->like_S_values(0.0);
        d->initial_shift(&Agt, &Bgt, k_sddmmA);
        d->sddmmA(Agt, Bgt, ones, als.ground_truth);
        d->de_shift(&Agt, &Bgt, k_sddmmA);
        VectorXd ones_t = d->like_ST_values(1.0);
        als.ground_truth_transpose = d->like_ST_values(0.0);
        d->initial_shift(&Agt, &Bgt, k_sddmmB);
        d->sddmmB(Agt, Bgt, ones_t, als.ground_truth_transpose);
        d->de_shift(&Agt, &Bgt, k_sddmmB);
        als.A = d->like_A_matrix(0.0);
        als.B = d->like_B_matrix(0.0);
        als.A.copy_from_host(hostA0);
        als.B.copy_from_host(hostB0);
        out2[0] = als.computeResidual();
        for (int i = 0; i < steps; i++) {
            als.cg_optimizer(Amat, cg_iters);
            als.cg_optimizer(Bmat, cg_iters);
        }
        out2[1] = als.computeResidual();
        if (hostA_out) als.A.copy_to_host(hostA_out);
        if (hostB_out) als.B.copy_to_host(hostB_out);
    });
}

// ---- GAT ------------------------------------------------------------------------------------------
int hnhd_gat_create(hnhd_alg_t *a, int n_layers, const int *layers3, double alpha, hnhd_gat_t **out) {
    return guarded([&] {
        if (!a || !layers3 || !out || n_layers <= 0) throw hnh::Error(HNH_E_INVALID, "hnhd_gat_create: bad argument");
        vector<GATLayer> layers;
        for (int i = 0; i < n_layers; i++) {
            if (layers3[3 * i] <= 0 || layers3[3 * i + 1] <= 0 || layers3[3 * i + 2] <= 0)
                throw hnh::Error(HNH_E_INVALID, "hnhd_gat_create: layer sizes must be positive");
            layers.emplace_back(layers3[3 * i], layers3[3 * i + 1], layers3[3 * i + 2]);
        }
        std::unique_ptr<hnhd_gat> g(new hnhd_gat);
        g->g.reset(new GAT(layers, a->alg.get()));
        g->g->leaky_relu_alpha = alpha;
        *out = g.release();
    });
}
static DenseMatrix &gat_weight(hnhd_gat_t *g, int layer, int head) {
    if (!g || layer < 0 || layer >= (int)g->g->layers.size()) throw hnh::Error(HNH_E_INVALID, "gat: no such layer");
    GATLayer &l = g->g->layers[(size_t)layer];
    if (head < 0 || head >= l.num_heads) throw hnh::Error(HNH_E_INVALID, "gat: no such head");
    return l.wMats[(size_t)head];
}
static DenseMatrix &gat_buffer(hnhd_gat_t *g, int buffer) {
    if (!g || buffer < 0 || buffer >= (int)g->g->buffers.size()) throw hnh::Error(HNH_E_INVALID, "gat: no such buffer");
    return g->g->buffers[(size_t)buffer];
}
int hnhd_gat_weight_shape(hnhd_gat_t *g, int layer, int head, int64_t *rows, int64_t *cols) {
    return guarded([&] {
        DenseMatrix &w = gat_weight(g, layer, head);
        if (rows) *rows = w.rows();
        if (cols) *cols = w.cols();
    });
}
int hnhd_gat_set_weight(hnhd_gat_t *g, int layer, int head, const double *host) {
    return guarded([&] {
        if (!host) throw hnh::Error(HNH_E_INVALID, "null host pointer");
        gat_weight(g, layer, head).copy_from_host(host);
    });
}
int hnhd_gat_buffer_shape(hnhd_gat_t *g, int buffer, int64_t *rows, int64_t *cols) {
    return guarded([&] {
        DenseMatrix &b = gat_buffer(g, buffer);
        if (rows) *rows = b.rows();
        if (cols) *cols = b.cols();
    });
}
int hnhd_gat_set_input(hnhd_gat_t *g, const double *host) {
    return guarded([&] {
        if (!host) throw hnh::Error(HNH_E_INVALID, "null host pointer");
        gat_buffer(g, 0).copy_from_host(host);
    });
}
int hnhd_gat_get_buffer(hnhd_gat_t *g, int buffer, double *host) {
    return guarded([&] {
        if (!host) throw hnh::Error(HNH_E_INVALID, "null host pointer");
        gat_buffer(g, buffer).copy_to_host(host);
    });
}
int hnhd_gat_forward(hnhd_gat_t *g) {
    return guarded([&] {
        if (!g) throw hnh::Error(HNH_E_INVALID, "null gat");
        g->g->forwardPass();
    });
}
int hnhd_gat_supports_backward(hnhd_gat_t *g) {
    if (!g) return hnh::set_error(HNH_E_INVALID, "null gat");
    return g->g->supportsBackward() ? 1 : 0;
}
int hnhd_gat_backward(hnhd_gat_t *g, const double *host_output_grad) {
    return guarded([&] {
        if (!g || !host_output_grad) throw hnh::Error(HNH_E_INVALID, "hnhd_gat_backward: null argument");
        GAT &net = *g->g;
        const string why = net.backwardUnsupportedReason();  // refuse before touching the device
        if (!why.empty()) throw hnh::Error(HNH_E_INVALID, "GAT::backwardPass: " + why);
        DenseMatrix grad(net.buffers.back().rows(), net.buffers.back().cols());
        grad.copy_from_host(host_output_grad);
        net.backwardPass(grad);
    });
}
int hnhd_gat_get_weight_grad(hnhd_gat_t *g, int layer, int head, double *host) {
    return guarded([&] {
        if (!host) throw hnh::Error(HNH_E_INVALID, "null host pointer");
        gat_weight(g, layer, head);  // validates layer and head
        if (g->g->wGrads.size() != g->g->layers.size())
            throw hnh::Error(HNH_E_INVALID, "hnhd_gat_get_weight_grad: no gradients (run hnhd_gat_backward first)");
        g->g->wGrads[(size_t)layer][(size_t)head].copy_to_host(host);
    });
}
int hnhd_gat_get_input_grad(hnhd_gat_t *g, double *host) {
    return guarded([&] {
        if (!g || !host) throw hnh::Error(HNH_E_INVALID, "hnhd_gat_get_input_grad: null argument");
        if (g->g->input_grad.size() != g->g->buffers[0].size())
            throw hnh::Error(HNH_E_INVALID, "hnhd_gat_get_input_grad: no gradients (run hnhd_gat_backward first)");
        g->g->input_grad.copy_to_host(host);
    });
}
int hnhd_gat_get_weight(hnhd_gat_t *g, int layer, int head, double *host) {
    return guarded([&] {
        if (!host) throw hnh::Error(HNH_E_INVALID, "null host pointer");
        gat_weight(g, layer, head).copy_to_host(host);
    });
}
int hnhd_gat_sgd_step(hnhd_gat_t *g, double lr) {
    return guarded([&] {
        if (!g) throw hnh::Error(HNH_E_INVALID, "null gat");
        g->g->applyGradients(lr);
    });
}
void hnhd_gat_destroy(hnhd_gat_t *g) { delete g; }

}  // extern "C"
