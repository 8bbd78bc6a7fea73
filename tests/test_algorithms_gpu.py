"""The distributed algorithm classes at p = 1 on the GPU, through the driver C ABI, against the
global scipy/numpy reference (second oracle, SURVEY.md 8c) and the dummyInitialize closed form.
Multi-rank parity lives in tests/test_multirank_gpu.py."""
import os

import numpy as np
import pytest

from distributed_sddmm_b200 import driver as D
from oracle import hnh_oracle as orc

pytestmark = pytest.mark.gpu
SEED = 0xC0FFEE + 3
ALGS = ["15d_fusion1", "15d_fusion2", "15d_sparse", "25d_dense_replicate", "25d_sparse_replicate"]
RTOL = 1e-11


def rel_err(got, ref):
    return np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-300)


@pytest.fixture(scope="module")
def world():
    D.world_init("self")
    yield
    D.world_finalize()


@pytest.fixture(scope="module")
def problem():
    logM, npr, R = 10, 8, 32
    N = 1 << logM
    rows, cols, vals = orc.er_tuples(logM, npr, SEED)
    rng = np.random.default_rng(17)
    A = rng.uniform(-1, 1, (N, R))
    B = rng.uniform(-1, 1, (N, R))
    sv = rng.uniform(0.5, 1.5, len(rows))  # values in CSR order of S (row asc, col asc)
    S, sddmm, spmmA, spmmB, fused = orc.global_reference(rows, cols, sv, A, B)
    # the same nonzeros in CSR order of S^T
    order_t = np.lexsort((rows, cols))
    return dict(logM=logM, npr=npr, R=R, N=N, A=A, B=B, sv=sv, sv_t=sv[order_t], sddmm=sddmm, sddmm_t=sddmm[order_t],
                spmmA=spmmA, spmmB=spmmB, fused=fused, S=S)


@pytest.mark.parametrize("name", ALGS)
def test_p1_operations_match_global_reference(world, problem, name):
    P = problem
    S = D.SpmatLocal.load_er(P["logM"], P["npr"], SEED)
    alg = D.Algorithm(name, S, P["R"], 1)
    A, B = alg.like_A_matrix(), alg.like_B_matrix()
    Sv, res = alg.like_S_values(1.0), alg.like_S_values(0.0)
    STv, res_t = alg.like_ST_values(1.0), alg.like_ST_values(0.0)
    Sv.from_host(P["sv"])
    STv.from_host(P["sv_t"])

    def load():
        A.from_host(P["A"])
        B.from_host(P["B"])

    # sddmmA: result = SValues o (A B^T sampled at S), in S's CSR order
    load()
    alg.initial_shift(A, B, "sddmmA")
    alg.sddmmA(A, B, Sv, res)
    alg.de_shift(A, B, "sddmmA")
    assert rel_err(res.to_host(), P["sddmm"]) < RTOL
    assert np.array_equal(A.to_host(), P["A"]) and np.array_equal(B.to_host(), P["B"])  # inputs untouched
    # sddmmB: the same numbers in S^T's order
    alg.initial_shift(A, B, "sddmmB")
    alg.sddmmB(A, B, STv, res_t)
    alg.de_shift(A, B, "sddmmB")
    assert rel_err(res_t.to_host(), P["sddmm_t"]) < RTOL
    # spmmA: A = S B (A's previous content is discarded)
    alg.initial_shift(A, B, "spmmA")
    alg.spmmA(A, B, Sv)
    alg.de_shift(A, B, "spmmA")
    assert rel_err(A.to_host(), P["spmmA"]) < RTOL
    # spmmB: B = S^T A
    load()
    alg.initial_shift(A, B, "spmmB")
    alg.spmmB(A, B, STv)
    alg.de_shift(A, B, "spmmB")
    assert rel_err(B.to_host(), P["spmmB"]) < RTOL
    # fusedSpMM(Amat): A = (SDDMM values) B
    load()
    alg.initial_shift(A, B, "sddmmA")
    alg.fusedSpMM(A, B, Sv, res, "A")
    alg.de_shift(A, B, "sddmmA")
    if name == "15d_fusion2":
        # local kernel fusion treats S as an all-ones pattern and leaves sddmm_buffer unfilled
        # (reference 15D_dense_shift.hpp:189,250-251)
        ones = np.ones(len(P["sv"]))
        _, _, _, _, fused1 = orc.global_reference(*_tuples(P), ones, P["A"], P["B"])
        assert rel_err(A.to_host(), fused1) < RTOL
    else:
        assert rel_err(A.to_host(), P["fused"]) < RTOL
        assert rel_err(res.to_host(), P["sddmm"]) < RTOL
    assert np.array_equal(B.to_host(), P["B"])


def _tuples(P):
    S = P["S"]
    rows = np.repeat(np.arange(P["N"]), np.diff(S.indptr)).astype(np.uint64)
    return rows, S.indices.astype(np.uint64)


@pytest.mark.parametrize("name", ALGS)
def test_p1_dummy_initialize_closed_form(world, name):
    """verify_operation of the reference (scratch.cpp:26-76) with a known answer: S == 1,
    X[i,k] = i*R + k  =>  SDDMM(i,j) has a closed form that is exact in fp64."""
    logM, npr, R = 12, 8, 16
    rows, cols, vals = orc.er_tuples(logM, npr, SEED)
    S = D.SpmatLocal.load_er(logM, npr, SEED)
    alg = D.Algorithm(name, S, R, 1)
    A, B = alg.like_A_matrix(), alg.like_B_matrix()
    alg.dummyInitialize(A, "A")
    alg.dummyInitialize(B, "B")
    Sv, res = alg.like_S_values(1.0), alg.like_S_values(0.0)
    alg.initial_shift(A, B, "sddmmA")
    alg.sddmmA(A, B, Sv, res)
    expect = orc.dummy_sddmm_closed_form(rows.astype(np.int64), cols.astype(np.int64), R)
    assert np.array_equal(res.to_host(), expect)


def test_benchmark_algorithm_record(world):
    S = D.SpmatLocal.load_er(12, 8, SEED)
    for name in ("15d_fusion1", "15d_fusion2"):
        rec = D.benchmark_algorithm(S, name, R=32, c=1, fused=True, trials=3, warmup=1)
        assert rec["alg_name"] == name and rec["num_trials"] == 3 and rec["fused"] is True
        assert rec["overall_throughput"] > 0 and rec["elapsed"] > 0
        assert rec["alg_info"]["nnz"] == S.info()["dist_nnz"]
        assert set(rec["perf_stats"]) == {"Replication Time", "Cyclic Shift Time", "Computation Time"}


def test_als_cg_reduces_residual(world):
    """One ALS step on an artificial rank-R ground truth must not blow up and should shrink the residual."""
    import ctypes as C
    from distributed_sddmm_b200 import lib
    S = D.SpmatLocal.load_er(10, 8, SEED)
    rec = D.benchmark_algorithm(S, "15d_fusion2", R=16, c=1, fused=True, app="als", trials=1, warmup=0)
    assert rec["overall_throughput"] > 0
    for name in ALGS:
        before, after = D.Algorithm(name, S, 16, 1).als_residuals(1)
        assert np.isfinite([before, after]).all() and after < before, (name, before, after)


# (written at the end of round 1 without GPU time; first run green on a B200 in round 2, gates removed)
@pytest.mark.parametrize("name,chunk", [("15d_fusion2", 77), ("15d_fusion2", 256), ("15d_fusion2", 4096),
                                        ("15d_fusion2", -1), ("15d_fusion1", 0), ("15d_sparse", 0)])
def test_p1_fused_host_operands_match_device_path(world, problem, name, chunk):
    """fusedSpMM_host (host operands in, result out; the 1.5D dense-shift algorithm pipelines upload / kernel /
    download in row chunks on one rank) gives bit-identical results to copy in + fusedSpMM + copy out."""
    P = problem
    S = D.SpmatLocal.load_er(P["logM"], P["npr"], SEED)
    alg = D.Algorithm(name, S, P["R"], 1)
    A, B = alg.like_A_matrix(), alg.like_B_matrix()
    for mode, like in (("A", alg.like_S_values), ("B", alg.like_ST_values)):
        Sv, res = like(1.0), like(0.0)
        A.from_host(P["A"])
        B.from_host(P["B"])
        alg.fusedSpMM(A, B, Sv, res, mode)
        want = (A if mode == "A" else B).to_host()
        want_values = res.to_host()
        res2 = like(0.0)
        hA, hB = np.ascontiguousarray(P["A"]), np.ascontiguousarray(P["B"])
        out = np.full_like(hA, np.nan)
        alg.fusedSpMM_host(A, B, Sv, res2, hA, hB, out, mode, chunk_rows=chunk)
        assert np.array_equal(out, want)
        if name != "15d_fusion2":  # local kernel fusion does not fill sddmm_buffer
            assert np.array_equal(res2.to_host(), want_values)
        # the staging matrices hold what the device path leaves there
        assert np.array_equal((A if mode == "A" else B).to_host(), want)


def test_gat_device_helpers(world):
    """hnh_leaky_relu_f64 / hnh_relu_cols_f64 / hnh_dgemm_f64 against numpy."""
    import torch
    from distributed_sddmm_b200 import lib
    L = lib()
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(5)
    x = rng.uniform(-1, 1, 10007)
    dx = torch.from_numpy(x).to(dev)
    D.check(L.hnh_leaky_relu_f64(dx.data_ptr(), dx.data_ptr(), x.size, 0.25, st))
    assert np.array_equal(dx.cpu().numpy(), np.maximum(x, 0) + np.minimum(x, 0) * 0.25)
    src = rng.uniform(-1, 1, (33, 5))
    dst = rng.uniform(-1, 1, (33, 17))
    dsrc, ddst = torch.from_numpy(src).to(dev), torch.from_numpy(dst).to(dev)
    D.check(L.hnh_relu_cols_f64(ddst.data_ptr(), 17, 10, dsrc.data_ptr(), 33, 5, st))
    want = dst.copy()
    want[:, 10:15] = np.maximum(src, 0)
    assert np.array_equal(ddst.cpu().numpy(), want)
    assert L.hnh_relu_cols_f64(ddst.data_ptr(), 17, 13, dsrc.data_ptr(), 33, 5, st) == -1  # window past the row end
    # the library's own fp64 tensor-core GEMM (dgemm_dmma_kernel): ragged edges, several K steps, several column tiles,
    # more row tiles than CTAs
    for m, n, k in ((70, 11, 19), (1, 1, 1), (64, 64, 16), (300, 130, 37), (5, 200, 3), (100000, 32, 256)):
        A, B = rng.uniform(-1, 1, (m, k)), rng.uniform(-1, 1, (k, n))
        dA, dB = torch.from_numpy(A).to(dev), torch.from_numpy(B).to(dev)
        dC = torch.full((m, n), float("nan"), dtype=torch.float64, device=dev)
        D.check(L.hnh_dgemm_f64(dC.data_ptr(), dA.data_ptr(), dB.data_ptr(), m, n, k, st))
        torch.cuda.synchronize()
        assert rel_err(dC.cpu().numpy(), A @ B) < 1e-13, (m, n, k)


@pytest.mark.parametrize("name", ALGS)
def test_p1_gat_forward_matches_global_model(world, name):
    """GAT forward pass on one rank (every algorithm has full-width operands there) against the numpy model
    that tests/test_oracle_vs_ref.py pins to the reference's gat.hpp."""
    from tests.mp_worker import gat_inputs
    logM, npr = 8, 6
    N = 1 << logM
    rows, cols, _ = orc.er_tuples(logM, npr, SEED)
    layers, X0, weights = gat_inputs(N, [[12, 8, 2], [16, 4, 3]], SEED)
    S = D.SpmatLocal.load_er(logM, npr, SEED)
    alg = D.Algorithm(name, S, layers[0][0], 1)
    net = D.GAT(alg, layers, 0.2)
    assert net.buffer_shape(0) == (N, 12) and net.buffer_shape(2) == (N, 12)
    for i, (fin, fph, heads) in enumerate(layers):
        for h in range(heads):
            assert net.weight_shape(i, h) == (fin, fph)
            net.set_weight(i, h, weights[i][h])
    net.set_input(X0)
    net.forward()
    want = orc.gat_forward_global(rows, cols, N, layers, weights, 0.2, X0)
    assert (want != 0).mean() > 0.2
    assert rel_err(net.buffer(2), want) < RTOL
    assert rel_err(net.buffer(1), orc.gat_forward_global(rows, cols, N, layers[:1], weights[:1], 0.2, X0)) < RTOL


@pytest.mark.parametrize("name", ALGS)
def test_p1_als_cg_matches_reference_als(world, name):
    """One alternating round of batched CG on given inputs against the reference's own Distributed_ALS (oracle/_ref, or
    its golden file)."""
    from tests import golden_util as G
    from tests.mp_worker import als_inputs
    logM, npr, R = 8, 6, 16
    N = 1 << logM
    Agt, Bgt, A0, B0 = als_inputs(N, R, SEED)
    S = D.SpmatLocal.load_er(logM, npr, SEED)
    alg = D.Algorithm(name, S, R, 1)
    res, A, B = D.als_run(alg, Agt, Bgt, A0, B0, 1, 10)
    want, _ = p1_als_reference(name)
    assert res[1] < 0.5 * res[0]
    assert np.allclose(res, want["residual"], rtol=1e-7, atol=0)
    assert G.rel_err(A, want["A"]) < 1e-7 and G.rel_err(B, want["B"]) < 1e-7


def p1_als_reference(name):
    def compute():
        from oracle import ref
        from tests.mp_worker import als_inputs
        logM, npr, R = 8, 6, 16
        N = 1 << logM
        rows, cols, _ = orc.er_tuples(logM, npr, SEED)
        want = ref.als(name, 1, 1, R, N, rows, cols, *als_inputs(N, R, SEED), 1, 10)
        return {"residual": np.asarray(want["residual"]), "A": want["A"], "B": want["B"]}
    from tests import mp_util as U
    return U.reference_arrays(f"als_p1_{name}", compute)


@pytest.mark.parametrize("R", [12, 192])
def test_p1_fusion2_fused_widths_outside_the_dispatch_table(world, R):
    """fusedSpMM of the local-kernel-fusion algorithm on one rank at a width without an in-place kernel (the
    reference's bench_heatmap.cpp sweeps R = 64 ... 448 in steps of 64): falls back to the accumulate-into-a-buffer
    path with the generic kernel."""
    logM, npr = 9, 6
    N = 1 << logM
    rows, cols, _ = orc.er_tuples(logM, npr, SEED)
    rng = np.random.default_rng(R)
    A0, B0 = rng.uniform(-1, 1, (N, R)), rng.uniform(-1, 1, (N, R))
    S = D.SpmatLocal.load_er(logM, npr, SEED)
    alg = D.Algorithm("15d_fusion2", S, R, 1)
    A, B = alg.like_A_matrix(), alg.like_B_matrix()
    Sv, res = alg.like_S_values(1.0), alg.like_S_values(0.0)
    for mode in ("A", "B"):
        A.from_host(A0)
        B.from_host(B0)
        if mode == "B":
            Sv, res = alg.like_ST_values(1.0), alg.like_ST_values(0.0)
        alg.fusedSpMM(A, B, Sv, res, mode)
        if mode == "A":
            _, _, _, _, want = orc.global_reference(rows, cols, np.ones(len(rows)), A0, B0)
            assert rel_err(A.to_host(), want) < RTOL
        else:
            _, _, _, _, want = orc.global_reference(cols, rows, np.ones(len(rows)), B0, A0)  # S^T in the role of S
            assert rel_err(B.to_host(), want) < RTOL
