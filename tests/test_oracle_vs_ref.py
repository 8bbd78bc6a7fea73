"""Pinning the oracle (CPU): the C restatement (oracle/hnh_oracle.c) and the scipy global reference
against OUTPUTS OF THE REFERENCE ITSELF -- oracle/_ref, the reference's own sources compiled unmodified
(MPI ranks as threads; MKL / Eigen / CombBLAS shimmed) -- for every algorithm and several (p, c).
Where oracle/_ref is not built, the reference's outputs come from the golden files scripts/make_golden.py wrote."""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import hnh_oracle as orc
from oracle import ref
from tests import golden_util as G
from tests import mp_util as U

OPS = ["sddmmA", "spmmA", "spmmB", "fusedA", "sddmmB", "fusedB"]


def problem(logM=8, npr=6, R=24, seed=7):
    N = 1 << logM
    rows, cols, _ = orc.er_tuples(logM, npr, seed)
    rng = np.random.default_rng(0)
    A, B = rng.uniform(-1, 1, (N, R)), rng.uniform(-1, 1, (N, R))
    sv = rng.uniform(0.5, 1.5, len(rows))
    return N, R, rows, cols, sv, A, B


def assert_close(want, desired, rtol, atol):
    """np.testing.assert_allclose(want, desired) for a reference array `want` that may be stored reduced."""
    if isinstance(want, G.Reduced):
        assert G.abs_err(desired, want) <= atol + rtol * np.abs(desired).max(), want
    else:
        np.testing.assert_allclose(want, desired, rtol=rtol, atol=atol)


CSR_FIELDS = ("rowStart", "col_idx", "row_idx", "values")


def restatement_reference():
    def compute():
        N, R, rows, cols, sv, A, B = problem()
        out = {}
        for alg in ("15d_fusion2", "15d_fusion1"):
            o = ref.run(alg, 1, 1, R, N, N, rows, cols, sv, A, B, ["sddmmA", "spmmA"])[0]
            if alg == "15d_fusion2":
                out.update({f"{alg}_S_b0_{f}": o["S_blocks"][0][f] for f in CSR_FIELDS})
            out.update({f"{alg}_S_rows": o["S_rows"], f"{alg}_S_cols": o["S_cols"], f"{alg}_sddmm_values": o["ops"][0]["values"],
                        f"{alg}_spmm_A": o["ops"][1]["A"]})
        return out
    return U.reference_arrays("oracle_restatement", compute,
                              exact=[f"15d_fusion2_S_b0_{f}" for f in CSR_FIELDS] +
                                    [f"{a}_{k}" for a in ("15d_fusion2", "15d_fusion1") for k in ("S_rows", "S_cols", "sddmm_values")])


def test_c_restatement_is_bit_exact_with_reference_kernels():
    """p = 1: the reference's CSRLocal (MKL-shim COO->CSR) and its StandardKernel::sddmm_local loop against
    oracle.coo_to_csr / sddmm_coo / spmm_csr on the same block."""
    N, R, rows, cols, sv, A, B = problem()
    want, _ = restatement_reference()
    for alg in ("15d_fusion2", "15d_fusion1"):
        if alg == "15d_fusion2":
            mine = orc.coo_to_csr(N, N, rows, cols, sv)
            for f in CSR_FIELDS:
                assert G.same(getattr(mine, f), want[f"{alg}_S_b0_{f}"]), f
        # SDDMM: reference result = SValues o (sum_k A[r,k] B[c,k]) in the reference's local value order
        csr = orc.coo_to_csr(N, N, rows, cols, sv)
        assert G.same(csr.row_idx, want[f"{alg}_S_rows"]) and G.same(csr.col_idx, want[f"{alg}_S_cols"])  # p = 1: CSR order of S
        v = orc.sddmm_coo(csr.row_idx, csr.col_idx, np.zeros(csr.nnz), A, B)
        assert G.same(sv * v, want[f"{alg}_sddmm_values"]), "SDDMM restatement differs from the reference loop"
        Y = orc.spmm_csr(csr.rowStart, csr.col_idx, csr.values, B, np.zeros((N, R)))
        assert_close(want[f"{alg}_spmm_A"], Y, rtol=0, atol=1e-13)


@pytest.mark.parametrize("alg,p,c", [
    ("15d_fusion1", 2, 1), ("15d_fusion1", 8, 2), ("15d_fusion1", 3, 1), ("15d_fusion2", 2, 2), ("15d_fusion2", 8, 4),
    ("15d_fusion2", 6, 2), ("15d_sparse", 4, 2), ("15d_sparse", 8, 1), ("15d_sparse", 2, 1), ("25d_dense_replicate", 4, 1),
    ("25d_dense_replicate", 8, 2), ("25d_sparse_replicate", 4, 1), ("25d_sparse_replicate", 8, 2), ("25d_sparse_replicate", 9, 1)])
# Not listed on purpose: rings of odd size > 1 whose CSR block travels (15d_sparse p/c = 3, 25d_dense s = 3).  The
# reference ships row_idx only in SDDMM passes and rowStart only in SpMM passes (SpmatLocal.hpp:223-240), so after an
# odd number of shifts the resident buffer keeps a stale array from an earlier pass and a mixed sequence of operations
# goes wrong there.  A B200 box only has p in {1, 2, 4, 8}; this library always ships rowStart (hnh/SpmatLocal.hpp).
def test_global_reference_matches_the_reference_code(alg, p, c):
    N, R, rows, cols, sv, A, B = problem()
    S, sddmm, spmmA, spmmB, fused = orc.global_reference(rows, cols, sv, A, B)
    if alg == "15d_fusion2":  # treats S as an all-ones pattern in fusedSpMM (15D_dense_shift.hpp:189)
        _, sd1, _, _, fused = orc.global_reference(rows, cols, np.ones(len(rows)), A, B)
        fusedB = sp.csr_matrix((sd1, S.indices, S.indptr), shape=(N, N)).T @ A
    else:
        fusedB = sp.csr_matrix((sddmm, S.indices, S.indptr), shape=(N, N)).T @ A
    want, _ = global_outputs_of_reference(alg, p, c)
    assert_close(want["sddmmA"], sddmm, rtol=1e-12, atol=1e-13)
    assert_close(want["sddmmB"], sddmm, rtol=1e-12, atol=1e-13)
    assert_close(want["spmmA"], spmmA, rtol=1e-11, atol=1e-12)
    assert_close(want["spmmB"], spmmB, rtol=1e-11, atol=1e-12)
    assert_close(want["fusedA"], fused, rtol=1e-11, atol=1e-12)
    assert_close(want["fusedB"], fusedB, rtol=1e-11, atol=1e-12)


def global_outputs_of_reference(alg, p, c):
    """The reference's per-rank outputs of every operation, assembled into global arrays."""
    def compute():
        N, R, rows, cols, sv, A, B = problem()
        key = rows.astype(np.int64) * N + cols.astype(np.int64)
        out = ref.run(alg, p, c, R, N, N, rows, cols, sv, A, B, OPS)
        got_a, got_b, cover = np.zeros(len(rows)), np.zeros(len(rows)), np.zeros(len(rows))
        for d in out:
            for which, op, acc in (("S", 0, got_a), ("ST", 4, got_b)):
                k = d[which + "_rows"] * N + d[which + "_cols"]
                idx = np.searchsorted(key, k)
                assert np.array_equal(key[np.minimum(idx, len(key) - 1)], k), "value slot with a coordinate that is not a nonzero"
                acc[idx] += d["ops"][op]["values"]
                if which == "S":
                    cover[idx] += 1
        assert np.all(cover == 1), "every nonzero's value lives on exactly one rank"
        return {"sddmmA": got_a, "sddmmB": got_b, "spmmA": ref.assemble_dense(out, "A", 1, N, R),
                "spmmB": ref.assemble_dense(out, "B", 2, N, R), "fusedA": ref.assemble_dense(out, "A", 3, N, R),
                "fusedB": ref.assemble_dense(out, "B", 5, N, R)}
    return U.reference_arrays(f"oracle_global_{alg}_p{p}_c{c}", compute)


def test_reference_benchmark_entry_point_runs(tmp_path):
    """The reference's own benchmark_algorithm (benchmark_dist.cpp:26-167) on its own loadTuples path: its matrix has
    the nonzeros of the oracle's generator."""
    import json

    def compute():
        out = tmp_path / "ref.json"
        ref.benchmark("15d_fusion1", 2, 1, 16, 10, 8, 0xC0FFEE, fused=True, output_file=str(out), threads_per_rank=2)
        rec = json.loads(out.read_text().strip().rstrip(","))
        assert rec["alg_name"] == "15d_fusion1" and rec["num_trials"] == 5 and rec["alg_info"]["p"] == 2
        return {"nnz": np.int64(rec["alg_info"]["nnz"])}
    want, _ = U.reference_arrays("oracle_benchmark_nnz", compute)
    assert int(want["nnz"]) == len(orc.er_tuples(10, 8, 0xC0FFEE)[0])


@pytest.mark.parametrize("alg,p,c", [("15d_fusion1", 1, 1), ("15d_fusion2", 1, 1), ("15d_sparse", 1, 1),
                                     ("25d_dense_replicate", 1, 1), ("25d_sparse_replicate", 1, 1),
                                     ("15d_fusion1", 2, 1), ("15d_fusion1", 4, 2), ("15d_fusion1", 8, 8),
                                     ("15d_fusion2", 2, 1), ("15d_fusion2", 4, 1), ("15d_fusion2", 8, 1)])
def test_gat_global_model_matches_the_reference_gat(alg, p, c):
    """orc.gat_forward_global against the reference's gat.hpp (forward pass, two layers, several heads, random
    weights, explicit alpha) wherever the dense operands keep their full width: one rank, or the 1.5D dense-shift
    algorithms.  (Fusion 2 with c > 1 is left out: there the reference's SpMM pass, called with initial_replicate =
    false, accumulates onto the gathered projection left by the SDDMM pass -- 15D_dense_shift.hpp:306-314 -- so its
    output is not the GAT formula; the GPU test compares that case against the reference run itself.)"""
    logM, npr = 7, 5
    N = 1 << logM
    rows, cols, _ = orc.er_tuples(logM, npr, 0xC0FFEE + 1)
    rng = np.random.default_rng(3)
    layers = [(6, 4, 2), (8, 3, 3)]
    weights = [[rng.uniform(-1, 1, (fin, fph)) for _ in range(h)] for fin, fph, h in layers]
    X0 = rng.uniform(-1, 1, (N, layers[0][0]))
    want = orc.gat_forward_global(rows, cols, N, layers, weights, 0.2, X0)
    assert (want != 0).mean() > 0.3 and (want == 0).mean() > 0.1  # both ReLU branches are exercised
    got, _ = U.reference_arrays(f"oracle_gat_{alg}_p{p}_c{c}", lambda: {
        "out": ref.gat(alg, p, c, N, rows, cols, np.ones(len(rows)), layers, weights, 0.2, X0)[0]})
    assert G.abs_err(want, got["out"]) / np.abs(want).max() < 1e-13


def als_problem(logM=7, npr=5, R=8, seed=0xC0FFEE + 8):
    N = 1 << logM
    rows, cols, _ = orc.er_tuples(logM, npr, seed)
    rng = np.random.default_rng(21)
    Agt, Bgt = rng.uniform(-1, 1, (N, R)) / R, rng.uniform(-1, 1, (N, R)) / R
    A0, B0 = 1.4 * rng.uniform(-1, 1, (N, R)) / R, rng.uniform(-1, 1, (N, R)) / R / 1.3
    return N, R, rows, cols, Agt, Bgt, A0, B0


@pytest.mark.skipif(not ref.available(), reason="compares the reference with itself: needs oracle/_ref/libhnh_ref.so")
def test_reference_als_is_layout_independent_and_converges():
    """The parity harness for BASELINE.json config 5's caller: the reference's Distributed_ALS / cg_optimizer on given
    ground-truth factors and starting embeddings.  Every algorithm and grid must produce the same embeddings (the
    arithmetic per row is the same; only summation orders differ), and one alternating round must shrink the
    residual.  The GPU tests compare the CUDA implementation with exactly these runs."""
    N, R, rows, cols, Agt, Bgt, A0, B0 = als_problem()
    base = ref.als("15d_fusion1", 1, 1, R, N, rows, cols, Agt, Bgt, A0, B0)
    assert 0 < base["residual"][1] < 0.5 * base["residual"][0]
    # the local kernel fusion variant treats S as all-ones in fusedSpMM -- the ALS pattern IS all-ones, so it agrees too
    for alg, p, c in [("15d_fusion2", 1, 1), ("15d_sparse", 1, 1), ("25d_dense_replicate", 1, 1), ("25d_sparse_replicate", 1, 1),
                      ("15d_fusion1", 4, 2), ("15d_fusion2", 8, 2), ("15d_sparse", 4, 1), ("25d_dense_replicate", 8, 2),
                      ("25d_sparse_replicate", 4, 1)]:
        out = ref.als(alg, p, c, R, N, rows, cols, Agt, Bgt, A0, B0)
        for k in (0, 1):
            assert abs(out["residual"][k] - base["residual"][k]) <= 1e-9 * base["residual"][0], (alg, p, c, out["residual"])
        assert np.abs(out["A"] - base["A"]).max() <= 1e-8 * np.abs(base["A"]).max(), (alg, p, c)
        assert np.abs(out["B"] - base["B"]).max() <= 1e-8 * np.abs(base["B"]).max(), (alg, p, c)
