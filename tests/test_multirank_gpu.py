"""Multi-rank parity ON THE GPU against the REFERENCE's own code (oracle/_ref, or the committed
golden files generated from it by scripts/make_golden.py): every public operation of every algorithm, rank by rank --
local value order bit-exact, fp64 outputs within 1e-11 relative (contract: 1e-5).

How the ranks are mapped: with at least `nproc` GPUs each rank gets its own GPU and the ring
shifts / collectives are NCCL; on a one-GPU box the ranks are processes sharing cuda:0 and the
External transport (gloo, device buffers staged through pinned memory) carries the messages, so
the algorithm code under test is identical."""
import json
import os

import numpy as np
import pytest
import torch

from tests import golden_util as G
from tests import mp_util as U

pytestmark = pytest.mark.gpu

CASES = {
    2: [dict(U.case("15d_fusion1", 1, 8, 7, 5), als=1), U.case("15d_fusion1", 2, 8, 7, 5), U.case("15d_fusion2", 1, 8, 7, 5),
        U.case("15d_fusion2", 2, 8, 7, 5), U.case("15d_sparse", 1, 8, 7, 5), U.case("15d_sparse", 2, 8, 7, 5),
        U.case("25d_sparse_replicate", 2, 8, 7, 5),
        U.case("15d_fusion2", 1, 8, 7, 5, n=101), U.case("15d_sparse", 1, 8, 7, 5, n=101),  # padded trailing blocks
        # wide factors (the r = 128 kernels)
        U.case("15d_fusion2", 1, 128, 9, 6, name="fusion2_r128"),
        U.case("15d_fusion1", 1, 128, 9, 6, name="fusion1_r128")],
    4: [U.case("15d_fusion1", 2, 8, 7, 5), dict(U.case("15d_fusion2", 1, 16, 7, 5), als=1), U.case("15d_fusion2", 4, 8, 7, 5),
        U.case("15d_sparse", 1, 8, 7, 5), dict(U.case("15d_sparse", 2, 32, 7, 5), als=1), dict(U.case("25d_dense_replicate", 1, 8, 7, 5), als=1),
        U.case("25d_sparse_replicate", 1, 8, 7, 5),
        U.case("15d_fusion1", 2, 8, 7, 5, n=99), U.case("25d_dense_replicate", 1, 8, 7, 5, n=99)],
    8: [U.case("15d_fusion1", 2, 8, 8, 5), U.case("15d_fusion2", 1, 8, 8, 5), U.case("15d_sparse", 1, 32, 8, 5),
        U.case("25d_dense_replicate", 2, 8, 8, 5), U.case("25d_sparse_replicate", 2, 8, 8, 5),
        U.case("15d_fusion2", 2, 128, 10, 6, name="fusion2_r128_p8")],
}


def transport_for(nproc):
    return "nccl" if torch.cuda.device_count() >= nproc else "gloo"


@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_all_operations_match_reference(nproc):
    cases = CASES[nproc]
    got = U.run_cases(nproc, cases, transport_for(nproc), timeout=900)
    checked, worst = 0, 0.0
    for c in cases:
        want, src = U.reference_for(c, nproc)
        assert want is not None, f"no reference for {c['name']} (p={nproc}): run scripts/make_golden.py"
        try:
            U.compare_layout(got[c["name"]], want, c["alg"])
            worst = max(worst, U.compare_ops(got[c["name"]], want, c["script"]))
        except AssertionError as e:
            raise AssertionError(f"case {c['name']} (p={nproc}, reference from {src}): {e}") from e
        checked += 1
    assert checked > 0, "neither oracle/_ref/libhnh_ref.so nor tests/golden files are available"
    # ALS-CG (the config-5 caller) on the same algorithm objects: runs on every layout, all ranks agree on
    # the world-reduced residual, and one alternating round shrinks it
    for c in cases:
        if c.get("als"):
            res = [r["als"] for r in got[c["name"]]]
            assert all(np.array_equal(res[0], x) for x in res), (c["name"], res)
            assert np.isfinite(res[0]).all() and res[0][1] < res[0][0], (c["name"], res[0])
    print(f"nproc={nproc}: {checked} cases, worst relative error {worst:.2e}")


GAT = dict(layers=[[6, 4, 2], [8, 3, 3]], alpha=0.2)
GAT_CASES = {
    2: [dict(U.case("15d_fusion1", 1, 6, 7, 5, script=[], name="gat_fusion1_c1"), gat=GAT),
        dict(U.case("15d_fusion2", 1, 6, 7, 5, script=[], name="gat_fusion2_c1"), gat=GAT),
        dict(U.case("15d_fusion2", 2, 6, 7, 5, script=[], name="gat_fusion2_c2"), gat=GAT)],
    4: [dict(U.case("15d_fusion1", 2, 6, 7, 5, script=[], name="gat_fusion1_c2"), gat=GAT),
        dict(U.case("15d_fusion2", 1, 6, 7, 5, script=[], name="gat_fusion2_c1"), gat=GAT)],
}


@pytest.mark.parametrize("nproc", [2, 4])
def test_gat_forward_matches_reference(nproc):
    """GAT forward pass (include/hnh/gat.hpp) rank by rank against the reference's gat.hpp run by oracle/_ref --
    including the fusion-2, c > 1 case where the reference's SpMM pass accumulates onto the gathered
    projection (15D_dense_shift.hpp:306-314 with initial_replicate = false)."""
    cases = GAT_CASES[nproc]
    got = U.run_cases(nproc, cases, transport_for(nproc), timeout=900)
    for c in cases:
        want, _ = gat_reference(c, nproc)
        for r in range(nproc):
            have, w = got[c["name"]][r]["gat_out"], want[f"r{r}_gat_out"]
            assert have.shape == tuple(w.shape), (c["name"], r, have.shape, w.shape)
            err = G.rel_err(have, w)
            assert err < 1e-11, (c["name"], r, err)


def gat_reference(c, nproc):
    """Every rank's GAT output of the reference's gat.hpp (oracle/_ref, or its golden file)."""
    def compute():
        from oracle import hnh_oracle as orc
        from oracle import ref
        from tests.mp_worker import gat_inputs
        N = 1 << c["logM"]
        rows, cols, _ = orc.er_tuples(c["logM"], c["npr"], c["seed"])
        layers, X0, weights = gat_inputs(N, c["gat"]["layers"], c["seed"])
        _, per_rank = ref.gat(c["alg"], nproc, c["c"], N, rows, cols, np.ones(len(rows)), layers, weights, c["gat"]["alpha"], X0)
        return {f"r{r}_gat_out": out for r, (out, _) in enumerate(per_rank)}
    return U.reference_arrays(f"{c['name']}_p{nproc}", compute)


HOSTPIPE_CASES = {
    2: [dict(U.case("15d_fusion2", 1, 8, 7, 5, script=[], name="hostpipe_c1_chunk24"), hostpipe=24),
        dict(U.case("15d_fusion2", 1, 8, 7, 5, script=[], name="hostpipe_c1_default"), hostpipe=0),
        dict(U.case("15d_fusion2", 2, 8, 7, 5, script=[], name="hostpipe_c2_plain"), hostpipe=16),   # c > 1: plain copy-in / copy-out
        dict(U.case("15d_fusion1", 1, 8, 7, 5, script=[], name="hostpipe_fusion1_plain"), hostpipe=16)],
    4: [dict(U.case("15d_fusion2", 1, 8, 7, 5, script=[], name="hostpipe_c1_chunk8"), hostpipe=8),
        dict(U.case("15d_fusion2", 1, 8, 7, 5, script=[], name="hostpipe_c1_n99", n=99), hostpipe=8)],
}


@pytest.mark.parametrize("nproc", [2, 4])
def test_fused_host_operands_multirank(nproc):
    """Distributed_Sparse::fusedSpMM_host on several ranks: bit-identical with upload + fusedSpMM + download (the blocks
    of a row are visited in the ring's order), for both modes, and the staging matrix ends up holding the result."""
    cases = HOSTPIPE_CASES[nproc]
    got = U.run_cases(nproc, cases, transport_for(nproc), timeout=900)
    for c in cases:
        for r, rank_out in enumerate(got[c["name"]]):
            for mode in ("A", "B"):
                want = rank_out[f"hostpipe_{mode}_want"]
                assert np.array_equal(rank_out[f"hostpipe_{mode}_got"], want), (c["name"], r, mode)
                assert np.array_equal(rank_out[f"hostpipe_{mode}_staged"], want), (c["name"], r, mode)


ALS_CASES = {
    2: [dict(U.case("15d_fusion1", 1, 8, 7, 5, script=[], name="alsp_fusion1_c1"), als_parity=1),
        dict(U.case("15d_fusion2", 2, 8, 7, 5, script=[], name="alsp_fusion2_c2"), als_parity=1),
        dict(U.case("15d_sparse", 1, 8, 7, 5, script=[], name="alsp_sparse_c1"), als_parity=1)],
    4: [dict(U.case("15d_fusion2", 1, 8, 7, 5, script=[], name="alsp_fusion2_c1"), als_parity=1),
        dict(U.case("15d_sparse", 2, 8, 7, 5, script=[], name="alsp_sparse_c2"), als_parity=1),
        dict(U.case("25d_dense_replicate", 1, 8, 7, 5, script=[], name="alsp_25d_dense"), als_parity=1),
        dict(U.case("25d_sparse_replicate", 1, 8, 7, 5, script=[], name="alsp_25d_sparse"), als_parity=1)],
}


@pytest.mark.parametrize("nproc", [2, 4])
def test_als_cg_matches_reference_als(nproc):
    """BASELINE.json config 5's caller: one alternating round of batched CG (10 iterations per side) on given ground
    truth and starting embeddings, against the reference's own Distributed_ALS / cg_optimizer run by oracle/_ref --
    residuals and every rank's local embeddings.  Tolerance 1e-7 relative (contract 1e-5): 20 CG iterations separate
    the two summation orders."""
    cases = ALS_CASES[nproc]
    got = U.run_cases(nproc, cases, transport_for(nproc), timeout=900)
    for c in cases:
        want, _ = als_reference(c, nproc)
        for r in range(nproc):
            g = got[c["name"]][r]
            assert np.allclose(g["als_res"], want["residual"], rtol=1e-7, atol=0), (c["name"], r, g["als_res"], want["residual"])
            for have, w in ((g["als_A"], want[f"r{r}_A"]), (g["als_B"], want[f"r{r}_B"])):
                assert have.shape == tuple(w.shape), (c["name"], r)
                assert G.abs_err(have, w) <= 1e-7 * G.absmax(w), (c["name"], r)


def als_reference(c, nproc):
    """Residuals and every rank's local embeddings of the reference's Distributed_ALS (oracle/_ref, or its golden file)."""
    def compute():
        from oracle import hnh_oracle as orc
        from oracle import ref
        from tests.mp_worker import als_inputs
        N = 1 << c["logM"]
        rows, cols, _ = orc.er_tuples(c["logM"], c["npr"], c["seed"])
        want = ref.als(c["alg"], nproc, c["c"], c["R"], N, rows, cols, *als_inputs(N, c["R"], c["seed"]), 1, 10)
        out = {"residual": np.asarray(want["residual"])}
        for r, (wA, wB) in enumerate(want["ranks"]):
            out[f"r{r}_A"], out[f"r{r}_B"] = wA, wB
        return out
    return U.reference_arrays(f"{c['name']}_p{nproc}", compute)


RECT_CASES = {
    2: [U.case("15d_fusion2", 1, 8, 7, 5, n=120, m=75, name="rect_fusion2"),
        U.case("15d_fusion1", 2, 8, 7, 5, n=70, m=128, name="rect_fusion1"),
        U.case("15d_sparse", 2, 8, 7, 5, n=70, m=128, name="rect_sparse")],
    4: [U.case("15d_fusion1", 1, 8, 7, 5, n=100, m=61, name="rect_fusion1"),
        U.case("15d_fusion2", 2, 8, 7, 5, n=128, m=77, name="rect_fusion2"),
        U.case("15d_sparse", 1, 8, 7, 5, n=100, m=61, name="rect_sparse"),
        U.case("25d_dense_replicate", 1, 8, 7, 5, n=90, m=128, name="rect_25d_dense"),
        U.case("25d_sparse_replicate", 1, 8, 7, 5, n=128, m=77, name="rect_25d_sparse")],
}


@pytest.mark.parametrize("nproc", [2, 4])
def test_rectangular_matrices_match_reference(nproc):
    """M != N (more columns than rows and the reverse, sizes that do not divide evenly): every public operation of
    every algorithm against the reference's own code, as in test_all_operations_match_reference."""
    cases = RECT_CASES[nproc]
    got = U.run_cases(nproc, cases, transport_for(nproc), timeout=900)
    for c in cases:
        want, src = U.reference_for(c, nproc)
        try:
            U.compare_layout(got[c["name"]], want, c["alg"])
            U.compare_ops(got[c["name"]], want, c["script"])
        except AssertionError as e:
            raise AssertionError(f"case {c['name']} (p={nproc}, reference from {src}): {e}") from e


TINY_CASES = [U.case("15d_fusion1", 1, 4, 4, 1, name="tiny_fusion1"), U.case("15d_fusion2", 2, 4, 4, 1, name="tiny_fusion2"),
              U.case("15d_fusion2", 1, 4, 4, 1, name="tiny_fusion2_c1"), U.case("15d_sparse", 4, 4, 4, 1, name="tiny_sparse"),
              U.case("15d_sparse", 1, 4, 4, 1, name="tiny_sparse_c1"),
              U.case("25d_dense_replicate", 1, 4, 4, 1, name="tiny_25d_dense"),
              U.case("25d_sparse_replicate", 1, 4, 4, 1, name="tiny_25d_sparse")]


def test_null_and_empty_blocks_match_reference():
    """A 16 x 16 matrix with one nonzero per row on 4 ranks: most blocks are null or empty (the reference skips them,
    sparse_kernels.cpp:25-27,71-73,85-87); every operation must still agree with it."""
    got = U.run_cases(4, TINY_CASES, transport_for(4), timeout=900)
    for c in TINY_CASES:
        want, src = U.reference_for(c, 4)
        try:
            U.compare_layout(got[c["name"]], want, c["alg"])
            U.compare_ops(got[c["name"]], want, c["script"])
        except AssertionError as e:
            raise AssertionError(f"case {c['name']} (reference from {src}): {e}") from e


# Device-side setup (SURVEY.md 8f-3): tuples generated, bucketed by owner, exchanged, sorted and turned into CSR blocks
# in HBM.  Forced on for these small matrices (by default it starts at 2^18 tuples per rank); the per-rank layout must be
# the reference's bit for bit, and every operation must still agree with it.
DEVSETUP_CASES = {
    1: [U.case("15d_fusion2", 1, 8, 7, 5), U.case("15d_fusion1", 1, 8, 7, 5), U.case("15d_sparse", 1, 8, 7, 5),
        U.case("25d_dense_replicate", 1, 8, 7, 5), U.case("25d_sparse_replicate", 1, 8, 7, 5),
        U.case("15d_sparse", 1, 16, 14, 8, name="cfg1_15d_sparse", load="er", script=["sddmmA", "fusedA"])],
    2: CASES[2] + RECT_CASES[2],
    4: CASES[4] + RECT_CASES[4] + TINY_CASES,
}


@pytest.mark.parametrize("nproc", [1, 2, 4])
def test_device_side_setup_matches_reference(nproc):
    from oracle import ref
    cases = [dict(c, als=0) for c in DEVSETUP_CASES[nproc]]
    got = U.run_cases(nproc, cases, transport_for(nproc) if nproc > 1 else "self", timeout=900, env_extra={"HNH_DEVICE_SETUP": "1"})
    checked = 0
    for c in cases:
        want, src = U.reference_for(c, nproc)
        assert want is not None, f"no reference for {c['name']} (p={nproc}): run scripts/make_golden.py"
        info = json.loads(str(got[c["name"]][0]["setup_times"]))
        assert any("(device)" in k for k in info), (c["name"], "the device setup path did not run", info)
        try:
            U.compare_layout(got[c["name"]], want, c["alg"])
            U.compare_ops(got[c["name"]], want, c["script"])
        except AssertionError as e:
            raise AssertionError(f"case {c['name']} (p={nproc}, device setup, reference from {src}): {e}") from e
        checked += 1
    assert checked > 0


def test_peer_ring_failure_on_one_rank_is_a_collective_fallback():
    """A rank that cannot map its neighbours' buffers (injected: HNH_TEST_PEERRING_FAIL) must not leave the others in the
    ring's barrier: every rank releases what it acquired and all take the transport's send/recv path together -- same
    results, and the algorithm reports which ring it really used."""
    cases = [U.case("15d_fusion2", 1, 8, 7, 5), U.case("15d_sparse", 1, 8, 7, 5), U.case("15d_fusion1", 1, 8, 7, 5)]
    got = U.run_cases(2, cases, transport_for(2), timeout=600, env_extra={"HNH_TEST_PEERRING_FAIL": "1"})
    for c in cases:
        want, src = U.reference_for(c, 2)
        assert want is not None, f"no reference for {c['name']}: run scripts/make_golden.py"
        U.compare_layout(got[c["name"]], want, c["alg"])
        U.compare_ops(got[c["name"]], want, c["script"])
        for rank_out in got[c["name"]]:
            assert json.loads(str(rank_out["info"]))["ring"] == "send/recv of the transport", c["name"]
