"""GAT backward pass on the GPU: the new kernels against numpy, GAT::backwardPass against the global model
(tests/gat_backward_model.py) on one rank for every algorithm and on 2 and 4 ranks for the layouts that support it,
and SGD steps."""
import numpy as np
import pytest
import torch

from distributed_sddmm_b200 import driver as D
from oracle import hnh_oracle as orc
from tests.gat_backward_model import gat_backward_global, kink_margins
from tests.mp_gat_backward_worker import output_grad, run_cases
from tests.mp_worker import gat_inputs

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


def test_backward_kernels_match_numpy(world):
    from distributed_sddmm_b200 import lib
    L = lib()
    dev = torch.device("cuda:0")
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(7)
    cuda = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    # C (k x n) = A^T B: ragged tiles, several K tiles, one and many row chunks
    for m, n, k in ((70, 11, 19), (1, 1, 1), (256, 64, 64), (300, 130, 37), (5000, 8, 12), (100000, 32, 130), (99999, 70, 3)):
        A, B = rng.uniform(-1, 1, (m, k)), rng.uniform(-1, 1, (m, n))
        dA, dB = cuda(A), cuda(B)
        dC = torch.full((k, n), float("nan"), dtype=torch.float64, device=dev)
        D.check(L.hnh_dgemm_tn_f64(dC.data_ptr(), dA.data_ptr(), dB.data_ptr(), m, n, k, st))
        torch.cuda.synchronize()
        got = dC.cpu().numpy()
        assert rel_err(got, A.T @ B) < 1e-13, (m, n, k)
        D.check(L.hnh_dgemm_tn_f64(dC.data_ptr(), dA.data_ptr(), dB.data_ptr(), m, n, k, st))
        torch.cuda.synchronize()
        assert np.array_equal(dC.cpu().numpy(), got), ("repeated call differs", m, n, k)
    dC = torch.full((3, 4), float("nan"), dtype=torch.float64, device=dev)
    D.check(L.hnh_dgemm_tn_f64(dC.data_ptr(), None, None, 0, 4, 3, st))  # no rows: zero
    torch.cuda.synchronize()
    assert not dC.cpu().numpy().any()
    # C (m x n) = A B^T (+ C)
    for m, n, k in ((70, 11, 19), (1, 1, 1), (64, 64, 16), (300, 130, 37), (5, 200, 3), (100000, 128, 32)):
        A, B, C0 = rng.uniform(-1, 1, (m, k)), rng.uniform(-1, 1, (n, k)), rng.uniform(-1, 1, (m, n))
        dA, dB = cuda(A), cuda(B)
        dC = torch.full((m, n), float("nan"), dtype=torch.float64, device=dev)
        D.check(L.hnh_dgemm_nt_f64(dC.data_ptr(), dA.data_ptr(), dB.data_ptr(), m, n, k, 0.0, st))
        torch.cuda.synchronize()
        assert rel_err(dC.cpu().numpy(), A @ B.T) < 1e-13, (m, n, k)
        dC = cuda(C0)
        D.check(L.hnh_dgemm_nt_f64(dC.data_ptr(), dA.data_ptr(), dB.data_ptr(), m, n, k, 1.0, st))
        torch.cuda.synchronize()
        assert rel_err(dC.cpu().numpy(), C0 + A @ B.T) < 1e-13, (m, n, k)
    # LeakyReLU slope and the ReLU-window gradient, with exact zeros
    x = rng.uniform(-1, 1, 10007)
    x[::7] = 0.0
    dx, dy = cuda(x), torch.empty(x.size, dtype=torch.float64, device=dev)
    D.check(L.hnh_leaky_relu_slope_f64(dy.data_ptr(), dx.data_ptr(), x.size, 0.25, st))
    torch.cuda.synchronize()
    assert np.array_equal(dy.cpu().numpy(), np.where(x > 0, 1.0, 0.25))
    grad, out = rng.uniform(-1, 1, (33, 17)), np.maximum(rng.uniform(-1, 1, (33, 17)), 0.0)
    assert (out == 0).any()
    dd = torch.full((33, 5), float("nan"), dtype=torch.float64, device=dev)
    dgrad, dout = cuda(grad), cuda(out)
    D.check(L.hnh_relu_cols_backward_f64(dd.data_ptr(), dgrad.data_ptr(), dout.data_ptr(), 17, 10, 33, 5, st))
    torch.cuda.synchronize()
    assert np.array_equal(dd.cpu().numpy(), np.where(out[:, 10:15] > 0, grad[:, 10:15], 0.0))


def p1_problem(logM, npr, layer_spec):
    N = 1 << logM
    rows, cols, _ = orc.er_tuples(logM, npr, SEED)
    layers, X0, weights = gat_inputs(N, layer_spec, SEED)
    # keep the comparison away from the derivative kinks (see tests/test_gat_backward_oracle.py)
    assert min(kink_margins(rows, cols, N, layers, weights, 0.2, X0)) > 1e-8
    return N, rows, cols, layers, X0, weights


@pytest.mark.parametrize("layer_spec", [[[12, 8, 2], [16, 4, 3]], [[64, 32, 2]]], ids=["two_layers", "r32"])
@pytest.mark.parametrize("name", ALGS)
def test_p1_gat_backward_matches_global_model(world, name, layer_spec):
    logM, npr = 8, 6
    N, rows, cols, layers, X0, weights = p1_problem(logM, npr, layer_spec)
    alg = D.Algorithm(name, D.SpmatLocal.load_er(logM, npr, SEED), layers[0][0], 1)
    net = D.GAT(alg, layers, 0.2)
    for i, (fin, fph, heads) in enumerate(layers):
        for h in range(heads):
            net.set_weight(i, h, weights[i][h])
    net.set_input(X0)
    net.forward()
    assert net.supports_backward()
    Ybar = output_grad(N, layers, SEED)
    net.backward(Ybar)
    dW, dX0 = gat_backward_global(rows, cols, N, layers, weights, 0.2, X0, Ybar)
    for i, (fin, fph, heads) in enumerate(layers):
        for h in range(heads):
            assert rel_err(net.weight_grad(i, h), dW[i][h]) < RTOL, (i, h)
    assert rel_err(net.input_grad(), dX0) < RTOL
    # the pass overwrites: a second call gives the same gradients, bit for bit
    first = net.weight_grad(0, 0)
    net.backward(Ybar)
    assert np.array_equal(net.weight_grad(0, 0), first)


def test_sgd_steps_lower_the_loss(world):
    """L = 1/2 |Y - T|^2 on a tiny problem: every step is W - lr * W_grad exactly, and L goes down."""
    logM, npr = 6, 4
    N, rows, cols, layers, X0, weights = p1_problem(logM, npr, [[8, 4, 2]])
    T = np.random.default_rng(3).uniform(0, 1, (N, 8))
    alg = D.Algorithm("15d_fusion1", D.SpmatLocal.load_er(logM, npr, SEED), 8, 1)
    net = D.GAT(alg, layers, 0.2)
    for h in range(2):
        net.set_weight(0, h, weights[0][h])
    net.set_input(X0)
    lr = 2.0 ** -16  # a power of two: lr * W_grad is exact, so W - lr * W_grad has one rounding on either side
    losses = []
    for step in range(3):
        net.forward()
        Y = net.buffer(1)
        losses.append(0.5 * ((Y - T) ** 2).sum())
        net.backward(Y - T)
        before = [net.weight(0, h) for h in range(2)]
        grads = [net.weight_grad(0, h) for h in range(2)]
        net.sgd_step(lr)
        for h in range(2):
            assert np.array_equal(net.weight(0, h), before[h] - lr * grads[h]), (step, h)
    net.forward()
    losses.append(0.5 * ((net.buffer(1) - T) ** 2).sum())
    assert all(b < a for a, b in zip(losses, losses[1:])), losses


BACKWARD = dict(logM=7, npr=6, seed=SEED, layers=[[6, 4, 2], [8, 3, 3]], alpha=0.2, lr=2.0 ** -12)
SUPPORTED = {"fusion1_c1", "fusion1_c2", "fusion2_c1"}


def multirank_cases(nproc):
    # the sparse-shift algorithm splits R over p / c, so it runs here with c = p (head widths 4 and 3)
    return [dict(BACKWARD, name=f"{alg}_c{c}", alg=f"15d_{alg}", c=c)
            for alg, c in (("fusion1", 1), ("fusion1", 2), ("fusion2", 1), ("fusion2", 2), ("sparse", nproc))]


@pytest.mark.parametrize("nproc", [2, 4])
def test_multirank_gat_backward_matches_global_model(nproc):
    """Each rank's rows of the input gradient and the weight gradients against the global model; the weight gradients,
    and the weights after an SGD step, bit-identical on every rank.  Layouts whose forward pass is not the global
    formula refuse the backward pass."""
    c0 = BACKWARD
    N = 1 << c0["logM"]
    rows, cols, _ = orc.er_tuples(c0["logM"], c0["npr"], c0["seed"])
    layers, X0, weights = gat_inputs(N, c0["layers"], c0["seed"])
    assert min(kink_margins(rows, cols, N, layers, weights, c0["alpha"], X0)) > 1e-8
    dW, dX0 = gat_backward_global(rows, cols, N, layers, weights, c0["alpha"], X0, output_grad(N, layers, c0["seed"]))
    # one GPU per rank (NCCL) where there are enough, else ranks sharing one GPU over gloo, as in test_multirank_gpu.py
    transport = "nccl" if torch.cuda.device_count() >= nproc else "gloo"
    cases = multirank_cases(nproc)
    got = run_cases(nproc, cases, transport)
    for case in cases:
        ranks = got[case["name"]]
        if case["name"] not in SUPPORTED:
            for r, out in enumerate(ranks):
                assert int(out["supports"]) == 0, (case["name"], r)
                assert int(out["backward_rc"]) == -1, (case["name"], r, int(out["backward_rc"]))
                assert "GAT::backwardPass" in str(out["backward_msg"]), (case["name"], r, str(out["backward_msg"]))
            continue
        covered = np.zeros(N, bool)
        for r, out in enumerate(ranks):
            assert int(out["supports"]) == 1, (case["name"], r)
            top, g = int(out["top_b"]), out["input_grad"]
            hi = min(top + g.shape[0], N)
            assert rel_err(g[:hi - top], dX0[top:hi]) < RTOL, (case["name"], r)
            covered[top:hi] = True
            for i, (fin, fph, heads) in enumerate(layers):
                for h in range(heads):
                    k = f"wgrad_{i}_{h}"
                    assert rel_err(out[k], dW[i][h]) < RTOL, (case["name"], r, k)
                    assert np.array_equal(out[k], ranks[0][k]), (case["name"], r, k, "differs between ranks")
                    w = f"weight_{i}_{h}"
                    assert np.array_equal(out[w], ranks[0][w]), (case["name"], r, w, "differs between ranks")
                    assert np.array_equal(out[w], weights[i][h] - case["lr"] * out[k]), (case["name"], r, w)
        assert covered.all(), case["name"]
