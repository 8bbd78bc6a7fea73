"""The global model of the GAT backward pass (tests/gat_backward_model.py) on the CPU: against torch autograd on a
torch restatement of the forward pass, and against central finite differences; plus argument validation of the
backward-pass entry points of the C ABI without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import hnh_oracle as orc
from tests.gat_backward_model import gat_backward_global, kink_margins
from tests.mp_worker import gat_inputs

LOGM, NPR, SEED = 7, 6, 0xC0FFEE + 3
LAYERS = [[6, 4, 2], [8, 3, 3]]
ALPHA = 0.2


@pytest.fixture(scope="module")
def problem():
    N = 1 << LOGM
    rows, cols, _ = orc.er_tuples(LOGM, NPR, SEED)
    layers, X0, weights = gat_inputs(N, LAYERS, SEED)
    Ybar = np.random.default_rng(SEED + 5).uniform(-1, 1, (N, layers[-1][1] * layers[-1][2]))
    return dict(N=N, rows=rows, cols=cols, layers=layers, X0=X0, weights=weights, Ybar=Ybar)


def torch_forward(rows, cols, N, layers, weights, alpha, X0):
    """gat_forward_global in torch (edge list in S's CSR order; SpMM as index_add), differentiable."""
    order = np.lexsort((cols, rows))
    ri = torch.from_numpy(rows[order].astype(np.int64))
    ci = torch.from_numpy(cols[order].astype(np.int64))
    X = X0
    for (fin, fph, heads), ws in zip(layers, weights):
        outs = []
        for h in range(heads):
            H = X @ ws[h]
            e = (H[ri] * H[ci]).sum(1)
            a = torch.nn.functional.leaky_relu(e, alpha)
            Z = torch.zeros(N, fph, dtype=torch.float64).index_add(0, ri, a[:, None] * H[ci])
            outs.append(torch.relu(Z))
        X = torch.cat(outs, 1)
    return X


def test_inputs_keep_clear_of_the_kinks(problem):
    """No edge score and no pre-ReLU output of a row with edges within 1e-8 of 0, so that the derivative conventions
    at the kinks (ReLU'(0) = 0, LeakyReLU'(0) = alpha) cannot decide any comparison below."""
    P = problem
    assert len(np.unique(P["rows"])) == P["N"], "every row needs an edge: a zero row makes edge scores exactly 0"
    min_e, min_z = kink_margins(P["rows"], P["cols"], P["N"], P["layers"], P["weights"], ALPHA, P["X0"])
    assert min_e > 1e-8 and min_z > 1e-8, (min_e, min_z)


def test_backward_model_matches_torch_autograd(problem):
    P = problem
    X0 = torch.tensor(P["X0"], requires_grad=True)
    ws = [[torch.tensor(w, requires_grad=True) for w in heads] for heads in P["weights"]]
    Y = torch_forward(P["rows"], P["cols"], P["N"], P["layers"], ws, ALPHA, X0)
    want_Y = orc.gat_forward_global(P["rows"], P["cols"], P["N"], P["layers"], P["weights"], ALPHA, P["X0"])
    assert np.abs(Y.detach().numpy() - want_Y).max() <= 1e-13 * np.abs(want_Y).max()
    assert (want_Y > 0).mean() > 0.2
    (Y * torch.from_numpy(P["Ybar"])).sum().backward()
    dW, dX0 = gat_backward_global(P["rows"], P["cols"], P["N"], P["layers"], P["weights"], ALPHA, P["X0"], P["Ybar"])
    for i, heads in enumerate(ws):
        for h, w in enumerate(heads):
            g = w.grad.numpy()
            assert np.abs(dW[i][h] - g).max() <= 1e-12 * np.abs(g).max(), (i, h)
    g = X0.grad.numpy()
    assert np.abs(dX0 - g).max() <= 1e-12 * np.abs(g).max()
    assert np.abs(g).max() > 0


def test_backward_model_matches_finite_differences(problem):
    P = problem
    rng = np.random.default_rng(11)
    dW, dX0 = gat_backward_global(P["rows"], P["cols"], P["N"], P["layers"], P["weights"], ALPHA, P["X0"], P["Ybar"])

    def loss(weights, X0):
        return float((orc.gat_forward_global(P["rows"], P["cols"], P["N"], P["layers"], weights, ALPHA, X0) * P["Ybar"]).sum())

    step = 1e-6
    checked = 0
    for _ in range(14):  # weight coordinates, every layer
        i = int(rng.integers(len(P["layers"])))
        h = int(rng.integers(P["layers"][i][2]))
        r, c = (int(rng.integers(n)) for n in P["weights"][i][h].shape)
        plus = [[w.copy() for w in heads] for heads in P["weights"]]
        minus = [[w.copy() for w in heads] for heads in P["weights"]]
        plus[i][h][r, c] += step
        minus[i][h][r, c] -= step
        fd = (loss(plus, P["X0"]) - loss(minus, P["X0"])) / (2 * step)
        assert abs(fd - dW[i][h][r, c]) <= 1e-6 * max(1.0, abs(fd)), (i, h, r, c, fd, dW[i][h][r, c])
        checked += 1
    for _ in range(6):  # input coordinates
        r, c = int(rng.integers(P["N"])), int(rng.integers(P["layers"][0][0]))
        plus, minus = P["X0"].copy(), P["X0"].copy()
        plus[r, c] += step
        minus[r, c] -= step
        fd = (loss(P["weights"], plus) - loss(P["weights"], minus)) / (2 * step)
        assert abs(fd - dX0[r, c]) <= 1e-6 * max(1.0, abs(fd)), (r, c, fd, dX0[r, c])
        checked += 1
    assert checked == 20


def test_backward_entry_points_validate_without_a_gpu(hnh):
    assert hnh.hnh_dgemm_tn_f64(None, None, None, -1, 4, 4, None) == -1
    assert b"bad shape" in hnh.hnh_last_error_string()
    assert hnh.hnh_dgemm_tn_f64(None, None, None, 4, 1 << 31, 4, None) == -1
    assert hnh.hnh_dgemm_tn_f64(None, None, None, 4, 0, 4, None) == 0     # empty C
    assert hnh.hnh_dgemm_tn_f64(None, None, None, 4, 4, 4, None) == -1    # null pointers
    assert hnh.hnh_dgemm_nt_f64(None, None, None, 4, 4, 4, 0.5, None) == -1
    assert b"beta" in hnh.hnh_last_error_string()
    assert hnh.hnh_dgemm_nt_f64(None, None, None, 4, -1, 4, 0.0, None) == -1
    assert hnh.hnh_dgemm_nt_f64(None, None, None, 0, 4, 4, 1.0, None) == 0
    assert hnh.hnh_relu_cols_backward_f64(None, None, None, 4, 2, 3, 3, None) == -1  # window past the row end
    assert hnh.hnh_relu_cols_backward_f64(None, None, None, 4, 0, 0, 3, None) == 0
    assert hnh.hnh_leaky_relu_slope_f64(None, None, -1, 0.2, None) == -1
    assert hnh.hnh_leaky_relu_slope_f64(None, None, 0, 0.2, None) == 0


def test_backward_compute_without_gpu_fails_loudly(hnh):
    if torch.cuda.is_available():
        pytest.skip("box has a GPU")
    buf = (C.c_double * 64)()
    p = C.addressof(buf)
    assert hnh.hnh_dgemm_tn_f64(p, p, p, 4, 2, 2, None) == -2
    assert hnh.hnh_dgemm_tn_f64(p, p, p, 100000, 2, 2, None) == -2  # split over row chunks
    assert hnh.hnh_dgemm_nt_f64(p, p, p, 4, 2, 2, 1.0, None) == -2
    assert hnh.hnh_relu_cols_backward_f64(p, p, p, 4, 0, 2, 4, None) == -2
    assert hnh.hnh_leaky_relu_slope_f64(p, p, 8, 0.2, None) == -2
