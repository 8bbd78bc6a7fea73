"""Global numpy/scipy model of the GAT backward pass (include/hnh/gat.hpp, GAT::backwardPass).

The reference has no backward pass (its gat.hpp:42-48 calls it work in progress), so unlike oracle/hnh_oracle.py
this model is not pinned against the reference's code: tests/test_gat_backward_oracle.py pins it against torch
autograd on a restatement of oracle.hnh_oracle.gat_forward_global, and against central finite differences."""
import numpy as np


def gat_backward_global(rows, cols, N, layers, weights, alpha, X0, Ybar):
    """Gradients of L through gat_forward_global, given Ybar = dL/d(output of the last layer): returns
    (dW[layer][head], dX0).  Follows the forward pass line for line, with torch's derivative conventions
    ReLU'(0) = 0 and LeakyReLU'(x) = 1 if x > 0 else alpha."""
    import scipy.sparse as sp

    S = sp.csr_matrix((np.ones(len(rows)), (rows.astype(np.int64), cols.astype(np.int64))), shape=(N, N))
    S.sort_indices()
    ri = np.repeat(np.arange(N), np.diff(S.indptr))
    ci = S.indices
    # the forward pass, keeping every layer's input and output
    Xs = [np.asarray(X0, np.float64)]
    for (fin, fph, heads), ws in zip(layers, weights):
        out = np.zeros((N, fph * heads))
        for h in range(heads):
            H = Xs[-1] @ np.asarray(ws[h], np.float64)
            e = np.einsum("ij,ij->i", H[ri], H[ci])
            a = np.maximum(e, 0.0) + np.minimum(e, 0.0) * alpha
            Z = sp.csr_matrix((a, ci, S.indptr), shape=(N, N)) @ H
            out[:, h * fph:(h + 1) * fph] = np.maximum(Z, 0.0)
        Xs.append(out)
    # and back
    grad = np.asarray(Ybar, np.float64)
    dW = [None] * len(layers)
    for i in reversed(range(len(layers))):
        fin, fph, heads = layers[i]
        X, Y = Xs[i], Xs[i + 1]
        dX = np.zeros_like(X)
        dW[i] = []
        for h in range(heads):
            W = np.asarray(weights[i][h], np.float64)
            win = slice(h * fph, (h + 1) * fph)
            H = X @ W
            e = np.einsum("ij,ij->i", H[ri], H[ci])
            a = np.maximum(e, 0.0) + np.minimum(e, 0.0) * alpha
            G = np.where(Y[:, win] > 0, grad[:, win], 0.0)                              # through the ReLU
            de = np.einsum("ij,ij->i", G[ri], H[ci]) * np.where(e > 0, 1.0, alpha)     # through Z = aH, LeakyReLU
            Ed = sp.csr_matrix((de, ci, S.indptr), shape=(N, N))
            Ea = sp.csr_matrix((a, ci, S.indptr), shape=(N, N))
            dH = Ed @ H + Ed.T @ H + Ea.T @ G  # e_uv = <H_u, H_v> (both ends of an edge), Z = aH
            dW[i].append(X.T @ dH)
            dX += dH @ W.T
        grad = dX
    return dW, grad


def kink_margins(rows, cols, N, layers, weights, alpha, X0):
    """Smallest |e| over all edge scores and smallest |Z| over all pre-ReLU outputs of rows with at least one edge,
    over every head of every layer: how far the inputs are from the points where a derivative convention decides."""
    import scipy.sparse as sp

    S = sp.csr_matrix((np.ones(len(rows)), (rows.astype(np.int64), cols.astype(np.int64))), shape=(N, N))
    S.sort_indices()
    ri = np.repeat(np.arange(N), np.diff(S.indptr))
    has_edges = np.diff(S.indptr) > 0
    X = np.asarray(X0, np.float64)
    min_e, min_z = np.inf, np.inf
    for (fin, fph, heads), ws in zip(layers, weights):
        out = np.zeros((N, fph * heads))
        for h in range(heads):
            H = X @ np.asarray(ws[h], np.float64)
            e = np.einsum("ij,ij->i", H[ri], H[S.indices])
            min_e = min(min_e, np.abs(e).min())
            a = np.maximum(e, 0.0) + np.minimum(e, 0.0) * alpha
            Z = sp.csr_matrix((a, S.indices, S.indptr), shape=(N, N)) @ H
            min_z = min(min_z, np.abs(Z[has_edges]).min())
            out[:, h * fph:(h + 1) * fph] = np.maximum(Z, 0.0)
        X = out
    return min_e, min_z
