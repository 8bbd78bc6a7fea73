#!/usr/bin/env python
"""GAT training step (include/hnh/gat.hpp: forwardPass, backwardPass, applyGradients) at the launched world size
(torchrun; one GPU per rank).  Workload: the config-2 matrix (Erdos-Renyi, N = 2^20, 32 nonzeros per row), layers
(128, 32, 4) x 2, for each algorithm in --algs.

Per algorithm: first a parity check at a small size against the global model (tests/gat_backward_model.py) -- every
rank checks its rows of the input gradient and the weight gradients, and the run stops if one is off by more than
1e-11 relative; then --warmup untimed training steps; then --steps timed ones, where forward, backward and the SGD step
are each timed with CUDA events on the compute stream and a synchronisation.  The backward call takes the output
gradient from (pinned) host memory, so its upload is timed on its own and reported next to it.  The sparse-operation
time is the algorithm's "Computation Time" counter over each phase.  Rank 0 prints one JSON line per algorithm (and
appends it to --out), with the GPU name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from distributed_sddmm_b200 import driver as D  # noqa: E402
from oracle import hnh_oracle as orc  # noqa: E402
from tests.gat_backward_model import gat_backward_global  # noqa: E402
from tests.mp_worker import gat_inputs, gather_local  # noqa: E402

SEED = 0xC0FFEE + 2  # config 2 (bench.py)


def gpu_info():
    """Name and power limit of this rank's GPU (a read-only nvidia-smi query)."""
    idx = torch.cuda.current_device()
    try:
        out = subprocess.run(["nvidia-smi", f"--id={idx}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the measurement stands; say that the card could not be read
        return dict(gpu=torch.cuda.get_device_name(idx), power_limit=f"unread ({e})")


def parity_check(name, c):
    """Small problem at this world size: this rank's gradients against the global model.  Returns the worst error."""
    logM, npr = 8, 6
    N = 1 << logM
    rows, cols, _ = orc.er_tuples(logM, npr, SEED)
    layers, X0, weights = gat_inputs(N, [[12, 8, 2], [16, 4, 3]], SEED)
    Ybar = np.random.default_rng(SEED + 5).uniform(-1, 1, (N, 12))
    alg = D.Algorithm(name, D.SpmatLocal.load_er(logM, npr, SEED), 12, c)
    top_b, top_a = alg.submatrices("B")[0][0], alg.submatrices("A")[0][0]
    net = D.GAT(alg, layers, 0.2)
    for i, (fin, fph, heads) in enumerate(layers):
        for h in range(heads):
            net.set_weight(i, h, weights[i][h])
    net.set_input(gather_local(X0, [(top_b, 0, net.buffer_shape(0)[0], 12)], net.buffer_shape(0)))
    net.forward()
    shape = net.buffer_shape(2)
    net.backward(gather_local(Ybar, [(top_a, 0, shape[0], shape[1])], shape))
    dW, dX0 = gat_backward_global(rows, cols, N, layers, weights, 0.2, X0, Ybar)
    rel = lambda got, ref: float(np.abs(got - ref).max() / np.abs(ref).max())  # noqa: E731
    g = net.input_grad()
    hi = min(top_b + g.shape[0], N)
    worst = rel(g[:hi - top_b], dX0[top_b:hi]) if hi > top_b else 0.0
    for i, (fin, fph, heads) in enumerate(layers):
        for h in range(heads):
            worst = max(worst, rel(net.weight_grad(i, h), dW[i][h]))
    del net, alg
    if not worst < 1e-11:
        raise SystemExit(f"parity check failed for {name} c={c}: relative error {worst:.3e}")
    return worst


def timed(fn):
    D.timer_start()
    fn()
    return D.timer_stop()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--logm", type=int, default=20)
    ap.add_argument("--npr", type=int, default=32)
    ap.add_argument("--algs", default="15d_fusion1,15d_fusion2")
    ap.add_argument("--c", type=int, default=1)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--lr", type=float, default=2.0 ** -20)
    ap.add_argument("--out", default=None, help="JSON-lines file rank 0 appends to")
    args = ap.parse_args()

    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    rank, world = D.world_init()
    info = gpu_info()
    layer_spec = [[128, 32, 4], [128, 32, 4]]
    S = D.SpmatLocal.load_er(args.logm, args.npr, SEED)
    for name in args.algs.split(","):
        worst = parity_check(name, args.c)
        alg = D.Algorithm(name, S, layer_spec[0][0], args.c)
        upload = alg.like_A_matrix()  # at R = 128: the shape of the output gradient, for timing its upload alone
        layers = [tuple(l) for l in layer_spec]
        # the same weights on every rank, scaled so that the activations stay O(1) through both layers
        wr = np.random.default_rng(SEED)
        weights = [[wr.uniform(-1, 1, (fin, fph)) * 0.05 for _ in range(heads)] for fin, fph, heads in layers]
        rng = np.random.default_rng(SEED + 1 + rank)  # this rank's rows of the input and of the output gradient
        net = D.GAT(alg, layers, 0.2)
        for i, (fin, fph, heads) in enumerate(layers):
            for h in range(heads):
                net.set_weight(i, h, weights[i][h])
        net.set_input(rng.uniform(-1, 1, net.buffer_shape(0)))
        out_shape = net.buffer_shape(len(layers))
        grad = torch.empty(out_shape, dtype=torch.float64, pin_memory=True).numpy()
        grad[:] = rng.uniform(-1, 1, out_shape)
        assert upload.shape == out_shape, (upload.shape, out_shape)

        def step():
            net.forward()
            net.backward(grad)
            net.sgd_step(args.lr)

        for _ in range(args.warmup):
            step()
        fwd, bwd, sgd, up = [], [], [], []
        comp = {"forward": 0.0, "backward": 0.0}
        for _ in range(args.steps):
            alg.reset_timers()
            fwd.append(timed(net.forward))
            comp["forward"] += alg.perf()["Computation Time"]
            alg.reset_timers()
            bwd.append(timed(lambda: net.backward(grad)))
            comp["backward"] += alg.perf()["Computation Time"]
            sgd.append(timed(lambda: net.sgd_step(args.lr)))
            up.append(timed(lambda: upload.from_host(grad)))
        med = lambda xs: float(np.median(xs))  # noqa: E731
        fwd_ms, bwd_ms, up_ms = med(fwd), med(bwd), med(up)
        comp_fwd_ms = comp["forward"] / args.steps * 1e3
        comp_bwd_ms = comp["backward"] / args.steps * 1e3
        if rank == 0:
            rec = dict(workload="gat_train", alg=name, c=args.c, p=world, logM=args.logm, nnz_per_row=args.npr,
                       layers=layer_spec, steps=args.steps, warmup=args.warmup, **info,
                       parity_max_rel_err_rank0=worst, parity_ok=True,
                       forward_ms=fwd_ms, backward_ms=bwd_ms, grad_upload_ms=up_ms, backward_minus_upload_ms=bwd_ms - up_ms,
                       sgd_step_ms=med(sgd), forward_ms_all=fwd, backward_ms_all=bwd, sgd_step_ms_all=sgd,
                       forward_sparse_ms=comp_fwd_ms, backward_sparse_ms=comp_bwd_ms,
                       forward_sparse_share=comp_fwd_ms / fwd_ms, backward_sparse_share=comp_bwd_ms / (bwd_ms - up_ms),
                       backward_over_forward_sparse=comp_bwd_ms / comp_fwd_ms)
            line = json.dumps(rec)
            print(line, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(line + "\n")
        del net, upload, alg
    del S
    D.world_finalize()


if __name__ == "__main__":
    main()
