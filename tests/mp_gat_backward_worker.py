"""Multi-process worker for the GAT backward-pass tests (launched by run_cases below, with the command line of
tests/mp_worker.py).  Every rank runs the forward pass, the backward pass from its rows of a seeded output gradient
and one SGD step, and writes <outdir>/<case>_rank<r>.npz with its row offsets, the gradients and the updated weights.  On a layout without a backward pass it records the return
code and message of hnhd_gat_backward instead."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests.mp_worker import gat_inputs, gather_local  # noqa: E402


def output_grad(N, layers, seed):
    """dL/d(network output) of the tests: seeded uniform(-1, 1), N x (heads * width of the last layer)."""
    fin, fph, heads = layers[-1]
    return np.random.default_rng(seed + 5).uniform(-1, 1, (N, fph * heads))


def run_cases(nproc, cases, transport, timeout=900):
    """This worker on nproc processes (torch.distributed.run, as tests/mp_util.run_cases does for mp_worker.py).
    Returns {case name: [per-rank dict]}."""
    from tests.mp_util import free_port
    with tempfile.TemporaryDirectory() as td:
        def launch():
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
                   "--master-addr", "127.0.0.1", "--master-port", str(free_port()), os.path.abspath(__file__),
                   json.dumps(cases), td, transport]
            return subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, OMP_NUM_THREADS="2"), stdout=subprocess.PIPE,
                                  stderr=subprocess.STDOUT, timeout=timeout, text=True)
        p = launch()
        if p.returncode != 0 and "Address already in use" in p.stdout:  # lost the race for the rendezvous port
            p = launch()
        if p.returncode != 0:
            raise RuntimeError("worker failed:\n" + p.stdout[-6000:])
        out = {}
        for case in cases:
            ranks = []
            for r in range(nproc):
                z = np.load(os.path.join(td, f"{case['name']}_rank{r}.npz"), allow_pickle=False)
                ranks.append({k: z[k] for k in z.files})
            out[case["name"]] = ranks
        return out


def main():
    cases = json.loads(sys.argv[1])
    outdir = sys.argv[2]
    transport = sys.argv[3]
    import torch
    if torch.cuda.is_available():
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")) % torch.cuda.device_count() if transport == "nccl" else 0)
    from distributed_sddmm_b200 import driver as D
    from distributed_sddmm_b200 import lib
    rank, world = D.world_init(transport)
    for case in cases:
        N = 1 << case["logM"]
        S = D.SpmatLocal.load_er(case["logM"], case["npr"], case["seed"])
        layers, X0, weights = gat_inputs(N, case["layers"], case["seed"])
        alg = D.Algorithm(case["alg"], S, layers[0][0], case["c"])
        net = D.GAT(alg, layers, case["alpha"])
        for i, (fin, fph, heads) in enumerate(layers):
            for h in range(heads):
                net.set_weight(i, h, weights[i][h])
        top_b = alg.submatrices("B")[0][0]
        top_a = alg.submatrices("A")[0][0]
        net.set_input(gather_local(X0, [(top_b, 0, net.buffer_shape(0)[0], layers[0][0])], net.buffer_shape(0)))
        net.forward()
        out_shape = net.buffer_shape(len(layers))
        grad = gather_local(output_grad(N, layers, case["seed"]), [(top_a, 0, out_shape[0], out_shape[1])], out_shape)
        out = dict(top_a=top_a, top_b=top_b, supports=int(net.supports_backward()))
        if out["supports"]:
            net.backward(grad)
            out["input_grad"] = net.input_grad()
            for i, (fin, fph, heads) in enumerate(layers):
                for h in range(heads):
                    out[f"wgrad_{i}_{h}"] = net.weight_grad(i, h)
            net.sgd_step(case["lr"])
            for i, (fin, fph, heads) in enumerate(layers):
                for h in range(heads):
                    out[f"weight_{i}_{h}"] = net.weight(i, h)
        else:
            g = np.ascontiguousarray(grad)
            out["backward_rc"] = lib().hnhd_gat_backward(net.h, g.ctypes.data)
            out["backward_msg"] = lib().hnh_last_error_string().decode()
        np.savez(os.path.join(outdir, f"{case['name']}_rank{rank}.npz"), **out)
        del net, alg, S
    D.world_finalize()


if __name__ == "__main__":
    main()
