"""Launch tests/mp_worker.py on N processes and load what the ranks wrote; reference-side helpers."""
import json
import os
import socket
import subprocess
import sys
import tempfile

import numpy as np

from tests import golden_util as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALL_OPS = ["sddmmA", "spmmA", "spmmB", "fusedA", "sddmmB", "fusedB"]


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def run_cases(nproc, cases, transport, timeout=600, env_extra=None):
    """Returns {case name: [per-rank dict]}.  env_extra: additional environment of the worker processes."""
    with tempfile.TemporaryDirectory() as td:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
               "--master-addr", "127.0.0.1", "--master-port", str(free_port()),
               os.path.join(ROOT, "tests", "mp_worker.py"), json.dumps(cases), td, transport]
        env = dict(os.environ, OMP_NUM_THREADS="2", **(env_extra or {}))
        p = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=timeout, text=True)
        if p.returncode != 0 and "Address already in use" in p.stdout:  # lost the race for the rendezvous port
            cmd[cmd.index("--master-port") + 1] = str(free_port())
            p = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=timeout, text=True)
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


def case(alg, c, R, logM, npr, seed=0xC0FFEE + 1, script=ALL_OPS, name=None, load="tuples", n=None, m=None):
    d = dict(name=name or f"{alg}_c{c}_R{R}_m{logM}" + (f"_n{n}" if n else "") + (f"_rows{m}" if m else ""), alg=alg, c=c, R=R,
             logM=logM, npr=npr, seed=seed, script=list(script), load=load)
    if n:
        d["n"] = n
    if m:
        d["m"] = m  # rectangular: m rows, n (or 2^logM) columns
    return d


def reference_for(case_, p):
    """The REFERENCE's per-rank view of the same case (oracle/_ref, or the committed golden file)."""
    from oracle import hnh_oracle as orc
    from oracle import ref
    from tests.mp_worker import global_inputs, sval
    N = case_.get("n") or (1 << case_["logM"])
    M = case_.get("m") or N
    rows, cols, _ = orc.er_tuples(case_["logM"], case_["npr"], case_["seed"], 0, M)
    keep = cols < N
    rows, cols = rows[keep], cols[keep]
    A, B = global_inputs(N, case_["R"], case_["seed"], M)
    golden = os.path.join(ROOT, "tests", "golden", f"{case_['name']}_p{p}.npz")
    if ref.available():
        vals = np.ones(len(rows)) if case_.get("load") == "er" else sval(rows, cols)
        ranks = ref.run(case_["alg"], p, case_["c"], case_["R"], M, N, rows, cols, vals, A, B, case_["script"])
        return ranks, "oracle/_ref"
    if os.path.exists(golden):
        return load_golden(golden, p), "tests/golden"
    return None, None


WRITE_GOLDEN = False  # set by scripts/make_golden.py: reference_arrays also stores what it computed


def reference_arrays(name, compute, exact=()):
    """A dict of reference arrays: `compute()` where oracle/_ref is built, else tests/golden/<name>.npz (written from
    the same `compute` by scripts/make_golden.py; the keys in `exact` are compared bit for bit, the others within a
    tolerance).  Returns (arrays, source)."""
    from oracle import ref
    path = os.path.join(ROOT, "tests", "golden", f"{name}.npz")
    if ref.available():
        arrays = compute()
        if WRITE_GOLDEN:
            out = {}
            for k, a in arrays.items():
                G.reduce_into(out, k, a, k in exact)
            G.save(path, out)
        return arrays, "oracle/_ref"
    z = G.open_golden(path)
    return {k: G.load(z, k) for k in {f.split("__")[0] for f in z.files}}, "tests/golden"


def flatten_ref(ranks, reduced=False, alg=None):
    """ref.run output -> flat dict of arrays (the golden-file format).  reduced: large arrays in the reduced form of
    tests/golden_util.py (layout: digests; operation outputs: sample + sketch)."""
    flat = {}
    put = (lambda k, a, exact: G.reduce_into(flat, k, a, exact)) if reduced else (lambda k, a, exact: flat.update({k: a}))
    for r, d in enumerate(ranks):
        for k in ("i", "j", "k", "localArows", "localAcols", "localBrows", "localBcols"):
            flat[f"r{r}_{k}"] = np.int64(d[k])
        for k in ("aSubmatrices", "bSubmatrices", "S_rows", "S_cols", "ST_rows", "ST_cols"):
            put(f"r{r}_{k}", d[k], True)
        for key in ("S", "ST"):
            flat[f"r{r}_{key}_nblocks"] = np.int64(len(d[key + "_blocks"]))
            for b, blk in enumerate(d[key + "_blocks"]):
                flat[f"r{r}_{key}_b{b}_null"] = np.bool_(blk is None)
                if blk is not None:
                    blk = dict(blk)
                    if reduced and alg == "25d_dense_replicate":  # see compare_layout: what this library must hold
                        blk["row_idx"] = np.repeat(np.arange(int(blk["rows"])), np.diff(np.asarray(blk["rowStart"])))
                    for f in ("rows", "cols", "transpose", "rowStart", "col_idx", "row_idx", "values"):
                        put(f"r{r}_{key}_b{b}_{f}", np.asarray(blk[f]), True)
        flat[f"r{r}_nops"] = np.int64(len(d["ops"]))
        for t, op in enumerate(d["ops"]):
            for f in ("A", "B", "values"):
                put(f"r{r}_op{t}_{f}", op[f], False)
    return flat


def load_golden(path, p):
    z = G.open_golden(path)
    ranks = []
    for r in range(p):
        g = lambda k: G.load(z, f"r{r}_{k}")  # noqa: E731
        d = {k: int(g(k)) for k in ("i", "j", "k", "localArows", "localAcols", "localBrows", "localBcols")}
        for k in ("aSubmatrices", "bSubmatrices", "S_rows", "S_cols", "ST_rows", "ST_cols"):
            d[k] = g(k)
        for key in ("S", "ST"):
            blocks = []
            for b in range(int(g(key + "_nblocks"))):
                if bool(g(f"{key}_b{b}_null")):
                    blocks.append(None)
                else:
                    blocks.append({f: g(f"{key}_b{b}_{f}") for f in ("rows", "cols", "transpose", "rowStart", "col_idx", "row_idx", "values")})
            d[key + "_blocks"] = blocks
        d["ops"] = [dict(A=g(f"op{t}_A"), B=g(f"op{t}_B"), values=g(f"op{t}_values")) for t in range(int(g("nops")))]
        ranks.append(d)
    return ranks


def compare_layout(got, want, alg):
    """Index / layout parity: bit-exact."""
    for r, (g, w) in enumerate(zip(got, want)):
        for k in ("i", "j", "k", "localArows", "localAcols", "localBrows", "localBcols"):
            assert int(g[k]) == int(w[k]), (r, k, int(g[k]), int(w[k]))
        assert G.same(g["aSubmatrices"], w["aSubmatrices"]), (r, "aSubmatrices")
        assert G.same(g["bSubmatrices"], w["bSubmatrices"]), (r, "bSubmatrices")
        for key in ("S", "ST"):
            wb = w[key + "_blocks"]
            assert int(g[key + "_nblocks"]) == len(wb), (r, key, "block count")
            for b, blk in enumerate(wb):
                assert bool(g[f"{key}_b{b}_null"]) == (blk is None), (r, key, b, "null-ness")
                if blk is None:
                    continue
                assert int(g[f"{key}_b{b}_rows"]) == int(blk["rows"]) and bool(g[f"{key}_b{b}_transpose"]) == bool(blk["transpose"])
                if alg != "15d_sparse":  # the reference declares too few columns there (15D_sparse_shift.hpp:132)
                    assert int(g[f"{key}_b{b}_cols"]) == int(blk["cols"])
                if len(blk["col_idx"]) == 0:
                    # an empty block: the reference builds it from one dummy (0, 0, 0.0) entry (SpmatLocal.hpp:93-97,
                    # 182-184), so its rowStart holds that entry's leftovers; nothing reads it (num_coords == 0)
                    assert len(g[f"{key}_b{b}_col_idx"]) == 0 and not np.any(g[f"{key}_b{b}_rowStart"]), (r, key, b, "empty block")
                    continue
                for f in ("rowStart", "col_idx", "row_idx", "values"):
                    have, ref_ = np.asarray(g[f"{key}_b{b}_{f}"]), blk[f]
                    if (f == "row_idx" and alg == "25d_dense_replicate" and not G.same(have, ref_)
                            and not isinstance(blk["rowStart"], G.Reduced)):
                        # The reference's setup skew ships the block in `both` mode and never waits for the row_idx
                        # receive (`else if`, SpmatLocal.hpp:248-255; SURVEY.md appendix B.2): whether its row_idx has
                        # landed when the block is dumped is a race in the reference itself (seen on a 128-core box).
                        # rowStart and col_idx (waited for, compared above) define the block; the delivered row_idx is
                        # their expansion, which is what this library must hold.
                        ref_ = np.repeat(np.arange(int(blk["rows"])), np.diff(np.asarray(blk["rowStart"])))
                    if not G.same(have, ref_):
                        if isinstance(ref_, G.Reduced):  # stored as a digest: no entries to show
                            raise AssertionError((r, key, b, f, f"shape {have.shape}", f"differs from {ref_}"))
                        where = np.flatnonzero(have != ref_)[:6] if have.shape == ref_.shape else []
                        raise AssertionError((r, key, b, f, f"shapes {have.shape} {ref_.shape}", f"first diffs at {list(where)}",
                                              f"have {have[where].tolist() if len(where) else ''}",
                                              f"want {ref_[where].tolist() if len(where) else ''}"))


def compare_ops(got, want, script, rtol=1e-11):
    worst = 0.0
    for r, (g, w) in enumerate(zip(got, want)):
        for key in ("S_rows", "S_cols", "ST_rows", "ST_cols"):
            assert G.same(g[key], w[key]), (r, key)  # order of the local value vectors: bit-exact
        for t, op in enumerate(script):
            for f in ("A", "B", "values"):
                a, b = g[f"op{t}_{f}"], w["ops"][t][f]
                assert a.shape == tuple(b.shape), (r, op, f, a.shape, b.shape)
                if a.size:
                    err = G.rel_err(a, b)
                    worst = max(worst, err)
                    assert err < rtol, (r, op, f, err)
    return worst
