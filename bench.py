#!/usr/bin/env python
"""bench.py -- FusedMM (SDDMM+SpMM) throughput of the B200-native HnH engine.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` (N>1 launched under
torch.distributed.run, one rank per GPU) prints ONE JSON line on rank 0.

* workload  : BASELINE.json configs[1] -- Erdos-Renyi N=2^20, 32 nnz/row, r=128, 1.5D
              dense-shift FusedMM: `fusedSpMM(A, B, S, result, Amat)` of
              Sparse15D_Dense_Shift, exactly what bench_erdos_renyi / benchmark_algorithm time
              (reference benchmark_dist.cpp:117-141; A=B=0.001, S=1.0, :102-106).  The C++ host
              classes of libhnh_b200.so run it; this file only drives them (ctypes) and measures.
* step      : one fusedSpMM call over the whole distributed matrix (strong scaling: the matrix
              is fixed, N GPUs share it).
* metric    : SDDMM+SpMM GFLOP/s with the reference's FLOP model 2*nnz*2*R per FusedMM
              (benchmark_dist.cpp:147).
* value     : inputs resident in HBM.   e2e: per-rank pinned host buffers, H2D/D2H inside the
              timed region.
* roofline  : local kernels' algorithmic bytes / their CUDA-event time vs MEASURED_PEAKS.json.
* cpu_baseline / --impl reference : the REFERENCE's own code (oracle/_ref: its sources compiled
              unmodified against MPI/MKL/Eigen/CombBLAS shims) on the host cores; falls back to
              the C port of its kernels (oracle/hnh_oracle.c) where oracle/_ref is not built.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SEED = 0xC0FFEE + 2  # config index 2 (SURVEY.md 8d)
FALLBACK_HBM_GBS = 6650.0
METRIC = "SDDMM+SpMM GFLOP/s (FusedMM, 4*nnz*R flop)"


# ------------------------------------------------------------------ helpers ---------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback"


def algorithmic_bytes(kind: str, nnz: int, m: int, r: int, beta0: bool = False) -> int:
    """SURVEY.md 8(d): fp64 w=8, int64 x=8, one local kernel call on a block with nnz nonzeros and
    m CSR rows.  beta0 variants do not read the old output / values."""
    w = x = 8
    if kind == "sddmm":
        return nnz * (r * w + x + (w if beta0 else 2 * w)) + (m + 1) * x + m * r * w
    if kind == "spmm":
        return nnz * (r * w + x + w) + (m + 1) * x + (1 if beta0 else 2) * m * r * w
    if kind == "fused":
        return nnz * (r * w + x + (w if beta0 else 2 * w)) + (m + 1) * x + (2 if beta0 else 3) * m * r * w
    raise ValueError(kind)


def fusedmm_bytes_per_rank(alg: str, nnz_rank: float, rows_stationary: int, steps: int, r: int) -> float:
    """Algorithmic HBM bytes one rank's local kernels move in one FusedMM (sum over ring steps).
    fusion 2: `steps` fused kernels on blocks of nnz_rank/steps nonzeros and rows_stationary rows;
    values written once, the accumulator written at step 0 and read+written afterwards.
    fusion 1: an SDDMM pass and an SpMM pass over the same blocks + the Hadamard / setCSRValues
    plumbing (3 + 2 value passes)."""
    w = x = 8
    m = rows_stationary
    if alg == "15d_fusion2":
        return nnz_rank * (r * w + x + w) + steps * ((m + 1) * x + m * r * w) + (2 * steps - 1) * m * r * w
    sddmm = nnz_rank * (r * w + x + w) + steps * ((m + 1) * x + m * r * w)
    spmm = nnz_rank * (r * w + x + w) + steps * ((m + 1) * x + 2 * m * r * w)
    return sddmm + spmm + 5 * w * nnz_rank


NVLINK_GBS_NOMINAL = 900.0  # NVLink 5, per GPU and direction (B200_PROFILING.md); MEASURED_PEAKS.json has no link figure


def nvlink_bytes_per_rank(alg: str, p: int, c: int, local_rows: int, r: int) -> float:
    """Bytes one rank RECEIVES over NVLink in one FusedMM of the 1.5D dense-shift algorithm (SURVEY.md 8(e)):
    every ring pass delivers p/c - 1 riding shards of local_rows x r doubles; replication (c > 1) adds the
    all-gather of the stationary operand (c - 1 shards in) and, for local kernel fusion, the reduce-scatter of
    the c x larger accumulator (c - 1 shard-sized partial sums in).  Fusion 2 makes one ring pass per FusedMM.
    Fusion 1 (replication reuse) makes two -- the SDDMM pass, and the SpMM pass in which the OUTPUT rides and
    therefore goes all the way round (p/c shifts) -- gathers once and never reduce-scatters."""
    shard = 8.0 * local_rows * r
    steps = p // c
    gather = (c - 1) * shard
    if alg == "15d_fusion2":
        return (steps - 1) * shard + 2 * gather
    return ((steps - 1) + (steps if steps > 1 else 0)) * shard + gather


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (NVML, 5 ms period)."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self.t = None
        self.err = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = f"nvml unavailable: {e}"
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.005)

    def stop(self):
        if self.t is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": [self.err or "no samples"]}
        self._stop.set()
        self.t.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.samples), "reasons": sorted(self.reasons)}


def workload_config(args):
    """What is computed -- identical in the native and the reference arm (the driver compares the two dicts).
    Everything that describes HOW a particular arm ran it (ranks, replication factor, transport, ...) is in `run`."""
    return {"workload": f"Erdos-Renyi N=2^{args.logM} nnz/row={args.nnz_per_row} r={args.R} FusedMM "
                        f"(Sparse15D_Dense_Shift::fusedSpMM, {args.alg}; A=B=0.001, S=1 as in benchmark_dist.cpp:102-106)",
            "logM": args.logM, "nnz_per_row": args.nnz_per_row, "R": args.R, "algorithm": args.alg,
            "seed": SEED, "index_type": "int64",
            "l2": "working set (dense factors + CSR, > 1 GiB per GPU) exceeds the 126 MB L2 and every step gathers "
                  "from a different block; no explicit flush between steps"}


# ------------------------------------------------------------------ CPU arm ---------------
class _quiet_stdout:
    """The reference prints progress with cout; keep bench.py's stdout to the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        self.null = os.open(os.devnull, os.O_WRONLY)
        os.dup2(self.null, 1)

    def __exit__(self, *a):
        os.dup2(self.saved, 1)
        os.close(self.null)
        os.close(self.saved)


def cpu_reference_fusedmm(args, warmup, steps, budget_s=45.0, want_pattern=False):
    """GFLOP/s of the reference's fusedSpMM on the host cores (rank 0 only).  Uses oracle/_ref (the reference's
    own code) when built, else the C port of its kernels.  The sample is the whole configured matrix; `steps` is
    reduced (never below 1) to keep warm-up + steps + set-up within `budget_s`, and only if even one step does not
    fit is the same configuration run at a smaller logM (same nnz/row and r: identical per-nonzero work).
    Returns (GFLOP/s, cores, kind, description, ms per step, steps timed, parity result or None)."""
    from oracle import ref
    cores = os.cpu_count() or 1
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        pass
    if ref.available():
        with _quiet_stdout():
            nnz0, s0 = ref.time_fused(args.alg, 1, 1, args.R, min(args.logM, 16), args.nnz_per_row, SEED, 1, 1, cores)
        gf0 = 4.0 * nnz0 * args.R / s0[-1] / 1e9
        setup_calls = 6  # construction (redistribution, sorts, two COO->CSR) costs about six call-equivalents
        logM = args.logM
        while True:
            call_s = 4.0 * (1 << logM) * args.nnz_per_row * args.R / (gf0 * 1e9)
            fit = int(budget_s / call_s) - setup_calls - warmup
            if fit >= 1 or logM <= 16:
                break
            logM -= 1
        steps = max(1, min(steps, fit))
        pattern_out = None
        with _quiet_stdout():
            if want_pattern and logM == args.logM and hasattr(ref.lib(), "ref_time_fused_check"):
                nnz, secs, pattern_out = ref.time_fused_check(args.alg, 1, args.R, logM, args.nnz_per_row, SEED, warmup,
                                                              steps, cores)
            else:
                nnz, secs = ref.time_fused(args.alg, 1, 1, args.R, logM, args.nnz_per_row, SEED, warmup, steps, cores)
        per = secs[warmup:]
        gf = 4.0 * nnz * args.R / per / 1e9
        desc = (f"the reference's own code (oracle/_ref: reference sources compiled unmodified; MKL/MPI/Eigen/"
                f"CombBLAS shimmed) {args.alg} p=1, {cores} OpenMP threads, Erdos-Renyi N=2^{logM} "
                f"nnz/row={args.nnz_per_row} r={args.R} (nnz={nnz}), {len(per)} fusedSpMM calls after {warmup} warm-up, "
                f"{np.mean(per)*1e3:.1f} ms each")
        return float(np.mean(gf)), cores, "reference", desc, float(np.mean(per)) * 1e3, len(per), pattern_out
    # fall-back: C port of the two local kernels on a row sample
    from distributed_sddmm_b200 import lib
    from oracle import hnh_oracle as orc
    L = lib()
    N, R = 1 << args.logM, args.R
    mrows = min(N, 1 << 17)
    cap = mrows * args.nnz_per_row
    r = np.empty(cap, np.uint64); c = np.empty(cap, np.uint64); v = np.empty(cap, np.float64)
    n = L.hnh_er_generate_host(args.logM, args.nnz_per_row, SEED, 0, mrows, r.ctypes.data, c.ctypes.data, v.ctypes.data, cap)
    csr = orc.coo_to_csr(mrows, N, r[:n], c[:n], v[:n])
    A = np.full((mrows, R), 0.001); B = np.full((N, R), 0.001)
    vals = np.zeros(n); out = np.zeros((mrows, R))
    ts = []
    for i in range(warmup + steps):
        vals[:] = 0; out[:] = 0
        t0 = time.perf_counter()
        orc.fused_block(csr.rowStart, csr.row_idx, csr.col_idx, vals, A, B, out)
        ts.append(time.perf_counter() - t0)
    per = np.array(ts[warmup:])
    gf = 4.0 * n * R / per / 1e9
    desc = (f"C port of the reference kernels (oracle/hnh_oracle.c; oracle/_ref not built), first {mrows} of {N} rows "
            f"against the full B, {orc.num_threads()} threads")
    return float(np.mean(gf)), orc.num_threads(), "port", desc, float(np.mean(per)) * 1e3, len(per), None


def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    warmup = min(args.warmup, 1)
    # every step is a full-size fusedSpMM of the reference (about 4 s on a 128-thread host): K of them when the run
    # stays within a few minutes, fewer otherwise -- `steps` in the line is what was timed
    g, cores, kind, desc, ms, steps_run, _ = cpu_reference_fusedmm(args, warmup, args.steps, budget_s=180.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": g, "unit": "GFLOP/s", "n_gpus": args.gpus, "steps": steps_run,
        "steps_requested": args.steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(args),
        "run": {"where": "cpu", "p": 1, "c": 1},
        "cpu_baseline": {"value": g, "unit": "GFLOP/s", "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": g, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------ parity leg ------------
PARITY_RTOL = 1e-5  # BASELINE.json north_star: fp64 values within 1e-5 relative


def pattern_local(subs, shape, salt, nrows_global):
    """This rank's shard of the global pattern operand: the submatrix blocks (top, left, rows, cols) stacked in local
    storage order (DenseSubmatrix descriptors, distributed_sparse.h:322-346); rows beyond the matrix are zero."""
    from oracle import ref
    flat = np.zeros(shape[0] * shape[1])
    at = 0
    for top, left, nr, nc in subs:
        blk = ref.pattern(int(nr), int(nc), salt, row0=int(top), col0=int(left))
        blk[max(0, nrows_global - int(top)):] = 0.0
        flat[at:at + nr * nc] = blk.reshape(-1)
        at += nr * nc
    return flat.reshape(shape)


def sample_parity(logM, npr, R, alg, A, B, Sv, res, rank, world, shifts=False, rows_per_block=2048):
    """FusedMM (mode A) of `alg` on the pattern operands; `rows_per_block` consecutive rows of every local submatrix
    block are compared with the C port of the reference kernels (oracle/hnh_oracle.c: SDDMM over the full width, then
    SpMM) on the same tuples -- for any layout, R-split ones included.  Returns (this rank's output, stats dict)."""
    import torch
    import torch.distributed as dist
    from distributed_sddmm_b200 import lib
    from oracle import hnh_oracle as orc
    from oracle import ref
    L = lib()
    N = 1 << logM
    subsA, subsB = alg.submatrices("A"), alg.submatrices("B")
    shapeA, shapeB = A.shape, B.shape
    A.from_host(pattern_local(subsA, shapeA, 1, N))
    B.from_host(pattern_local(subsB, shapeB, 2, N))
    if shifts:
        alg.initial_shift(A, B, "sddmmA")
    alg.fusedSpMM(A, B, Sv, res, "A")
    if shifts:
        alg.de_shift(A, B, "sddmmA")
    got = A.to_host()
    err, rows_checked, nnz_checked, local_error = 0.0, 0, 0, None
    try:  # a failure of the checker on one rank must not leave the others waiting in the reductions below
        flat, at = got.reshape(-1), 0
        for top, left, nr, nc in subsA:
            top, left, nr, nc = int(top), int(left), int(nr), int(nc)
            blk = flat[at:at + nr * nc].reshape(nr, nc)
            at += nr * nc
            live = max(0, min(nr, N - top))
            n_s = min(live, rows_per_block)
            if n_s == 0:
                continue
            lo = top + (live - n_s) // 3
            cap = n_s * npr
            r_, c_, v_ = np.empty(cap, np.uint64), np.empty(cap, np.uint64), np.empty(cap, np.float64)
            n = L.hnh_er_generate_host(logM, npr, SEED, lo, lo + n_s, r_.ctypes.data, c_.ctypes.data, v_.ctypes.data, cap)
            r_, c_, v_ = r_[:n], c_[:n], v_[:n]
            ucols, inv = np.unique(c_, return_inverse=True)
            csr = orc.coo_to_csr(n_s, len(ucols), r_ - np.uint64(lo), inv.astype(np.uint64), v_)
            want = np.zeros((n_s, R))
            orc.fused_block(csr.rowStart, csr.row_idx, csr.col_idx, np.zeros(csr.nnz), ref.pattern(n_s, R, 1, row0=lo),
                            ref.pattern_rows(ucols, R, 2), want)
            want = want[:, left:left + nc]
            have = blk[lo - top:lo - top + n_s]
            err = max(err, float(np.abs(have - want).max() / max(float(np.abs(want).max()), 1e-300)))
            rows_checked += n_s
            nnz_checked += int(n)

    except Exception as e:  # noqa: BLE001
        local_error, err = f"{type(e).__name__}: {e}", float("inf")
    stats = torch.tensor([err, float(rows_checked), float(nnz_checked)], dtype=torch.float64)
    if world > 1:
        worst, tot = stats.clone(), stats.clone()
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        err, rows_checked, nnz_checked = float(worst[0]), int(tot[1]), int(tot[2])
    rec = {"checker": "oracle/hnh_oracle.c (C port of sparse_kernels.cpp:44-55 + CSR SpMM), same tuples",
           "rows": rows_checked, "nnz": nnz_checked, "max_rel_err": err}
    if local_error:
        rec["error_on_this_rank"] = local_error
    return got, rec


_progress = lambda what: None  # noqa: E731  (set by run_native)


def parity_check(args, alg, A, B, Sv, res, rank, world, pattern_ref, want_full):
    """One fusedSpMM on position-dependent operands (oracle/ref.py::pattern, exactly representable) at the FULL
    benchmark size, on the data plane that was just timed (same algorithm object, same rings), checked two ways:
      sample: consecutive output rows of every rank against the C port of the reference kernels
              (oracle/hnh_oracle.c, pinned bit-exact to the reference's loop) on the same tuples;
      full  : every output row against one fusedSpMM of the reference's own code (oracle/_ref, p = 1) -- computed on
              rank 0 and handed to the ranks over gloo.
    Returns the `parity_check` object of the JSON line; never raises (a failure is reported, not hidden)."""
    import torch
    import torch.distributed as dist
    from oracle import ref
    out = {"tolerance": PARITY_RTOL, "inputs": "A = pattern(1), B = pattern(2) (oracle/ref.py), S pattern all ones"}
    try:
        N, R = 1 << args.logM, args.R
        topA, leftA, nrA, ncA = (int(x) for x in alg.submatrices("A")[0])
        _progress("parity: FusedMM on the pattern operands + row sample against the C port")
        got, out["sample"] = sample_parity(args.logM, args.nnz_per_row, R, alg, A, B, Sv, res, rank, world)
        A.fill(0.001)
        B.fill(0.001)
        live = max(0, min(nrA, N - topA))
        rows_s = out["sample"]["rows"]

        # ---- full: the reference's own fusedSpMM ----
        if want_full:
            # rank 0 computes the reference first; only then do the ranks agree (one broadcast) on whether there is
            # anything to compare with -- a failure of the CPU run cannot strand the others in a collective
            ref_error = None
            if rank == 0 and pattern_ref is None:
                _progress("parity: the reference's fusedSpMM on the host cores (rank 0)")
                try:
                    if not (ref.available() and hasattr(ref.lib(), "ref_time_fused_check")):
                        raise RuntimeError("oracle/_ref is not built")
                    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
                    with _quiet_stdout():
                        _, _, pattern_ref = ref.time_fused_check(args.alg, 1, R, args.logM, args.nnz_per_row, SEED, 0, 0, cores)
                except Exception as e:  # noqa: BLE001
                    ref_error, pattern_ref = f"{type(e).__name__}: {e}", None
            flag = torch.tensor([1 if (rank == 0 and pattern_ref is not None) else 0])
            if world > 1:
                dist.broadcast(flag, src=0)
            if int(flag[0]):
                _progress("parity: handing the reference rows to the ranks")
                if world > 1:  # hand every rank its rows (gloo send/recv, 64 MiB pieces)
                    where = [None] * world
                    dist.all_gather_object(where, (int(topA), int(live)))
                    piece = max(1, (64 << 20) // (8 * R))
                    if rank == 0:
                        mine = pattern_ref[topA:topA + live]
                        for dst_rank in range(1, world):
                            top_r, live_r = where[dst_rank]
                            for off in range(0, live_r, piece):
                                m = min(piece, live_r - off)
                                dist.send(torch.from_numpy(np.ascontiguousarray(pattern_ref[top_r + off:top_r + off + m])),
                                          dst=dst_rank)
                    else:
                        mine = np.empty((live, R))
                        for off in range(0, live, piece):
                            m = min(piece, live - off)
                            buf = torch.empty((m, R), dtype=torch.float64)
                            dist.recv(buf, src=0)
                            mine[off:off + m] = buf.numpy()
                else:
                    mine = pattern_ref[topA:topA + live]
                _progress("parity: comparing")
                loc = torch.tensor([float(np.abs(got[:live] - mine).max()), float(np.abs(mine).max())], dtype=torch.float64)
                sq = torch.tensor([float(np.sum(got[:live] ** 2)), float(np.sum(mine ** 2))], dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(loc, op=dist.ReduceOp.MAX)
                    dist.all_reduce(sq, op=dist.ReduceOp.SUM)
                out["full"] = {"checker": "oracle/_ref (the reference's own sources, p = 1): one fusedSpMM on the same tuples "
                                          "and operands", "rows": N, "max_rel_err": float(loc[0] / max(float(loc[1]), 1e-300)),
                               "fingerprint_squared_norm": {"native": float(sq[0]), "reference": float(sq[1])}}
            else:
                out["full"] = None
                if ref_error:
                    out["full_skipped"] = ref_error
        errs = [out["sample"]["max_rel_err"]] + ([out["full"]["max_rel_err"]] if out.get("full") else [])
        out["max_rel_err"] = max(errs)
        out["n"] = (N if out.get("full") else rows_s)
        out["pass"] = bool(np.isfinite(out["max_rel_err"]) and out["max_rel_err"] <= PARITY_RTOL)
    except Exception as e:  # noqa: BLE001
        import traceback
        out["error"] = f"{type(e).__name__}: {e}"
        out["trace"] = traceback.format_exc()[-600:]
        out["pass"] = False
    return out


DUMP_SEED = 20261017
DUMP_BYTES = 64_000_000   # every file of every rank together, headers included


def dump_outputs(out_dir, A, values, rank, world):
    """What the last timed fusedSpMM returned to this rank's caller -- A (the FusedMM output, mode A) and the SDDMM
    values -- as float64 .npy files under `out_dir`.  Each rank gets an equal share of DUMP_BYTES, two thirds for A
    and one third for the values; an output larger than its share is cut to a fixed seeded sample of rows / values
    (sorted indices, identical for identical arguments), so two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    share = DUMP_BYTES // world - 2 * 128  # an .npy header is 128 bytes
    row_bytes = 8 * max(1, A.shape[1])
    rows, nvals = min(A.shape[0], (2 * share // 3) // row_bytes), min(values.size, (share // 3) // 8)
    rng = np.random.default_rng(DUMP_SEED)
    if rows < A.shape[0]:
        A = A[np.sort(rng.choice(A.shape[0], rows, replace=False))]
    if nvals < values.size:
        values = values[np.sort(rng.choice(values.size, nvals, replace=False))]
    np.save(os.path.join(out_dir, f"fused_output_A{suffix}.npy"), np.ascontiguousarray(A, np.float64))
    np.save(os.path.join(out_dir, f"sddmm_values{suffix}.npy"), np.ascontiguousarray(values, np.float64))


# ------------------------------------------------------------------ GPU arm ---------------
def run_native(args):
    import torch
    from distributed_sddmm_b200 import driver as D
    from distributed_sddmm_b200 import lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU arm)")
    # --share-gpu (testing aid, never a measurement): all ranks on cuda:0 over the gloo-backed External transport, to
    # exercise the multi-rank control flow of this file on a one-GPU box
    torch.cuda.set_device(0 if args.share_gpu else local_rank)
    L = lib()
    rank, world = D.world_init("gloo" if (args.share_gpu and world > 1) else None)
    import torch.distributed as dist
    t_start = time.perf_counter()

    def progress(what):
        """Phase marker on stderr (rank 0): a hung or slow phase of a remote run can be told from its log."""
        if rank == 0:
            print(f"[bench +{time.perf_counter() - t_start:7.1f} s] {what}", file=sys.stderr, flush=True)

    global _progress
    _progress = progress

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sync_barrier():
        L.hnhd_device_synchronize()
        if world > 1:
            L.hnhd_barrier()

    N, R, c = 1 << args.logM, args.R, args.c
    progress("generating the matrix")
    S = D.SpmatLocal.load_er(args.logM, args.nnz_per_row, SEED)
    nnz = S.info()["dist_nnz"]
    progress("building the algorithm object (redistribution, CSR blocks)")
    alg = D.Algorithm(args.alg, S, R, c)
    info = alg.info()
    A, B = alg.like_A_matrix(0.001), alg.like_B_matrix(0.001)
    Sv, res = alg.like_S_values(1.0), alg.like_S_values(0.0)
    steps_ring = world // c

    def step():
        alg.fusedSpMM(A, B, Sv, res, "A")

    progress(f"warm-up ({args.warmup}) and timed loop ({args.steps})")
    for _ in range(args.warmup):
        step()
    sync_barrier()
    alg.reset_timers()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.hnh_launch_count()
    sync_barrier()
    D.timer_start()
    for _ in range(args.steps):
        step()
    ms_total = D.timer_stop()
    sync_barrier()
    launches = L.hnh_launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs:  # before the legs below overwrite A
        dump_outputs(args.dump_outputs, A.to_host(), res.to_host(), rank, world)
    ms = max_over_ranks(ms_total) / args.steps
    flops = 4.0 * nnz * R
    gflops = flops / (ms * 1e-3) / 1e9
    perf = alg.perf()  # collective: averages over ranks

    # ---- roofline of the local kernels (dominant: the fused / SpMM kernel) ----
    comp_ms = perf["Computation Time"] * 1e3 / args.steps
    nnz_rank = float(np.mean(info["nnz_procs"]))
    rows_stationary = alg.dims.localArows * c
    bytes_rank = fusedmm_bytes_per_rank(args.alg, nnz_rank, rows_stationary, steps_ring, R)
    peak, peak_kind = measured_peaks()
    achieved = bytes_rank / (comp_ms * 1e-3) / 1e9 if comp_ms > 0 else 0.0
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_kind": f"of {peak_kind}",
                "kernel": ("fused_row_kernel" if args.alg == "15d_fusion2" else "sddmm_row_kernel + spmm_row_kernel") +
                          f"<{R}>, {steps_ring} launch(es) per step per GPU",
                "kernel_ms_per_step": comp_ms, "algorithmic_bytes_per_step_per_gpu": bytes_rank}
    # The per-block launches of a multi-rank step re-read the row-side factor and read + write the accumulator once
    # per ring step; `frac` counts those bytes (they are what the launched kernels must move).  The share of ONE launch
    # over all of the rank's nonzeros -- what a perfectly fused step would move -- is reported beside it.
    minimal = nnz_rank * (R * 8 + 8 + 8) + (rows_stationary + 1) * 8 + 2 * rows_stationary * R * 8
    roofline["minimal_bytes_per_step_per_gpu"] = minimal
    roofline["frac_on_minimal_bytes"] = (minimal / (comp_ms * 1e-3) / 1e9 / peak) if comp_ms > 0 else 0.0
    # DRAM bytes per launch of this kernel from the committed ncu capture of the same command (a profiler cannot run
    # inside the timed region); only for the exact configuration that was captured
    prof = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(prof) and world == 1 and (args.logM, args.nnz_per_row) == (20, 32):
        try:
            tj = json.load(open(prof))
            roofline["traffic"] = tj.get(f"{'fused' if args.alg == '15d_fusion2' else 'spmm'}_{R}")
            roofline["traffic_source"] = "profiles/r02_traffic.json (ncu --set full, same kernel and config)"
        except Exception:  # noqa: BLE001
            pass
    shift_ms = perf.get("Cyclic Shift Time", 0.0) * 1e3 / args.steps
    repl_ms = perf.get("Replication Time", 0.0) * 1e3 / args.steps

    # ---- the other fusion strategy, for the record (not the headline) ----
    other = None
    if world == 1 and not args.no_other:
        oname = "15d_fusion1" if args.alg == "15d_fusion2" else "15d_fusion2"
        oalg = D.Algorithm(oname, S, R, c)
        oSv, ores = oalg.like_S_values(1.0), oalg.like_S_values(0.0)
        for _ in range(2):
            oalg.fusedSpMM(A, B, oSv, ores, "A")
        sync_barrier()
        D.timer_start()
        for _ in range(max(3, args.steps // 2)):
            oalg.fusedSpMM(A, B, oSv, ores, "A")
        oms = D.timer_stop() / max(3, args.steps // 2)
        other = {oname: {"ms_per_step": oms, "gflops": flops / (oms * 1e-3) / 1e9}}
        del oalg, oSv, ores

    progress("timed loop done")
    # ---- the north-star transport, for the record: the same ring as grouped NCCL send/recv (HNH_RING=nccl) ----
    if world > 1 and not args.no_other:
        try:
            os.environ["HNH_RING"] = "nccl"
            nalg = D.Algorithm(args.alg, S, R, c)
            nSv, nres = nalg.like_S_values(1.0), nalg.like_S_values(0.0)
            for _ in range(2):
                nalg.fusedSpMM(A, B, nSv, nres, "A")
            sync_barrier()
            D.timer_start()
            for _ in range(5):
                nalg.fusedSpMM(A, B, nSv, nres, "A")
            nms = max_over_ranks(D.timer_stop()) / 5
            sync_barrier()
            other = dict(other or {}, nccl_send_recv_ring={"ms_per_step": nms, "gflops": flops / (nms * 1e-3) / 1e9,
                                                          "ring": nalg.info().get("ring")})
            del nalg, nSv, nres
        finally:
            os.environ.pop("HNH_RING", None)

    # ---- e2e: per-rank pinned HOST buffers in, result out, copies inside the timed region ----
    progress("e2e leg (host operands)")
    shapeA, shapeB = A.shape, B.shape
    hA = torch.full(shapeA, 0.001, dtype=torch.float64).pin_memory()
    hB = torch.full(shapeB, 0.001, dtype=torch.float64).pin_memory()
    hO = torch.empty(shapeA, dtype=torch.float64).pin_memory()
    e2e_steps = max(2, min(args.steps, 5))

    def e2e_step():
        if not args.e2e_plain:
            alg.fusedSpMM_host(A, B, Sv, res, hA, hB, hO, "A")
            return
        D.check(L.hnhd_dense_from_host(A.h, hA.data_ptr()), "from_host")
        D.check(L.hnhd_dense_from_host(B.h, hB.data_ptr()), "from_host")
        alg.fusedSpMM(A, B, Sv, res, "A")
        D.check(L.hnhd_dense_to_host(A.h, hO.data_ptr()), "to_host")

    e2e_step()
    sync_barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    sync_barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) / e2e_steps * 1e3)
    h2d = (shapeA[0] * shapeA[1] + shapeB[0] * shapeB[1]) * 8 * world
    d2h = shapeA[0] * shapeA[1] * 8 * world
    e2e = {"value": flops / (e2e_ms * 1e-3) / 1e9, "unit": "GFLOP/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "api": ("per rank: Distributed_Sparse::fusedSpMM_host (pinned host A, B in; result out; uploads, kernels and "
                   "download pipelined)" if not args.e2e_plain else
                   "per rank: DenseMatrix::copy_from_host(A), (B) from pinned memory; fusedSpMM; copy_to_host(A)")}
    del hA, hB, hO

    # ---- CPU baseline on the host cores (rank 0, N = 1 only; bounded sample) ----
    cpu = None
    pattern_ref = None
    want_full = args.parity == "full"
    progress("cpu baseline / parity leg")
    if world == 1 and not args.no_cpu_baseline:
        g, cores, kind, desc, _, _, pattern_ref = cpu_reference_fusedmm(args, 1, 3, want_pattern=want_full)
        cpu = {"value": g, "unit": "GFLOP/s", "cores": cores, "kind": kind, "sample": desc}

    # ---- parity leg (outside every timed region) ----
    parity = None
    if args.parity != "off":
        parity = parity_check(args, alg, A, B, Sv, res, rank, world, pattern_ref, want_full)

    nvlink = None
    if world > 1:
        try:  # explanatory only: never let it cost the line
            nb = nvlink_bytes_per_rank(args.alg, world, c, alg.dims.localBrows, R)
            nvlink = {"bytes_in_per_gpu_per_step": nb, "peak_gbs": NVLINK_GBS_NOMINAL, "peak_kind": "nominal",
                      "bound_ms": nb / (NVLINK_GBS_NOMINAL * 1e9) * 1e3, "achieved_gbs": nb / (ms * 1e-3) / 1e9,
                      # every pushed shard is read once here and written once at the neighbour by the copy engines
                      "copy_engine_hbm_bytes_per_gpu_per_step": 2.0 * nb}
        except Exception:  # noqa: BLE001
            nvlink = None

    ring_info = alg.info().get("ring")  # collective (per-rank nnz are gathered): every rank must make this call
    progress("done")
    if rank == 0:
        line = {
            "metric": METRIC, "value": gflops, "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "run": {"where": "cuda", "p": world, "c": c, "nnz": nnz, "ring_steps": steps_ring,
                    "local_rows": alg.dims.localArows, "transport": info.get("transport"),
                    "ring": ring_info,
                    "collectives": ("NCCL all-gather / reduce-scatter over row_world" if c > 1 else "none")},
            "hbm_gbs_achieved_per_gpu": bytes_rank / (ms * 1e-3) / 1e9,
            "roofline": roofline,
            "phase_ms_per_step": {"computation": comp_ms, "cyclic_shift": shift_ms, "replication": repl_ms},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "parity_check": parity,
        }
        if other:
            line["other"] = other
        if nvlink:
            line["nvlink"] = nvlink
        print(json.dumps(line))
    del alg, S
    D.world_finalize()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--logM", type=int, default=20)
    ap.add_argument("--nnz-per-row", type=int, default=32)
    ap.add_argument("--R", type=int, default=128)
    ap.add_argument("--c", type=int, default=0, help="replication factor (0 = the tuned default for this GPU count)")
    ap.add_argument("--alg", default="15d_fusion2", choices=["15d_fusion1", "15d_fusion2"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other", action="store_true")
    ap.add_argument("--e2e-plain", action="store_true",
                    help="e2e leg as copy_from_host(A), (B); fusedSpMM; copy_to_host instead of the default "
                         "Distributed_Sparse::fusedSpMM_host (upload / kernels / download pipelined)")
    ap.add_argument("--share-gpu", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--parity", default="full", choices=["full", "sample", "off"],
                    help="correctness leg after the timed loops (never timed): 'sample' = a row sample per rank against the "
                         "C port of the reference kernels; 'full' = that plus every output row against one fusedSpMM of "
                         "oracle/_ref (the reference's own code) on the same tuples and operands")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="native arm: write what the last timed step computed (A and the SDDMM values, or a fixed "
                         "sample of them) as DIR/<name>.npy, float64, at most 64 MB over all ranks")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes what the native (GPU) arm computed; the reference arm has nothing to dump")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.c <= 0:
        args.c = default_c(args.alg, world)
    if args.warmup < 3 and args.impl == "native":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_native(args)


def default_c(alg: str, world: int) -> int:
    """Replication factor per GPU count (measured sweep, profiles/r01_scaling.md)."""
    table = {1: 1, 2: 1, 4: 1, 8: 1}
    return table.get(world, 1)


if __name__ == "__main__":
    sys.exit(main())
