"""Thin Python front end of the C++ host classes (through include/hnh_b200_driver.h).

Mirrors the reference's usage pattern (bench_erdos_renyi.cpp / benchmark_dist.cpp / scratch.cpp):

    world_init()                       # MPI_Init
    S = SpmatLocal.load_er(logM, nnz)  # SpmatLocal S; S.loadTuples(false, logM, nnz, "")
    d_ops = Algorithm("15d_fusion2", S, R, c)   # new Sparse15D_Dense_Shift(&S, R, c, 2, &kernel)
    A, B = d_ops.like_A_matrix(0.001), d_ops.like_B_matrix(0.001)
    Sv, res = d_ops.like_S_values(1.0), d_ops.like_S_values(0.0)
    d_ops.fusedSpMM(A, B, Sv, res, "A")

Everything heavy happens in libhnh_b200.so; numpy arrays cross the boundary only in tests.
"""
from __future__ import annotations

import ctypes as C
import json
import os

import numpy as np

from ._lib import AlgDims, check, lib

OP = {"sddmmA": 0, "sddmmB": 1, "spmmA": 2, "spmmB": 3, "fusedA": 4, "fusedB": 5, "initial_shift": 6, "de_shift": 7}
KMODE = {"sddmmA": 0, "spmmA": 1, "spmmB": 2, "sddmmB": 3}

_transport_keepalive = None


def world_init(transport: str | None = None):
    """MPI_Init of this library.  transport: None -> from the environment (WORLD_SIZE == 1: self;
    otherwise NCCL on GPU boxes, the gloo-backed External transport on CPU-only boxes)."""
    global _transport_keepalive
    L = lib()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if transport is None:
        if world == 1:
            transport = "self"
        else:
            import torch
            transport = "nccl" if torch.cuda.is_available() else "gloo"
    if transport == "self":
        check(L.hnhd_init_self(), "hnhd_init_self")
    elif transport == "nccl":
        import torch
        import torch.distributed as dist
        if not dist.is_initialized():
            dist.init_process_group("gloo")
        uid = C.create_string_buffer(128)
        if rank == 0:
            check(L.hnhd_nccl_unique_id(uid), "hnhd_nccl_unique_id")
        t = torch.frombuffer(bytearray(uid.raw), dtype=torch.uint8).clone()
        dist.broadcast(t, src=0)
        check(L.hnhd_init_nccl(rank, world, bytes(t.numpy().tobytes())), "hnhd_init_nccl")
    elif transport == "gloo":
        from .gloo_transport import GlooTransport
        _transport_keepalive = GlooTransport()
        check(L.hnhd_init_external(rank, world, C.byref(_transport_keepalive.table)), "hnhd_init_external")
    else:
        raise ValueError(transport)
    return L.hnhd_world_rank(), L.hnhd_world_size()


def world_finalize(destroy_process_group: bool = True):
    """MPI_Finalize of this library; also tears the torch.distributed group down cleanly."""
    global _transport_keepalive
    check(lib().hnhd_finalize(), "hnhd_finalize")
    _transport_keepalive = None
    if destroy_process_group:
        try:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                dist.barrier()
                dist.destroy_process_group()
        except Exception:  # noqa: BLE001
            pass


class SpmatLocal:
    def __init__(self, handle):
        self.h = handle

    @classmethod
    def load_er(cls, logM: int, nnz_per_row: int, seed: int = 0xC0FFEE):
        h = C.c_void_p()
        check(lib().hnhd_spmat_load_er(logM, nnz_per_row, seed, C.byref(h)), "hnhd_spmat_load_er")
        return cls(h)

    @classmethod
    def load_file(cls, filename: str):
        h = C.c_void_p()
        check(lib().hnhd_spmat_load_file(filename.encode(), C.byref(h)), "hnhd_spmat_load_file")
        return cls(h)

    @classmethod
    def from_tuples(cls, M, N, rows, cols, vals):
        rows = np.ascontiguousarray(rows, np.uint64)
        cols = np.ascontiguousarray(cols, np.uint64)
        vals = np.ascontiguousarray(vals, np.float64)
        h = C.c_void_p()
        check(lib().hnhd_spmat_from_tuples(M, N, rows.ctypes.data, cols.ctypes.data, vals.ctypes.data, len(rows),
                                           C.byref(h)), "hnhd_spmat_from_tuples")
        return cls(h)

    def info(self):
        M, N, nnz, loc = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_int64()
        check(lib().hnhd_spmat_info(self.h, C.byref(M), C.byref(N), C.byref(nnz), C.byref(loc)), "hnhd_spmat_info")
        return {"M": M.value, "N": N.value, "dist_nnz": nnz.value, "local_tuples": loc.value}

    def tuples(self):
        n = self.info()["local_tuples"]
        r, c, v = np.zeros(n, np.uint64), np.zeros(n, np.uint64), np.zeros(n, np.float64)
        check(lib().hnhd_spmat_tuples(self.h, r.ctypes.data, c.ctypes.data, v.ctypes.data, n), "hnhd_spmat_tuples")
        return r, c, v

    def __del__(self):
        try:
            lib().hnhd_spmat_destroy(self.h)
        except Exception:
            pass


class Dense:
    def __init__(self, handle):
        self.h = handle

    @property
    def shape(self):
        r, c = C.c_int64(), C.c_int64()
        lib().hnhd_dense_shape(self.h, C.byref(r), C.byref(c))
        return r.value, c.value

    def fill(self, v):
        check(lib().hnhd_dense_fill(self.h, v), "hnhd_dense_fill")

    def from_host(self, arr):
        arr = np.ascontiguousarray(arr, np.float64)
        assert arr.shape == self.shape, (arr.shape, self.shape)
        check(lib().hnhd_dense_from_host(self.h, arr.ctypes.data), "hnhd_dense_from_host")

    def to_host(self):
        out = np.empty(self.shape, np.float64)
        check(lib().hnhd_dense_to_host(self.h, out.ctypes.data), "hnhd_dense_to_host")
        return out

    def data_ptr(self):
        return lib().hnhd_dense_data(self.h)

    def __del__(self):
        try:
            lib().hnhd_dense_destroy(self.h)
        except Exception:
            pass


class Vec:
    def __init__(self, handle):
        self.h = handle

    def __len__(self):
        return int(lib().hnhd_vec_size(self.h))

    def fill(self, v):
        check(lib().hnhd_vec_fill(self.h, v), "hnhd_vec_fill")

    def from_host(self, arr):
        arr = np.ascontiguousarray(arr, np.float64)
        assert len(arr) == len(self)
        check(lib().hnhd_vec_from_host(self.h, arr.ctypes.data), "hnhd_vec_from_host")

    def to_host(self):
        out = np.empty(len(self), np.float64)
        check(lib().hnhd_vec_to_host(self.h, out.ctypes.data), "hnhd_vec_to_host")
        return out

    def __del__(self):
        try:
            lib().hnhd_vec_destroy(self.h)
        except Exception:
            pass


class Algorithm:
    """A Distributed_Sparse subclass instance with the library's StandardKernel plugged in."""

    def __init__(self, name: str, S: SpmatLocal, R: int, c: int):
        self.name = name
        self.h = C.c_void_p()
        check(lib().hnhd_alg_create(name.encode(), S.h, R, c, C.byref(self.h)), f"hnhd_alg_create({name})")
        d = AlgDims()
        check(lib().hnhd_alg_dims(self.h, C.byref(d)), "hnhd_alg_dims")
        self.dims = d

    def submatrices(self, which):
        n = self.dims.n_a_submatrices if which == "A" else self.dims.n_b_submatrices
        out = np.zeros(4 * n, np.int32)
        lib().hnhd_alg_submatrices(self.h, 0 if which == "A" else 1, out.ctypes.data, 4 * n)
        return out.reshape(n, 4)

    def _mk_dense(self, which, v):
        h = C.c_void_p()
        check(lib().hnhd_dense_like(self.h, which, v, C.byref(h)), "hnhd_dense_like")
        return Dense(h)

    def like_A_matrix(self, v=0.0):
        return self._mk_dense(0, v)

    def like_B_matrix(self, v=0.0):
        return self._mk_dense(1, v)

    def _mk_vec(self, which, v):
        h = C.c_void_p()
        check(lib().hnhd_vec_like(self.h, which, v, C.byref(h)), "hnhd_vec_like")
        return Vec(h)

    def like_S_values(self, v=0.0):
        return self._mk_vec(0, v)

    def like_ST_values(self, v=0.0):
        return self._mk_vec(1, v)

    def dummyInitialize(self, m: Dense, which: str):
        check(lib().hnhd_dense_dummy_initialize(self.h, m.h, 0 if which == "A" else 1), "dummyInitialize")

    def _op(self, op, A, B, S=None, R=None, aux=0):
        check(lib().hnhd_alg_op(self.h, OP[op], A.h if A else None, B.h if B else None, S.h if S else None,
                                R.h if R else None, aux), op)

    def sddmmA(self, A, B, S, R):
        self._op("sddmmA", A, B, S, R)

    def sddmmB(self, A, B, S, R):
        self._op("sddmmB", A, B, S, R)

    def spmmA(self, A, B, S):
        self._op("spmmA", A, B, S)

    def spmmB(self, A, B, S):
        self._op("spmmB", A, B, S)

    def fusedSpMM(self, A, B, S, R, mode="A"):
        self._op("fusedA" if mode == "A" else "fusedB", A, B, S, R)

    def fusedSpMM_host(self, A, B, S, R, hostA, hostB, hostOut, mode="A", chunk_rows=0):
        """fusedSpMM with host operands (torch CPU tensors or numpy arrays, float64, contiguous; pinned memory
        makes the copies asynchronous).  chunk_rows: 0 default pipeline, < 0 no pipeline."""
        ptr = lambda t: t.data_ptr() if hasattr(t, "data_ptr") else t.ctypes.data  # noqa: E731
        check(lib().hnhd_alg_fused_host(self.h, A.h, B.h, S.h, R.h, ptr(hostA), ptr(hostB), ptr(hostOut),
                                        0 if mode == "A" else 1, chunk_rows), "hnhd_alg_fused_host")

    def initial_shift(self, A, B, mode):
        self._op("initial_shift", A, B, aux=KMODE[mode])

    def de_shift(self, A, B, mode):
        self._op("de_shift", A, B, aux=KMODE[mode])

    def info(self):
        buf = C.create_string_buffer(1 << 16)
        n = lib().hnhd_alg_info_json(self.h, buf, len(buf))
        if n < 0:
            check(n, "hnhd_alg_info_json")
        return json.loads(buf.value.decode())

    def perf(self):
        buf = C.create_string_buffer(1 << 16)
        n = lib().hnhd_alg_perf_json(self.h, buf, len(buf))
        if n < 0:
            check(n, "hnhd_alg_perf_json")
        return json.loads(buf.value.decode())

    def reset_timers(self):
        check(lib().hnhd_alg_reset_timers(self.h), "reset_timers")

    def als_residuals(self, steps=1):
        """(residual before, residual after) `steps` rounds of ALS-CG on an artificial ground truth."""
        out = (C.c_double * 2)()
        check(lib().hnhd_als_residuals(self.h, steps, out), "hnhd_als_residuals")
        return out[0], out[1]

    def blocks(self, which="S"):
        """Host copies of the local CSR blocks: list of None | dict(rows, cols, transpose, rowStart, col_idx,
        row_idx, values)."""
        w = 0 if which == "S" else 1
        out = []
        L = lib()
        for b in range(L.hnhd_alg_block_count(self.h, w)):
            rows, cols, nnz = C.c_int64(), C.c_int64(), C.c_int64()
            tr, null = C.c_int(), C.c_int()
            check(L.hnhd_alg_block_meta(self.h, w, b, C.byref(rows), C.byref(cols), C.byref(nnz), C.byref(tr),
                                        C.byref(null)), "block_meta")
            if null.value:
                out.append(None)
                continue
            rs = np.zeros(rows.value + 1, np.int64)
            ci, ri = np.zeros(nnz.value, np.int64), np.zeros(nnz.value, np.int64)
            v = np.zeros(nnz.value, np.float64)
            check(L.hnhd_alg_block_arrays(self.h, w, b, rs.ctypes.data, ci.ctypes.data, ri.ctypes.data, v.ctypes.data),
                  "block_arrays")
            out.append(dict(rows=rows.value, cols=cols.value, transpose=bool(tr.value), rowStart=rs, col_idx=ci,
                            row_idx=ri, values=v))
        return out

    def __del__(self):
        try:
            lib().hnhd_alg_destroy(self.h)
        except Exception:
            pass


def setup_times(reset: bool = False) -> dict:
    """Wall-clock seconds of this process' setup phases so far (hnh::SetupPhase)."""
    buf = C.create_string_buffer(1 << 14)
    n = lib().hnhd_setup_times_json(buf, len(buf), int(reset))
    if n < 0:
        check(n, "hnhd_setup_times_json")
    return json.loads(buf.value.decode())


def timer_start():
    check(lib().hnhd_timer_start(), "timer_start")


def timer_stop() -> float:
    ms = C.c_double()
    check(lib().hnhd_timer_stop(C.byref(ms)), "timer_stop")
    return ms.value


def benchmark_algorithm(S: SpmatLocal, name: str, R: int, c: int, fused=True, app="vanilla", trials=5, warmup=0,
                        output_file: str | None = None):
    buf = C.create_string_buffer(1 << 18)
    n = lib().hnhd_benchmark_algorithm(S.h, name.encode(), output_file.encode() if output_file else None, int(fused), R,
                                       c, app.encode(), trials, warmup, buf, len(buf))
    if n < 0:
        check(n, "hnhd_benchmark_algorithm")
    return json.loads(buf.value.decode())


class GAT:
    """Multi-head graph attention (include/hnh/gat.hpp): forward pass, backward pass and a plain SGD step.
    layers: [(input_features, features_per_head, num_heads), ...].  The algorithm object must outlive this one."""

    def __init__(self, alg: Algorithm, layers, leaky_relu_alpha: float = 0.2):
        self.alg = alg
        self.layers = [tuple(int(x) for x in l) for l in layers]
        flat = (C.c_int * (3 * len(self.layers)))(*[x for l in self.layers for x in l])
        self.h = C.c_void_p()
        check(lib().hnhd_gat_create(alg.h, len(self.layers), flat, float(leaky_relu_alpha), C.byref(self.h)), "gat_create")

    def weight_shape(self, layer: int, head: int):
        r, c = C.c_int64(), C.c_int64()
        check(lib().hnhd_gat_weight_shape(self.h, layer, head, C.byref(r), C.byref(c)), "gat_weight_shape")
        return r.value, c.value

    def set_weight(self, layer: int, head: int, w):
        w = np.ascontiguousarray(w, dtype=np.float64)
        assert w.shape == self.weight_shape(layer, head), (w.shape, self.weight_shape(layer, head))
        check(lib().hnhd_gat_set_weight(self.h, layer, head, w.ctypes.data), "gat_set_weight")

    def buffer_shape(self, i: int):
        r, c = C.c_int64(), C.c_int64()
        check(lib().hnhd_gat_buffer_shape(self.h, i, C.byref(r), C.byref(c)), "gat_buffer_shape")
        return r.value, c.value

    def set_input(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        assert x.shape == self.buffer_shape(0), (x.shape, self.buffer_shape(0))
        check(lib().hnhd_gat_set_input(self.h, x.ctypes.data), "gat_set_input")

    def buffer(self, i: int):
        out = np.empty(self.buffer_shape(i), dtype=np.float64)
        check(lib().hnhd_gat_get_buffer(self.h, i, out.ctypes.data), "gat_get_buffer")
        return out

    def forward(self):
        check(lib().hnhd_gat_forward(self.h), "gat_forward")

    def supports_backward(self) -> bool:
        rc = lib().hnhd_gat_supports_backward(self.h)
        if rc < 0:
            check(rc, "gat_supports_backward")
        return rc == 1

    def backward(self, grad):
        """Gradients of L from grad = dL/d(output of the last layer) (this rank's rows), after forward() with the
        current weights.  Collective over the ranks; overwrites the gradients."""
        grad = np.ascontiguousarray(grad, dtype=np.float64)
        want = self.buffer_shape(len(self.layers))
        assert grad.shape == want, (grad.shape, want)
        check(lib().hnhd_gat_backward(self.h, grad.ctypes.data), "gat_backward")

    def weight_grad(self, layer: int, head: int):
        out = np.empty(self.weight_shape(layer, head), dtype=np.float64)
        check(lib().hnhd_gat_get_weight_grad(self.h, layer, head, out.ctypes.data), "gat_get_weight_grad")
        return out

    def input_grad(self):
        out = np.empty(self.buffer_shape(0), dtype=np.float64)
        check(lib().hnhd_gat_get_input_grad(self.h, out.ctypes.data), "gat_get_input_grad")
        return out

    def weight(self, layer: int, head: int):
        out = np.empty(self.weight_shape(layer, head), dtype=np.float64)
        check(lib().hnhd_gat_get_weight(self.h, layer, head, out.ctypes.data), "gat_get_weight")
        return out

    def sgd_step(self, lr: float):
        """W -= lr * W_grad for every weight (after backward())."""
        check(lib().hnhd_gat_sgd_step(self.h, float(lr)), "gat_sgd_step")

    def __del__(self):
        try:
            lib().hnhd_gat_destroy(self.h)
        except Exception:
            pass


def als_run(alg: Algorithm, Agt, Bgt, A0, B0, steps: int = 1, cg_iters: int = 10):
    """Distributed_ALS on caller inputs (this rank's local shards, numpy float64): ground truth from (Agt, Bgt),
    embeddings (A0, B0), `steps` alternating cg_optimizer rounds.  Returns ((residual before, after), A, B)."""
    mats = [np.ascontiguousarray(m, dtype=np.float64) for m in (Agt, Bgt, A0, B0)]
    res = (C.c_double * 2)()
    outA, outB = np.empty_like(mats[2]), np.empty_like(mats[3])
    check(lib().hnhd_als_run(alg.h, *[m.ctypes.data for m in mats], steps, cg_iters, res, outA.ctypes.data, outB.ctypes.data),
          "hnhd_als_run")
    return (res[0], res[1]), outA, outB
