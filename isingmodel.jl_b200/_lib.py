"""ctypes binding of ``libising_b200.so`` (the C ABI declared in ``include/ising_b200.h``).

There is no CPU fallback: if the shared library is missing, ``load()`` raises; if there is no CUDA
device, ``isb_create`` fails with ``ISB_ERR_CUDA`` and ``context()`` raises ``IsbError``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ISING_B200_LIB") or os.path.join(_HERE, "libising_b200.so")
CSRC = os.path.join(_HERE, "csrc")

# enums of include/ising_b200.h
OK, ERR_ARG, ERR_SIZE, ERR_NONFINITE, ERR_CUDA, ERR_UNSUPPORTED, ERR_NCCL, ERR_STATE = range(8)
RULE_HOPFIELD, RULE_GLAUBER, RULE_METROPOLIS = 0, 1, 2
BIP_SCA, BIP_MA = 0, 1
ORDER_SEQUENTIAL, ORDER_LIST, ORDER_RANDOM, ORDER_CHECKERBOARD = 0, 1, 2, 3
FLUCT_PHILOX, FLUCT_SHARED, FLUCT_PER_REPLICA = 0, 1, 2
PREC_F64, PREC_F32, PREC_AUTO, PREC_BF16X3, PREC_BF16X1, PREC_BF16X2, PREC_FP16X2, PREC_FP16X1 = 0, 1, 2, 3, 4, 5, 6, 7
PREC_I8X3, PREC_I8X2, PREC_I8X4 = 8, 9, 10
EXCH_LOCAL, EXCH_NCCL, EXCH_COPY = 0, 1, 2
I8_PRECS = (PREC_I8X3, PREC_I8X2, PREC_I8X4)

_ERR_NAMES = {1: "ISB_ERR_ARG", 2: "ISB_ERR_SIZE", 3: "ISB_ERR_NONFINITE", 4: "ISB_ERR_CUDA",
              5: "ISB_ERR_UNSUPPORTED", 6: "ISB_ERR_NCCL", 7: "ISB_ERR_STATE"}


class IsbError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{_ERR_NAMES.get(code, code)}: {message}")
        self.code = code
        self.message = message


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every CUDA source of the package for sm_100a into ``libising_b200.so`` (in-tree)."""
    cmd = ["make", "-C", CSRC, "-j", str(min(8, os.cpu_count() or 1))]
    if force:
        cmd.append("-B")
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("building libising_b200.so failed")
    return LIB_PATH


# name -> (restype, argtypes); every symbol declared in include/ising_b200.h
_vp, _i, _i64, _u64, _d = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_double
SIGNATURES = {
    "isb_version": (_i, []),
    "isb_device_count": (_i, []),
    "isb_create": (_i, [_i, C.POINTER(_vp)]),
    "isb_destroy": (None, [_vp]),
    "isb_last_error": (C.c_char_p, [_vp]),
    "isb_set_stream": (_i, [_vp, _vp]),
    "isb_synchronize": (_i, [_vp]),
    "isb_model_dense": (_i, [_vp, _i, _vp, _i64, _vp, _i, C.POINTER(_i), C.POINTER(_vp)]),
    "isb_model_sparse": (_i, [_vp, _i, _vp, _vp, _vp, _vp, C.POINTER(_i), C.POINTER(_vp)]),
    "isb_model_bipartite": (_i, [_vp, _i, _i, _vp, _i64, _vp, _vp, _i, C.POINTER(_vp)]),
    "isb_model_destroy": (None, [_vp]),
    "isb_model_retain": (_i, [_vp]),
    "isb_model_effective_couplings": (_i, [_vp, _vp, _i64]),
    "isb_model_num_visible": (_i, [_vp]),
    "isb_model_num_hidden": (_i, [_vp]),
    "isb_ens_create": (_i, [_vp, _i, C.POINTER(_vp)]),
    "isb_ens_clone": (_i, [_vp, C.POINTER(_vp)]),
    "isb_ens_select_replicas": (_i, [_vp, _vp]),
    "isb_ens_destroy": (None, [_vp]),
    "isb_ens_replicas": (_i, [_vp]),
    "isb_ens_set_spins": (_i, [_vp, _vp, _i64]),
    "isb_ens_get_spins": (_i, [_vp, _vp, _i64]),
    "isb_ens_set_hidden": (_i, [_vp, _vp, _i64]),
    "isb_ens_get_hidden": (_i, [_vp, _vp, _i64]),
    "isb_ens_energy": (_i, [_vp, _vp]),
    "isb_ens_magnetization": (_i, [_vp, _vp]),
    "isb_ens_local_field": (_i, [_vp, _vp, _i64]),
    "isb_ens_local_aux_bias": (_i, [_vp, _vp, _i64]),
    "isb_ssf_run": (_i, [_vp, _i, _i64, _i, _vp, _i, _i, _vp, _u64, _u64, _vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    "isb_ssf_run_snap": (_i, [_vp, _i, _i64, _i, _vp, _i, _i, _vp, _u64, _u64, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp,
                              _i64]),
    "isb_ssf_run_hist": (_i, [_vp, _i, _i64, _i, _vp, _i, _i, _vp, _u64, _u64, _vp, _i64, _i64, _i64, _vp]),
    "isb_ssf_run_pt": (_i, [_vp, _i, _i, _vp, _i64, _i64, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "isb_ssf_run_pa": (_i, [_vp, _i, _i, _i64, _vp, _d, _i64, _i, _i, _u64, _u64, _u64, _vp, _vp, _vp, _vp, _vp]),
    "isb_sw_run": (_i, [_vp, _i64, _u64, _u64, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
    "isb_philox_fluct": (_i, [_vp, _i, _i, _u64, _u64, _i, _i, _i64, _vp]),
    "isb_philox_nodes": (_i, [_vp, _i, _u64, _u64, _i64, _vp]),
    "isb_philox_raw": (_i, [_vp, _vp, _vp, _i, _vp]),
    "isb_bip_run": (_i, [_vp, _i, _i64, _i, _vp, _vp, _u64, _u64, _vp, _i64, _i64, _i64, _vp]),
    "isb_bip_run_snap": (_i, [_vp, _i, _i64, _i, _vp, _vp, _u64, _u64, _vp, _i64, _i64, _i64, _vp, _vp, _i64, _vp, _i64]),
    "isb_philox_bip_fluct": (_i, [_vp, _i, _i, _u64, _u64, _i, _i, _i, _i, _i64, _vp]),
    "isb_shard_model_rows": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _i, C.POINTER(_vp)]),
    "isb_shard_model_rows_q": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _i, _d, C.POINTER(_vp)]),
    "isb_shard_model_sk": (_i, [_vp, _i, _i, _i, _u64, _d, _i, C.POINTER(_vp)]),
    "isb_sk_rows": (_i, [_vp, _i, _u64, _i, _i, _vp]),
    "isb_model_shard_block": (_i, [_vp]),
    "isb_shard_halfstep_dev": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _u64, _u64, _d]),
    "isb_shard_run_create": (_i, [_vp, _i, _i, C.POINTER(_vp)]),
    "isb_shard_run_destroy": (None, [_vp]),
    "isb_nccl_unique_id": (_i, [_vp]),
    "isb_shard_run_init_nccl": (_i, [_vp, _vp]),
    "isb_shard_run_set_nccl_comm": (_i, [_vp, _vp]),
    "isb_shard_run_ipc_export": (_i, [_vp, _vp]),
    "isb_shard_run_ipc_import": (_i, [_vp, _i, _vp]),
    "isb_shard_run_barrier": (_i, [_vp]),
    "isb_shard_run_set_spins": (_i, [_vp, _vp, _i64]),
    "isb_shard_run_get_spins": (_i, [_vp, _i, _vp, _i64]),
    "isb_shard_run_steps": (_i, [_vp, _i, _i64, _vp, _i64, _u64, _u64]),
    "isb_shard_run_last_stats": (_i, [_vp, C.POINTER(_d), C.POINTER(_i64), C.POINTER(_i)]),
    "isb_ens_last_stats": (_i, [_vp, C.POINTER(_d), C.POINTER(_i64), C.POINTER(_i64), C.POINTER(_i64)]),
    "isb_ens_last_flips": (_i64, [_vp]),
    "isb_ens_last_near_ties": (_i64, [_vp]),
    "isb_ens_last_exact_fallbacks": (_i64, [_vp]),
    "isb_ens_set_tie_eps": (_i, [_vp, _d]),
    "isb_ens_set_temperature_scale": (_i, [_vp, _vp]),
}

_lib = None


def load():
    """dlopen the product library; raises (no fallback) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OSError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def check(rc: int, ctx_handle=None):
    if rc != OK:
        msg = load().isb_last_error(ctx_handle)
        raise IsbError(rc, msg.decode() if msg else "")


class Context:
    """One CUDA device (isb_ctx)."""

    def __init__(self, device: int = 0):
        L = load()
        h = _vp()
        rc = L.isb_create(int(device), C.byref(h))
        if rc != OK:
            check(rc, None)
        self.handle = h
        self.device = int(device)

    def close(self):
        if self.handle:
            load().isb_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int):
        check(load().isb_set_stream(self.handle, _vp(cuda_stream)), self.handle)

    def synchronize(self):
        check(load().isb_synchronize(self.handle), self.handle)

    # --- Philox dumps (parity tests)
    def philox_raw(self, ctr, key):
        ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
        key = np.ascontiguousarray(key, dtype=np.uint32)
        out = np.zeros_like(ctr)
        check(load().isb_philox_raw(self.handle, ptr(ctr), ptr(key), ctr.shape[0], ptr(out)), self.handle)
        return out

    def philox_fluct(self, rule, seed, step_offset, r0, nr, nsteps):
        out = np.zeros((nr, nsteps), dtype=np.float64)
        check(load().isb_philox_fluct(self.handle, rule, PREC_F64, seed, step_offset, r0, nr, nsteps, ptr(out)),
              self.handle)
        return out

    def philox_nodes(self, n, seed, step_offset, nsteps):
        out = np.zeros(nsteps, dtype=np.int32)
        check(load().isb_philox_nodes(self.handle, n, seed, step_offset, nsteps, ptr(out)), self.handle)
        return out

    def sk_rows(self, n, seed, row0, nrows):
        """Rows of the device-generated synthetic SK matrix J (isb_sk_rows)."""
        out = np.zeros((nrows, n), dtype=np.float64)
        check(load().isb_sk_rows(self.handle, int(n), int(seed), int(row0), int(nrows), ptr(out)), self.handle)
        return out

    def philox_bip_fluct(self, rule, seed, step_offset, layer, nunits, r0, nr, nsteps):
        out = np.zeros((nr, nsteps, nunits), dtype=np.float64)
        check(load().isb_philox_bip_fluct(self.handle, rule, PREC_F64, seed, step_offset, layer, nunits, r0, nr,
                                          nsteps, ptr(out)), self.handle)
        return out


_contexts: dict[int, Context] = {}


def context(device: int | None = None) -> Context:
    """Process-wide context of a device (default: LOCAL_RANK, else 0)."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    ctx = _contexts.get(device)
    if ctx is None or not ctx.handle:
        ctx = Context(device)
        _contexts[device] = ctx
    return ctx


class Model:
    """isb_model: couplings resident in HBM."""

    def __init__(self, ctx: Context, handle, kind: str, warn: int = 0):
        self.ctx, self.handle, self.kind, self.warn = ctx, handle, kind, warn

    @classmethod
    def dense(cls, ctx: Context, J, h, prec=PREC_AUTO):
        A = np.asfortranarray(np.asarray(J, dtype=np.float64))
        if A.ndim != 2:
            raise IsbError(ERR_SIZE, "J must be a matrix")
        h = None if h is None else np.ascontiguousarray(h, dtype=np.float64)
        m, w = _vp(), C.c_int(0)
        check(load().isb_model_dense(ctx.handle, A.shape[0], ptr(A), max(1, A.shape[0]), ptr(h), prec,
                                     C.byref(w), C.byref(m)), ctx.handle)
        return cls(ctx, m, "dense", w.value)

    @classmethod
    def sparse(cls, ctx: Context, J, h):
        """J: a scipy.sparse matrix (any format) -> 0-based CSC across the ABI (isb_model_sparse)."""
        import scipy.sparse as sp
        A = sp.csc_matrix(J, dtype=np.float64)
        A.sort_indices()
        if A.shape[0] != A.shape[1]:
            raise IsbError(ERR_SIZE, "J must be square")
        colptr = np.ascontiguousarray(A.indptr, dtype=np.int64)
        rowval = np.ascontiguousarray(A.indices, dtype=np.int32)
        nzval = np.ascontiguousarray(A.data, dtype=np.float64)
        h = None if h is None else np.ascontiguousarray(h, dtype=np.float64)
        m, w = _vp(), C.c_int(0)
        check(load().isb_model_sparse(ctx.handle, A.shape[0], ptr(colptr), ptr(rowval), ptr(nzval), ptr(h), C.byref(w),
                                      C.byref(m)), ctx.handle)
        return cls(ctx, m, "sparse", w.value)

    @classmethod
    def bipartite(cls, ctx: Context, W, h, b, prec=PREC_F64):
        A = np.asfortranarray(np.asarray(W, dtype=np.float64))
        if A.ndim != 2:
            raise IsbError(ERR_SIZE, "W must be a matrix")
        h = None if h is None else np.ascontiguousarray(h, dtype=np.float64)
        b = None if b is None else np.ascontiguousarray(b, dtype=np.float64)
        m = _vp()
        check(load().isb_model_bipartite(ctx.handle, A.shape[0], A.shape[1], ptr(A), max(1, A.shape[0]), ptr(h),
                                         ptr(b), prec, C.byref(m)), ctx.handle)
        return cls(ctx, m, "bipartite")

    @classmethod
    def shard_rows(cls, ctx: Context, n, n_blocks, block, Wrows, h_blk=None, b_blk=None, prec=PREC_BF16X3, wmax=0.0):
        """Row block `block` of a symmetric W (Wrows: [n // n_blocks][n]) — isb_shard_model_rows(_q).  wmax: the largest
        off-diagonal |W| of the whole matrix (int8 digit planes: every rank must use the same fixed-point grid)."""
        A = np.ascontiguousarray(Wrows, dtype=np.float64)
        h_blk = None if h_blk is None else np.ascontiguousarray(h_blk, dtype=np.float64)
        b_blk = None if b_blk is None else np.ascontiguousarray(b_blk, dtype=np.float64)
        m = _vp()
        check(load().isb_shard_model_rows_q(ctx.handle, int(n), int(n_blocks), int(block), ptr(A), ptr(h_blk),
                                            ptr(b_blk), prec, float(wmax), C.byref(m)), ctx.handle)
        obj = cls(ctx, m, "shard")
        obj.prec = prec
        return obj

    @classmethod
    def shard_sk(cls, ctx: Context, n, n_blocks, block, seed, q, prec=PREC_BF16X3):
        """Row block of the synthetic SK embedding W = (J + qI)/2 generated on the device — isb_shard_model_sk."""
        m = _vp()
        check(load().isb_shard_model_sk(ctx.handle, int(n), int(n_blocks), int(block), int(seed), float(q), prec,
                                        C.byref(m)), ctx.handle)
        obj = cls(ctx, m, "shard")
        obj.prec = prec
        return obj

    def shard_halfstep(self, R, layer, rule, in_full_ptr, out_block_ptr, seed, step_abs, T, replica_offset=0):
        """isb_shard_halfstep_dev with raw device pointers (ints)."""
        check(load().isb_shard_halfstep_dev(self.handle, int(R), int(replica_offset), int(layer), int(rule), _vp(in_full_ptr),
                                            _vp(out_block_ptr), int(seed), int(step_abs), float(T)), self.ctx.handle)

    def effective_couplings(self):
        """The couplings exactly as the kernels use them (isb_model_effective_couplings): [nv][nh]."""
        nv, nh = self.num_visible, self.num_hidden
        W = np.zeros((nv, nh), dtype=np.float64, order="F")
        check(load().isb_model_effective_couplings(self.handle, ptr(W), max(1, nv)), self.ctx.handle)
        return np.ascontiguousarray(W)

    @property
    def num_visible(self):
        return load().isb_model_num_visible(self.handle)

    @property
    def num_hidden(self):
        return load().isb_model_num_hidden(self.handle)

    def close(self):
        if self.handle:
            load().isb_model_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ShardRun:
    """isb_shard_run: the step loop of the row-sharded SCA inside the library (one object per rank).  The caller only
    carries the 128-byte NCCL id / the 64-byte IPC handles between the ranks (``wire`` does it over torch.distributed)."""

    def __init__(self, model: Model, R: int, exchange: int):
        h = _vp()
        check(load().isb_shard_run_create(model.handle, int(R), int(exchange), C.byref(h)), model.ctx.handle)
        self.model, self.handle, self.R, self.exchange = model, h, int(R), int(exchange)
        self.n = model.num_visible

    def close(self):
        if self.handle:
            load().isb_shard_run_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        check(rc, self.model.ctx.handle)

    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        check(load().isb_nccl_unique_id(C.cast(buf, _vp)), None)
        return buf.raw

    def init_nccl(self, id128: bytes):
        buf = C.create_string_buffer(bytes(id128), 128)
        self._chk(load().isb_shard_run_init_nccl(self.handle, C.cast(buf, _vp)))

    def ipc_export(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._chk(load().isb_shard_run_ipc_export(self.handle, C.cast(buf, _vp)))
        return buf.raw

    def ipc_import(self, rank: int, handle64: bytes):
        buf = C.create_string_buffer(bytes(handle64), 64)
        self._chk(load().isb_shard_run_ipc_import(self.handle, int(rank), C.cast(buf, _vp)))

    def wire(self, dist, group=None):
        """Exchange the NCCL id or the IPC handles over torch.distributed (any transport would do: 128 / 64 bytes)."""
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        if self.exchange == EXCH_NCCL:
            box = [self.nccl_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            self.init_nccl(box[0])
        elif self.exchange == EXCH_COPY:
            handles = [None] * world
            dist.all_gather_object(handles, self.ipc_export(), group=group)
            for q, h in enumerate(handles):
                if q != rank:
                    self.ipc_import(q, h)
            dist.barrier(group=group)

    def barrier(self):
        self._chk(load().isb_shard_run_barrier(self.handle))

    def set_spins(self, S):
        S = np.ascontiguousarray(S, dtype=np.int8).reshape(self.R, self.n)
        self._chk(load().isb_shard_run_set_spins(self.handle, ptr(S), self.n))

    def get_spins(self, layer: int = 0):
        S = np.zeros((self.R, self.n), dtype=np.int8)
        self._chk(load().isb_shard_run_get_spins(self.handle, int(layer), ptr(S), self.n))
        return S

    def steps(self, rule, nsteps, T, *, seed=0, step_offset=0):
        Ta = np.ascontiguousarray(np.atleast_1d(T), dtype=np.float64)
        self._chk(load().isb_shard_run_steps(self.handle, int(rule), int(nsteps), ptr(Ta), Ta.size, int(seed), int(step_offset)))

    def last_stats(self):
        ms, nl, ng = _d(0), _i64(0), _i(0)
        load().isb_shard_run_last_stats(self.handle, C.byref(ms), C.byref(nl), C.byref(ng))
        return {"device_ms": ms.value, "launches": nl.value, "groups": ng.value}


class Ensemble:
    """isb_ens: R replicas of one model."""

    def __init__(self, model: Model, R: int):
        e = _vp()
        check(load().isb_ens_create(model.handle, int(R), C.byref(e)), model.ctx.handle)
        self.model, self.handle, self.R = model, e, int(R)
        self.nv, self.nh = model.num_visible, model.num_hidden

    def clone(self):
        """isb_ens_clone: an independent device-side copy (deepcopy of the host object)."""
        e = _vp()
        check(load().isb_ens_clone(self.handle, C.byref(e)), self.model.ctx.handle)
        new = object.__new__(Ensemble)
        new.model, new.handle, new.R, new.nv, new.nh = self.model, e, self.R, self.nv, self.nh
        return new

    def close(self):
        if self.handle:
            load().isb_ens_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        check(rc, self.model.ctx.handle)

    def set_spins(self, S):
        S = np.ascontiguousarray(S, dtype=np.int8).reshape(self.R, -1)
        self._chk(load().isb_ens_set_spins(self.handle, ptr(S), S.shape[1]))

    def get_spins(self):
        S = np.empty((self.R, self.nv), dtype=np.int8)
        self._chk(load().isb_ens_get_spins(self.handle, ptr(S), self.nv))
        return S

    def set_hidden(self, Tm):
        Tm = np.ascontiguousarray(Tm, dtype=np.int8).reshape(self.R, -1)
        self._chk(load().isb_ens_set_hidden(self.handle, ptr(Tm), Tm.shape[1]))

    def get_hidden(self):
        Tm = np.empty((self.R, self.nh), dtype=np.int8)
        self._chk(load().isb_ens_get_hidden(self.handle, ptr(Tm), self.nh))
        return Tm

    def energy(self):
        E = np.zeros(self.R, dtype=np.float64)
        self._chk(load().isb_ens_energy(self.handle, ptr(E)))
        return E

    def magnetization(self):
        M = np.zeros(self.R, dtype=np.float64)
        self._chk(load().isb_ens_magnetization(self.handle, ptr(M)))
        return M

    def local_field(self):
        F = np.zeros((self.R, self.nv), dtype=np.float64)
        self._chk(load().isb_ens_local_field(self.handle, ptr(F), self.nv))
        return F

    def local_aux_bias(self):
        A = np.zeros((self.R, self.nh), dtype=np.float64)
        self._chk(load().isb_ens_local_aux_bias(self.handle, ptr(A), self.nh))
        return A

    def set_temperature_scale(self, scale):
        """Per-replica temperature factors (R values) for every later run; None clears them."""
        a = None if scale is None else np.ascontiguousarray(scale, dtype=np.float64)
        if a is not None and a.size != self.R:
            raise IsbError(ERR_SIZE, f"temperature scale has {a.size} entries for {self.R} replicas")
        self._chk(load().isb_ens_set_temperature_scale(self.handle, ptr(a)))

    def set_tie_eps(self, eps: float):
        self._chk(load().isb_ens_set_tie_eps(self.handle, float(eps)))

    def ssf_run(self, rule, nsteps, *, order=ORDER_SEQUENTIAL, nodes=None, start=0, fluct=None,
                fluct_per_replica=False, seed=0, step_offset=0, T=None, steps_per_T=1, trace_every=0,
                want_E=True, want_M=True, want_S=False, hist=None):
        """isb_ssf_run / isb_ssf_run_snap. Returns dict(flips[R], E[ntr][R] | None, M[ntr][R] | None, S[ntr][R][N] | None).
        With ``hist`` (int64[2^N], accumulated into) the call is isb_ssf_run_hist and returns {"hist": hist}."""
        nsteps = int(nsteps)
        nodes_a = None if nodes is None else np.ascontiguousarray(nodes, dtype=np.int32)
        if nodes_a is not None:
            order = ORDER_LIST
            if nodes_a.size != nsteps:
                raise IsbError(ERR_SIZE, f"node list has {nodes_a.size} entries for {nsteps} steps")
        if fluct is None:
            mode, fl = FLUCT_PHILOX, None
        else:
            fl = np.ascontiguousarray(fluct, dtype=np.float64)
            mode = FLUCT_PER_REPLICA if fluct_per_replica else FLUCT_SHARED
            need = nsteps * (self.R if fluct_per_replica else 1)
            if fl.size != need:
                raise IsbError(ERR_SIZE, f"fluctuation array has {fl.size} entries, expected {need}")
        Ta = None if T is None else np.ascontiguousarray(np.atleast_1d(T), dtype=np.float64)
        ntr = nsteps // trace_every if trace_every > 0 else 0
        if hist is not None:
            if hist.dtype != np.int64 or not hist.flags.c_contiguous or hist.size != 1 << min(self.nv, 62):
                raise IsbError(ERR_SIZE, "hist must be a contiguous int64 array with 2^N entries")
            self._chk(load().isb_ssf_run_hist(self.handle, rule, nsteps, order, ptr(nodes_a), int(start), mode, ptr(fl),
                                              int(seed), int(step_offset), ptr(Ta), 0 if Ta is None else Ta.size,
                                              int(steps_per_T), int(trace_every), ptr(hist)))
            return {"hist": hist}
        E = np.zeros((ntr, self.R)) if (ntr and want_E) else None
        M = np.zeros((ntr, self.R)) if (ntr and want_M) else None
        S = np.zeros((ntr, self.R, self.nv), dtype=np.int8) if (ntr and want_S) else None
        flips = np.zeros(self.R, dtype=np.int64)
        self._chk(load().isb_ssf_run_snap(self.handle, rule, nsteps, order, ptr(nodes_a), int(start), mode, ptr(fl),
                                          int(seed), int(step_offset), ptr(Ta), 0 if Ta is None else Ta.size,
                                          int(steps_per_T), int(trace_every), ptr(E), ptr(M), ptr(flips), ptr(S),
                                          self.nv))
        return {"flips": flips, "E": E, "M": M, "S": S}

    def ssf_run_pt(self, rule, levels, rounds, steps_per_round, *, order=ORDER_SEQUENTIAL, start=0, seed=0, step_offset=0,
                   round_offset=0, level_of=None, want_E=True, want_M=False, want_Q=False):
        """isb_ssf_run_pt: ``rounds`` rounds of ``steps_per_round`` steps, each followed by one replica exchange, all on the
        device.  ``level_of`` (R entries, default: slot s of every ladder holds level s) is the level each replica holds.
        Returns dict(level_of[R] (final), E / M [rounds][levels][ladders] | None, Q [rounds][levels][ladders/2] | None,
        accepted[levels-1], flips[R])."""
        lv = np.ascontiguousarray(levels, dtype=np.float64).reshape(-1)
        L, rounds = lv.size, int(rounds)
        G = self.R // L if L else 0
        if level_of is None:       # slot s of every ladder holds level s (a mismatch of R and L is the library's error)
            level_of = np.arange(self.R) % L if L else np.zeros(self.R)
        lo = np.array(level_of, dtype=np.int32).reshape(-1)
        if lo.size != self.R:
            raise IsbError(ERR_SIZE, f"level_of has {lo.size} entries for {self.R} replicas")
        E = np.zeros((rounds, L, G)) if want_E else None
        M = np.zeros((rounds, L, G)) if want_M else None
        Q = np.zeros((rounds, L, G // 2)) if want_Q else None
        acc = np.zeros(max(L - 1, 0), dtype=np.int64)
        flips = np.zeros(self.R, dtype=np.int64)
        self._chk(load().isb_ssf_run_pt(self.handle, int(rule), L, ptr(lv), rounds, int(steps_per_round), int(order),
                                        int(start), int(seed), int(step_offset), int(round_offset), ptr(lo), ptr(E),
                                        ptr(M), ptr(Q), ptr(acc), ptr(flips)))
        return {"level_of": lo, "E": E, "M": M, "Q": Q, "accepted": acc, "flips": flips}

    def select_replicas(self, src):
        """isb_ens_select_replicas: replica r takes the state (spins and cached fields, bit for bit) of replica src[r]."""
        a = np.ascontiguousarray(src, dtype=np.int32).reshape(-1)
        if a.size != self.R:
            raise IsbError(ERR_SIZE, f"src has {a.size} entries for {self.R} replicas")
        self._chk(load().isb_ens_select_replicas(self.handle, ptr(a)))

    def ssf_run_pa(self, rule, n_pop, T, steps_per_T, *, T_next=0.0, order=ORDER_SEQUENTIAL, start=0, seed=0,
                   step_offset=0, T_offset=0, family=None, want_E=True, want_M=False):
        """isb_ssf_run_pa: population annealing over the temperatures T (``steps_per_T`` steps each), resampling every
        population after each step towards the next temperature (after the last one towards ``T_next`` when > 0), all on
        the device.  ``family`` (R int32 labels or None) follows the resampling.  Returns dict(E / M [nT][R] | None (by
        slot, before that step's resampling), lnQ [nT - 1 + (T_next > 0)][n_pop], family[R] | None, flips[R])."""
        Ta = np.ascontiguousarray(np.atleast_1d(T), dtype=np.float64).reshape(-1)
        nT, n_pop = Ta.size, int(n_pop)
        fam = None if family is None else np.array(family, dtype=np.int32).reshape(-1)
        if fam is not None and fam.size != self.R:
            raise IsbError(ERR_SIZE, f"family has {fam.size} entries for {self.R} replicas")
        n_res = max(nT - 1 + (1 if T_next > 0 else 0), 0) if nT else 0
        E = np.zeros((nT, self.R)) if want_E else None
        M = np.zeros((nT, self.R)) if want_M else None
        lnQ = np.zeros((n_res, max(n_pop, 0)))
        flips = np.zeros(self.R, dtype=np.int64)
        self._chk(load().isb_ssf_run_pa(self.handle, int(rule), n_pop, nT, ptr(Ta), float(T_next), int(steps_per_T),
                                        int(order), int(start), int(seed), int(step_offset), int(T_offset), ptr(fam),
                                        ptr(E), ptr(M), ptr(lnQ), ptr(flips)))
        return {"E": E, "M": M, "lnQ": lnQ, "family": fam, "flips": flips}

    def sw_run(self, nsweeps, T, *, sweeps_per_T=1, trace_every=0, seed=0, sweep_offset=0, want_E=True, want_M=True,
               want_csq=True):
        """isb_sw_run: ``nsweeps`` Swendsen-Wang sweeps of every replica (sparse models), sweep k at T[k // sweeps_per_T]
        times the replica's temperature factor.  Returns dict(E / M [ntr][R] float64 | None, csq [ntr][R] int64 | None
        (sum of |C|^2 over the clusters of the traced sweep), flips[R]); ntr = nsweeps // trace_every."""
        nsweeps = int(nsweeps)
        Ta = np.ascontiguousarray(np.atleast_1d(T), dtype=np.float64).reshape(-1)
        ntr = nsweeps // trace_every if trace_every > 0 else 0
        E = np.zeros((ntr, self.R)) if (ntr and want_E) else None
        M = np.zeros((ntr, self.R)) if (ntr and want_M) else None
        csq = np.zeros((ntr, self.R), dtype=np.int64) if (ntr and want_csq) else None
        flips = np.zeros(self.R, dtype=np.int64)
        self._chk(load().isb_sw_run(self.handle, nsweeps, int(seed), int(sweep_offset), ptr(Ta), Ta.size, int(sweeps_per_T),
                                    int(trace_every), ptr(E), ptr(M), ptr(csq), ptr(flips)))
        return {"E": E, "M": M, "csq": csq, "flips": flips}

    def bip_run(self, rule, nsteps, *, Fv=None, Fh=None, fluct_per_replica=False, seed=0, step_offset=0, T=None,
                steps_per_T=1, trace_every=0, want_S=False):
        """isb_bip_run / isb_bip_run_snap. Fv: [nsteps][nv] (shared) or [R][nsteps][nv]; returns E[ntr][R] or None,
        or (E, Sv[ntr][R][nv], Sh[ntr][R][nh]) with want_S."""
        nsteps = int(nsteps)
        if Fv is None and Fh is None:
            mode, fv, fh = FLUCT_PHILOX, None, None
        else:
            fv = np.ascontiguousarray(Fv, dtype=np.float64)
            fh = np.ascontiguousarray(Fh, dtype=np.float64)
            mode = FLUCT_PER_REPLICA if fluct_per_replica else FLUCT_SHARED
            rep = self.R if fluct_per_replica else 1
            if fv.size != rep * nsteps * self.nv or fh.size != rep * nsteps * self.nh:
                raise IsbError(ERR_SIZE, "fluctuation arrays do not match (replicas, steps, units)")
        Ta = None if T is None else np.ascontiguousarray(np.atleast_1d(T), dtype=np.float64)
        ntr = nsteps // trace_every if trace_every > 0 else 0
        E = np.zeros((ntr, self.R)) if ntr else None
        Sv = np.zeros((ntr, self.R, self.nv), dtype=np.int8) if (ntr and want_S) else None
        Sh = np.zeros((ntr, self.R, self.nh), dtype=np.int8) if (ntr and want_S) else None
        self._chk(load().isb_bip_run_snap(self.handle, rule, nsteps, mode, ptr(fv), ptr(fh), int(seed), int(step_offset),
                                          ptr(Ta), 0 if Ta is None else Ta.size, int(steps_per_T), int(trace_every),
                                          ptr(E), ptr(Sv), self.nv, ptr(Sh), self.nh))
        return (E, Sv, Sh) if want_S else E

    def last_stats(self):
        ms, nl, hi, do = _d(0), _i64(0), _i64(0), _i64(0)
        load().isb_ens_last_stats(self.handle, C.byref(ms), C.byref(nl), C.byref(hi), C.byref(do))
        return {"kernel_ms": ms.value, "launches": nl.value, "h2d_bytes": hi.value, "d2h_bytes": do.value,
                "flips": load().isb_ens_last_flips(self.handle),
                "near_ties": load().isb_ens_last_near_ties(self.handle),
                "exact_fallbacks": load().isb_ens_last_exact_fallbacks(self.handle)}
