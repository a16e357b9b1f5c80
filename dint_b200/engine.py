"""ctypes binding of libdint_b200.so (include/dint_b200.h): the GPU-resident stand-in for one
reference server process (`server <threads>` / `server_shard <id> <threads>`).

There is no CPU implementation behind this class: if the CUDA library cannot be built/loaded, or no
CUDA device is present, construction raises.
"""
import ctypes as C
import os

import numpy as np

from . import _build
from .wire import MSG_SIZE, LOG_ENTRY_SIZE, KIND_NAMES

DINT_OK, DINT_EPROTO = 0, -71


class DintCfg(C.Structure):
    _fields_ = [("lock_slots", C.c_uint32), ("log_ring", C.c_uint32), ("subs_sizing", C.c_uint32),
                ("subs_populate", C.c_uint32), ("accts_sizing", C.c_uint32), ("accts_populate", C.c_uint32),
                ("n_shards", C.c_uint32), ("shard_id", C.c_uint32), ("chunk", C.c_uint32),
                ("kv_capacity_log2", C.c_uint32 * 5), ("flags", C.c_uint32), ("txn_shards", C.c_uint32),
                ("txn_shard_id", C.c_uint32), ("reserved", C.c_uint32 * 2)]


class DintStats(C.Structure):
    _fields_ = [("requests", C.c_uint64), ("chunks", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("conflicted", C.c_uint64), ("max_run", C.c_uint64), ("errors", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("kv_rebuilds", C.c_uint64),
                ("fallback_chunks", C.c_uint64), ("reserved", C.c_uint64 * 2)]


class DintPeerPtrs(C.Structure):
    _fields_ = [("p", C.c_uint64 * 8)]

    @classmethod
    def of(cls, ptrs):
        o = cls()
        for i, v in enumerate(ptrs):
            o.p[i] = int(v)
        return o


class DintKernelTime(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("launches", C.c_uint64), ("total_ms", C.c_double)]


_lib = None

# every symbol include/dint_b200.h declares
ABI_SYMBOLS = [
    "dint_msg_size", "dint_default_cfg", "dint_create", "dint_destroy", "dint_populate", "dint_load",
    "dint_submit", "dint_submit_device", "dint_route_owner", "dint_route_partition", "dint_route_unpermute", "dint_route_tile_records", "dint_route_dispatch", "dint_route_combine", "dint_p2p_wait", "dint_p2p_signal", "dint_shard_create", "dint_shard_destroy", "dint_shard_submit_many", "dint_shard_submit_host", "dint_shard_submit_many_v", "dint_shard_flags", "dint_cluster_create", "dint_cluster_populate", "dint_cluster_submit", "dint_cluster_engine", "dint_cluster_size", "dint_cluster_overflow_retries", "dint_shard_recover", "dint_cluster_destroy", "dint_clients_create", "dint_clients_run", "dint_clients_stats", "dint_clients_peek", "dint_clients_destroy", "dint_txn_clients_create", "dint_txn_clients_run", "dint_txn_clients_stats", "dint_txn_clients_peek", "dint_txn_clients_destroy", "dint_snapshot_create", "dint_snapshot_restore", "dint_snapshot_destroy", "dint_sync", "dint_kv_get", "dint_kv_count", "dint_lock_state",
    "dint_lock_slot", "dint_dump_log", "dint_log_entry_size", "dint_get_stats", "dint_reset_stats",
    "dint_profile", "dint_kernel_times", "dint_last_error", "dint_host_alloc", "dint_host_free",
    "dint_test_fasthash64", "dint_test_fastmod", "dint_test_host_slices",
]


def lib():
    """Load (building first if the sources are newer) libdint_b200.so.  Raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if _build.find_nvcc() is not None:
        _build.build()
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing and nvcc is not available: dint_b200 has no CPU fallback")
    L = C.CDLL(path)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    L.dint_msg_size.restype = u32; L.dint_msg_size.argtypes = [i32]
    L.dint_default_cfg.restype = None; L.dint_default_cfg.argtypes = [i32, C.POINTER(DintCfg)]
    L.dint_create.restype = i32; L.dint_create.argtypes = [i32, C.POINTER(DintCfg), i32, C.POINTER(vp)]
    L.dint_destroy.restype = None; L.dint_destroy.argtypes = [vp]
    L.dint_populate.restype = i32; L.dint_populate.argtypes = [vp]
    L.dint_load.restype = i32; L.dint_load.argtypes = [vp, i32, vp, vp, u64]
    L.dint_submit.restype = i32; L.dint_submit.argtypes = [vp, vp, u64, vp]
    L.dint_submit_device.restype = i32; L.dint_submit_device.argtypes = [vp, vp, u64, vp, vp]
    L.dint_route_owner.restype = i32; L.dint_route_owner.argtypes = [vp, vp, u64, vp, vp]
    L.dint_route_partition.restype = i32; L.dint_route_partition.argtypes = [vp, vp, vp, u64, u32, vp, vp, vp, vp]
    pp = C.POINTER(DintPeerPtrs)
    L.dint_route_tile_records.restype = u32; L.dint_route_tile_records.argtypes = [vp]
    L.dint_route_dispatch.restype = i32; L.dint_route_dispatch.argtypes = [vp, vp, vp, u64, u32, u32, u32, pp, pp, u32, vp, vp, vp, vp]
    L.dint_route_combine.restype = i32; L.dint_route_combine.argtypes = [vp, pp, vp, vp, u64, u32, u32, vp, vp]
    L.dint_p2p_wait.restype = i32; L.dint_p2p_wait.argtypes = [vp, vp, u32, u32, vp, vp]
    L.dint_p2p_signal.restype = i32; L.dint_p2p_signal.argtypes = [vp, pp, u32, u32, u32, vp]
    L.dint_shard_create.restype = i32; L.dint_shard_create.argtypes = [vp, u32, u32, u32, u32, pp, pp, pp, u64, C.POINTER(vp)]
    L.dint_shard_submit_many_v.restype = i32; L.dint_shard_submit_many_v.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(vp), C.POINTER(u64), C.POINTER(u32), C.POINTER(vp), vp]
    L.dint_shard_submit_host.restype = i32; L.dint_shard_submit_host.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(vp), u64, C.POINTER(vp)]
    L.dint_cluster_create.restype = i32; L.dint_cluster_create.argtypes = [i32, C.POINTER(DintCfg), i32, C.POINTER(i32), u64, C.POINTER(vp)]
    L.dint_cluster_populate.restype = i32; L.dint_cluster_populate.argtypes = [vp]
    L.dint_cluster_submit.restype = i32; L.dint_cluster_submit.argtypes = [vp, vp, u64, vp, vp]
    L.dint_cluster_engine.restype = vp; L.dint_cluster_engine.argtypes = [vp, i32]
    L.dint_cluster_size.restype = u32; L.dint_cluster_size.argtypes = [vp]
    L.dint_cluster_overflow_retries.restype = u64; L.dint_cluster_overflow_retries.argtypes = [vp]
    L.dint_shard_recover.restype = i32; L.dint_shard_recover.argtypes = [vp, u32, C.POINTER(u32)]
    L.dint_cluster_destroy.restype = None; L.dint_cluster_destroy.argtypes = [vp]
    L.dint_clients_create.restype = i32; L.dint_clients_create.argtypes = [vp, u32, u64, u32, C.c_double, u32, C.POINTER(vp)]
    L.dint_clients_run.restype = i32; L.dint_clients_run.argtypes = [vp, u32, vp]
    L.dint_clients_stats.restype = i32; L.dint_clients_stats.argtypes = [vp, C.POINTER(u64)]
    L.dint_clients_peek.restype = i32; L.dint_clients_peek.argtypes = [vp, vp, vp]
    L.dint_clients_destroy.restype = None; L.dint_clients_destroy.argtypes = [vp]
    L.dint_txn_clients_create.restype = i32; L.dint_txn_clients_create.argtypes = [C.POINTER(vp), u32, u32, u32, u32, C.POINTER(vp)]
    L.dint_txn_clients_run.restype = i32; L.dint_txn_clients_run.argtypes = [vp, u32, vp]
    L.dint_txn_clients_stats.restype = i32; L.dint_txn_clients_stats.argtypes = [vp, C.POINTER(u64)]
    L.dint_txn_clients_peek.restype = i32; L.dint_txn_clients_peek.argtypes = [vp, vp, vp, vp, C.POINTER(u64)]
    L.dint_txn_clients_destroy.restype = None; L.dint_txn_clients_destroy.argtypes = [vp]
    L.dint_snapshot_create.restype = i32; L.dint_snapshot_create.argtypes = [vp, C.POINTER(vp)]
    L.dint_snapshot_restore.restype = i32; L.dint_snapshot_restore.argtypes = [vp, vp]
    L.dint_snapshot_destroy.restype = None; L.dint_snapshot_destroy.argtypes = [vp]
    L.dint_shard_destroy.restype = None; L.dint_shard_destroy.argtypes = [vp]
    L.dint_shard_submit_many.restype = i32; L.dint_shard_submit_many.argtypes = [vp, u32, C.POINTER(vp), C.POINTER(vp), u64, C.POINTER(vp), vp]
    L.dint_shard_flags.restype = i32; L.dint_shard_flags.argtypes = [vp, C.POINTER(u32)]
    L.dint_route_unpermute.restype = i32; L.dint_route_unpermute.argtypes = [vp, vp, vp, u64, vp, vp]
    L.dint_sync.restype = i32; L.dint_sync.argtypes = [vp]
    L.dint_kv_get.restype = i32; L.dint_kv_get.argtypes = [vp, i32, u64, vp, C.POINTER(u32)]
    L.dint_kv_count.restype = C.c_int64; L.dint_kv_count.argtypes = [vp, i32]
    L.dint_lock_state.restype = i32; L.dint_lock_state.argtypes = [vp, i32, u32, C.POINTER(u32)]
    L.dint_lock_slot.restype = u32; L.dint_lock_slot.argtypes = [vp, i32, u64]
    L.dint_dump_log.restype = i32; L.dint_dump_log.argtypes = [vp, vp, C.POINTER(u64)]
    L.dint_log_entry_size.restype = u32; L.dint_log_entry_size.argtypes = [i32]
    L.dint_get_stats.restype = i32; L.dint_get_stats.argtypes = [vp, C.POINTER(DintStats)]
    L.dint_reset_stats.restype = None; L.dint_reset_stats.argtypes = [vp]
    L.dint_profile.restype = i32; L.dint_profile.argtypes = [vp, i32]
    L.dint_kernel_times.restype = i32; L.dint_kernel_times.argtypes = [vp, C.POINTER(DintKernelTime), i32]
    L.dint_last_error.restype = C.c_char_p; L.dint_last_error.argtypes = []
    L.dint_host_alloc.restype = vp; L.dint_host_alloc.argtypes = [C.c_size_t]
    L.dint_host_free.restype = None; L.dint_host_free.argtypes = [vp]
    L.dint_test_fasthash64.restype = u64; L.dint_test_fasthash64.argtypes = [u64, i32]
    L.dint_test_fastmod.restype = u32; L.dint_test_fastmod.argtypes = [u64, u32]
    _lib = L
    return L


class DintError(RuntimeError):
    def __init__(self, code, what):
        msg = lib().dint_last_error().decode(errors="replace")
        super().__init__(f"{what}: error {code} ({msg})")
        self.code = code


def default_cfg(kind, **over):
    cfg = DintCfg()
    lib().dint_default_cfg(kind, C.byref(cfg))
    for k, v in over.items():
        if k == "kv_capacity_log2":
            for i, x in enumerate(v):
                cfg.kv_capacity_log2[i] = x
        else:
            setattr(cfg, k, v)
    return cfg


class PinnedBuffer:
    """Page-locked host buffer exposed as a numpy uint8 array (dint_host_alloc)."""

    def __init__(self, nbytes):
        self.nbytes = max(int(nbytes), 1)
        self.ptr = lib().dint_host_alloc(self.nbytes)
        if not self.ptr:
            raise MemoryError("dint_host_alloc failed")
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_uint8)), shape=(self.nbytes,))

    def close(self):
        if self.ptr:
            self.array = None
            lib().dint_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Engine:
    """One GPU-resident server of the given kind.

    submit() has the semantics of feeding the requests, in order, to ONE thread of the reference
    server and collecting its replies (see include/dint_b200.h).
    """

    def __init__(self, kind, device=0, populate=False, **cfg_over):
        self.kind = kind
        self.msg = MSG_SIZE[kind]
        self.cfg = default_cfg(kind, **cfg_over)
        self.device = device
        h = C.c_void_p()
        rc = lib().dint_create(kind, C.byref(self.cfg), device, C.byref(h))
        if rc != 0:
            raise DintError(rc, f"dint_create({KIND_NAMES[kind]})")
        self.h = h
        if populate:
            self.populate()

    def close(self):
        if getattr(self, "h", None):
            lib().dint_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- population ------------------------------------------------------------------------------
    def populate(self):
        rc = lib().dint_populate(self.h)
        if rc != 0:
            raise DintError(rc, "dint_populate")

    def load(self, table, keys, vals):
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        vals = np.ascontiguousarray(vals, dtype=np.uint8)
        rc = lib().dint_load(self.h, table, keys.ctypes.data, vals.ctypes.data, keys.size)
        if rc != 0:
            raise DintError(rc, "dint_load")

    # -- request path ----------------------------------------------------------------------------
    def submit(self, req, out=None, check=True):
        """Host path: req is a uint8 array of n*msg bytes (or structured wire records)."""
        raw = np.ascontiguousarray(req).view(np.uint8).reshape(-1)
        n = raw.size // self.msg
        if raw.size != n * self.msg:
            raise ValueError("request buffer is not a whole number of wire records")
        if out is None:
            out = np.empty_like(raw)
        rc = lib().dint_submit(self.h, raw.ctypes.data, n, out.ctypes.data)
        if rc != 0 and (check or rc != DINT_EPROTO):
            raise DintError(rc, "dint_submit")
        return out

    def submit_device(self, req_ptr, n, resp_ptr, stream=0):
        """Device path: raw device pointers (16-byte aligned), asynchronous on `stream`."""
        rc = lib().dint_submit_device(self.h, C.c_void_p(req_ptr), n, C.c_void_p(resp_ptr),
                                      C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise DintError(rc, "dint_submit_device")

    def submit_tensor(self, req, out=None, stream=None):
        """Device path on torch CUDA uint8 tensors; runs on the current torch stream by default."""
        import torch
        assert req.is_cuda and req.dtype == torch.uint8 and req.is_contiguous()
        n = req.numel() // self.msg
        if out is None:
            out = torch.empty_like(req)
        s = stream if stream is not None else torch.cuda.current_stream(req.device).cuda_stream
        self.submit_device(req.data_ptr(), n, out.data_ptr(), s)
        return out

    def route_owner(self, req, stream=None):
        """owner shard (uint8 CUDA tensor) of every wire record in the CUDA uint8 tensor `req`."""
        import torch
        n = req.numel() // self.msg
        owner = torch.empty(n, dtype=torch.uint8, device=req.device)
        s = stream if stream is not None else torch.cuda.current_stream(req.device).cuda_stream
        rc = lib().dint_route_owner(self.h, C.c_void_p(req.data_ptr()), n, C.c_void_p(owner.data_ptr()),
                                    C.c_void_p(s) if s else None)
        if rc != 0:
            raise DintError(rc, "dint_route_owner")
        return owner

    def route_partition(self, req, owner, n_shards):
        """Stable partition of the CUDA uint8 tensor `req` by `owner` (uint8 tensor): returns (sorted, perm, counts)."""
        import torch
        n = owner.numel()
        out = torch.empty_like(req)
        perm = torch.empty(n, dtype=torch.int32, device=req.device)
        counts = torch.empty(n_shards, dtype=torch.int32, device=req.device)
        s = torch.cuda.current_stream(req.device).cuda_stream
        rc = lib().dint_route_partition(self.h, C.c_void_p(req.data_ptr()), C.c_void_p(owner.data_ptr()), n, n_shards,
                                        C.c_void_p(out.data_ptr()), C.c_void_p(perm.data_ptr()), C.c_void_p(counts.data_ptr()),
                                        C.c_void_p(s) if s else None)
        if rc != 0:
            raise DintError(rc, "dint_route_partition")
        return out, perm, counts

    def route_state(self, n, device):
        """Buffers the dispatch fills for the combine: (owner uint8 [n], tilebase int32 [tiles * 8])."""
        import torch
        tr = lib().dint_route_tile_records(self.h)
        tiles = (n + tr - 1) // tr
        return (torch.empty(max(n, 1), dtype=torch.uint8, device=device),
                torch.empty(max(tiles, 1) * 8, dtype=torch.int32, device=device))

    def route_dispatch(self, req, n, n_shards, rank, cap, slab_ptrs, flags, owner_in=None, sig_ptrs=None, epoch=0, state=None,
                       stream=None):
        """Fused stable partition of n records into per-shard slabs (see dint_route_dispatch).  slab_ptrs /
        sig_ptrs: DintPeerPtrs; flags: int32 CUDA tensor (>= 2).  Returns the (owner, tilebase) state."""
        import torch
        if state is None:
            state = self.route_state(n, req.device)
        s = stream if stream is not None else torch.cuda.current_stream(req.device).cuda_stream
        rc = lib().dint_route_dispatch(self.h, C.c_void_p(req.data_ptr()), C.c_void_p(owner_in.data_ptr()) if owner_in is not None else None,
                                       n, n_shards, rank, cap, C.byref(slab_ptrs), C.byref(sig_ptrs) if sig_ptrs is not None else None,
                                       epoch, C.c_void_p(state[0].data_ptr()), C.c_void_p(state[1].data_ptr()),
                                       C.c_void_p(flags.data_ptr()), C.c_void_p(s) if s else None)
        if rc != 0:
            raise DintError(rc, "dint_route_dispatch")
        return state

    def route_combine(self, reply_ptrs, state, n, n_shards, cap, out, stream=None):
        import torch
        s = stream if stream is not None else torch.cuda.current_stream(out.device).cuda_stream
        rc = lib().dint_route_combine(self.h, C.byref(reply_ptrs), C.c_void_p(state[0].data_ptr()), C.c_void_p(state[1].data_ptr()),
                                      n, n_shards, cap, C.c_void_p(out.data_ptr()), C.c_void_p(s) if s else None)
        if rc != 0:
            raise DintError(rc, "dint_route_combine")
        return out

    @staticmethod
    def slab_ptrs(base_ptr, n_shards, stride_bytes):
        """DintPeerPtrs for slabs laid out back to back in one local buffer."""
        return DintPeerPtrs.of([base_ptr + o * stride_bytes for o in range(n_shards)])

    def route_unpermute(self, sorted_resp, perm, out=None):
        import torch
        n = perm.numel()
        if out is None:
            out = torch.empty_like(sorted_resp)     # pass `out` (n_original * msg bytes) when perm has padding slots
        s = torch.cuda.current_stream(sorted_resp.device).cuda_stream
        rc = lib().dint_route_unpermute(self.h, C.c_void_p(sorted_resp.data_ptr()), C.c_void_p(perm.data_ptr()), n,
                                        C.c_void_p(out.data_ptr()), C.c_void_p(s) if s else None)
        if rc != 0:
            raise DintError(rc, "dint_route_unpermute")
        return out

    def snapshot(self):
        """Device-to-device copy of the whole server state; returns a handle for restore()."""
        h = C.c_void_p()
        rc = lib().dint_snapshot_create(self.h, C.byref(h))
        if rc != 0:
            raise DintError(rc, "dint_snapshot_create")
        return h

    def restore(self, snap, stream=None):
        """Asynchronous on the current torch stream (or `stream`): order it between submit calls."""
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        rc = lib().dint_snapshot_restore(snap, C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise DintError(rc, "dint_snapshot_restore")

    def free_snapshot(self, snap):
        lib().dint_snapshot_destroy(snap)

    def sync(self, check=True):
        rc = lib().dint_sync(self.h)
        if rc != 0 and (check or rc != DINT_EPROTO):
            raise DintError(rc, "dint_sync")
        return rc

    # -- inspection ------------------------------------------------------------------------------
    def kv_get(self, table, key):
        val = (C.c_uint8 * 40)()
        ver = C.c_uint32(0)
        rc = lib().dint_kv_get(self.h, table, key, val, C.byref(ver))
        if rc < 0:
            raise DintError(rc, "dint_kv_get")
        return None if rc == 1 else (bytes(val), ver.value)

    def kv_count(self, table):
        return lib().dint_kv_count(self.h, table)

    def lock_slot(self, table, key):
        return lib().dint_lock_slot(self.h, table, key)

    def lock_state(self, table, slot):
        out = (C.c_uint32 * 2)()
        rc = lib().dint_lock_state(self.h, table, slot, out)
        if rc != 0:
            raise DintError(rc, "dint_lock_state")
        return out[0], out[1]

    def dump_log(self):
        es = LOG_ENTRY_SIZE[self.kind]
        n = self.cfg.log_ring
        out = np.zeros((n, es), dtype=np.uint8)
        appended = C.c_uint64(0)
        rc = lib().dint_dump_log(self.h, out.ctypes.data, C.byref(appended))
        if rc != 0:
            raise DintError(rc, "dint_dump_log")
        return out, appended.value

    def stats(self):
        s = DintStats()
        rc = lib().dint_get_stats(self.h, C.byref(s))
        if rc != 0:
            raise DintError(rc, "dint_get_stats")
        return {k: getattr(s, k) for k, _ in DintStats._fields_ if k != "reserved"}

    def reset_stats(self):
        lib().dint_reset_stats(self.h)

    PROF_CLASSIFY, PROF_LOG_SCAN, PROF_APPLY, PROF_ORDERED, PROF_LOAD = 1, 2, 4, 8, 16

    def profile(self, enable=True):
        """True/1 = time every kernel with CUDA events, False/0 = off, or a mask of Engine.PROF_*."""
        rc = lib().dint_profile(self.h, int(enable))
        if rc != 0:
            raise DintError(rc, "dint_profile")

    def kernel_times(self):
        arr = (DintKernelTime * 16)()
        k = lib().dint_kernel_times(self.h, arr, 16)
        return {arr[i].name.decode(): (arr[i].launches, arr[i].total_ms) for i in range(max(k, 0))}


class GpuClients:
    """lock_fasst closed-loop clients resident on the GPU next to `engine` (dint_clients_*)."""

    def __init__(self, engine, n_clients, seed=20230, n_keys=24_000_000, zipf_theta=0.0, read_pct=80):
        self.engine, self.n = engine, n_clients
        h = C.c_void_p()
        rc = lib().dint_clients_create(engine.h, n_clients, seed, n_keys, zipf_theta, read_pct, C.byref(h))
        if rc != 0:
            raise DintError(rc, "dint_clients_create")
        self.h = h

    def run(self, rounds, stream=None):
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        rc = lib().dint_clients_run(self.h, rounds, C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise DintError(rc, "dint_clients_run")

    def stats(self):
        out = (C.c_uint64 * 5)()
        rc = lib().dint_clients_stats(self.h, out)
        if rc != 0:
            raise DintError(rc, "dint_clients_stats")
        return dict(zip(["requests", "committed", "validation_aborts", "lock_rejects", "rounds"], [int(x) for x in out]))

    def peek(self):
        rq = np.empty(self.n * 9, dtype=np.uint8)
        rs = np.empty(self.n * 9, dtype=np.uint8)
        rc = lib().dint_clients_peek(self.h, rq.ctypes.data, rs.ctypes.data)
        if rc != 0:
            raise DintError(rc, "dint_clients_peek")
        return rq, rs

    def close(self):
        if getattr(self, "h", None):
            lib().dint_clients_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GpuTxnClients:
    """TATP / SmallBank closed-loop clients resident on the GPU, driving the shard engines `engines` (engine i = shard i,
    all of one kind, on one device) -- dint_txn_clients_*.  Same clients, draw for draw, as
    dint_b200.txn_workloads.TxnWorkload(kind, n_clients, len(engines), subscribers, gid0)."""

    def __init__(self, engines, n_clients, subscribers=None, gid0=0):
        from .wire import TATP
        self.engines = list(engines)
        self.kind, self.msg = self.engines[0].kind, self.engines[0].msg
        if subscribers is None:
            subscribers = 7_000_000 if self.kind == TATP else 24_000_000
        arr = (C.c_void_p * len(self.engines))(*[e.h.value for e in self.engines])
        h = C.c_void_p()
        rc = lib().dint_txn_clients_create(arr, len(self.engines), n_clients, gid0, subscribers, C.byref(h))
        if rc != 0:
            raise DintError(rc, "dint_txn_clients_create")
        self.h = h

    def run(self, rounds, stream=None):
        """`rounds` closed-loop rounds on `stream` (default: the current torch stream); returns when the last round's
        requests are written (one host sync per round)."""
        if stream is None:
            import torch
            stream = torch.cuda.current_stream().cuda_stream
        rc = lib().dint_txn_clients_run(self.h, rounds, C.c_void_p(stream) if stream else None)
        if rc != 0:
            raise DintError(rc, "dint_txn_clients_run")

    def stats(self):
        """The dict TxnWorkload.stats() returns: requests, txns, committed, rounds, by_type {name: (begun, committed)}."""
        from .txn_workloads import stats_dict
        out = (C.c_uint64 * 18)()
        rc = lib().dint_txn_clients_stats(self.h, out)
        if rc != 0:
            raise DintError(rc, "dint_txn_clients_stats")
        return stats_dict(self.kind, out)

    def peek(self):
        """(requests uint8 [n * msg], destination shard uint8 [n], last round's replies uint8 [m * msg]) in client order:
        what TxnWorkload.next() returns for the pending round, and what was fed for the last one."""
        n = (C.c_uint64 * 2)()
        rc = lib().dint_txn_clients_peek(self.h, None, None, None, n)
        if rc != 0:
            raise DintError(rc, "dint_txn_clients_peek")
        rq = np.empty(max(int(n[0]), 1) * self.msg, dtype=np.uint8)
        dst = np.empty(max(int(n[0]), 1), dtype=np.uint8)
        rs = np.empty(max(int(n[1]), 1) * self.msg, dtype=np.uint8)
        rc = lib().dint_txn_clients_peek(self.h, rq.ctypes.data, dst.ctypes.data, rs.ctypes.data, n)
        if rc != 0:
            raise DintError(rc, "dint_txn_clients_peek")
        return rq[: int(n[0]) * self.msg], dst[: int(n[0])], rs[: int(n[1]) * self.msg]

    def close(self):
        if getattr(self, "h", None):
            lib().dint_txn_clients_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GpuCluster:
    """G shard engines driven by ONE process (dint_cluster_*): the C-level multi-GPU server.  devices: CUDA ordinals,
    all distinct (NVLink peer access) or all the same (several shards resident on one GPU)."""

    def __init__(self, kind, n_shards, devices=None, max_batch=0, populate=False, **cfg_over):
        self.kind, self.msg, self.G = kind, MSG_SIZE[kind], n_shards
        cfg = self.cfg = default_cfg(kind, **cfg_over)
        dv = (C.c_int * n_shards)(*devices) if devices is not None else None
        h = C.c_void_p()
        rc = lib().dint_cluster_create(kind, C.byref(cfg), n_shards, dv, max_batch, C.byref(h))
        if rc != 0:
            raise DintError(rc, f"dint_cluster_create({KIND_NAMES[kind]}, {n_shards})")
        self.h = h
        if populate:
            rc = lib().dint_cluster_populate(self.h)
            if rc != 0:
                raise DintError(rc, "dint_cluster_populate")

    def submit(self, req, dst=None, out=None, check=True):
        raw = np.ascontiguousarray(req).view(np.uint8).reshape(-1)
        n = raw.size // self.msg
        if out is None:
            out = np.empty_like(raw)
        d = None if dst is None else np.ascontiguousarray(dst, dtype=np.uint8)
        rc = lib().dint_cluster_submit(self.h, raw.ctypes.data, n, None if d is None else d.ctypes.data, out.ctypes.data)
        if rc != 0 and (check or rc != DINT_EPROTO):
            raise DintError(rc, "dint_cluster_submit")
        return out

    def overflow_retries(self):
        return int(lib().dint_cluster_overflow_retries(self.h))

    def engine(self, shard):
        """A non-owning Engine view of one shard (state inspection)."""
        e = Engine.__new__(Engine)
        e.kind, e.msg, e.device, e.cfg = self.kind, self.msg, None, self.cfg
        e.h = C.c_void_p(lib().dint_cluster_engine(self.h, shard))
        e.close = lambda: None
        return e

    def close(self):
        if getattr(self, "h", None):
            lib().dint_cluster_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
