"""TATP (and SmallBank) closed-loop transaction drivers (libdint_wl.so, csrc/txn_workloads.cc) and the
G-shard "cluster" they talk to.

    wl = TxnWorkload(wire.TATP, n_clients=4096, n_shards=3, subscribers=7_000_000)
    cl = Cluster([Engine(wire.TATP, populate=True) for _ in range(3)])      # or oracles, for the tests
    for _ in range(rounds):
        req, dst = wl.next()              # variable number of wire records per round + destination shard
        wl.feed(cl.submit(req, dst))
"""
import ctypes as C

import numpy as np

from . import _build
from .wire import MSG_SIZE, TATP

_lib = None
TATP_TXN_NAMES = ["get_subscriber_data", "get_access_data", "get_new_destination", "update_subscriber_data",
                  "update_location", "insert_call_forwarding", "delete_call_forwarding"]
SMALLBANK_TXN_NAMES = ["amalgamate", "balance", "deposit_checking", "send_payment", "transact_saving", "write_check"]


def lib():
    global _lib
    if _lib is None:
        _build.build()
        L = C.CDLL(_build.WL_LIB)
        L.dint_txn_create.restype = C.c_void_p
        L.dint_txn_create.argtypes = [C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.dint_txn_destroy.argtypes = [C.c_void_p]
        L.dint_txn_max_round.restype = C.c_uint32
        L.dint_txn_max_round.argtypes = [C.c_void_p]
        L.dint_txn_next.restype = C.c_uint64
        L.dint_txn_next.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.dint_txn_feed.argtypes = [C.c_void_p, C.c_void_p]
        L.dint_txn_stats.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        _lib = L
    return _lib


class TxnWorkload:
    def __init__(self, kind, n_clients, n_shards=3, subscribers=None, gid0=0):
        """subscribers: kSubscriberNum (tatp, reference 7,000,000) or kAccountNum (smallbank, 24,000,000) of the
        key generators -- must match what the servers populated."""
        if subscribers is None:
            subscribers = 7_000_000 if kind == TATP else 24_000_000
        self.kind, self.msg, self.n_shards = kind, MSG_SIZE[kind], n_shards
        self.h = lib().dint_txn_create(kind, n_clients, gid0, n_shards, subscribers)
        if not self.h:
            raise RuntimeError("dint_txn_create failed")
        cap = lib().dint_txn_max_round(self.h)
        self._req = np.empty(cap * self.msg, dtype=np.uint8)
        self._dst = np.empty(cap, dtype=np.uint8)
        self._n = 0

    def close(self):
        if self.h:
            lib().dint_txn_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def next(self):
        """One round: (requests uint8 [n * msg], destination shard uint8 [n]) -- views, valid until the next call."""
        self._n = int(lib().dint_txn_next(self.h, self._req.ctypes.data, self._dst.ctypes.data))
        return self._req[: self._n * self.msg], self._dst[: self._n]

    def feed(self, resp):
        resp = np.ascontiguousarray(resp).view(np.uint8).reshape(-1)
        assert resp.size == self._n * self.msg
        lib().dint_txn_feed(self.h, resp.ctypes.data)

    def stats(self):
        out = (C.c_uint64 * 18)()
        lib().dint_txn_stats(self.h, out)
        return stats_dict(self.kind, out)


def stats_dict(kind, out):
    """The dint_txn_stats layout (18 counters) as a dict; by_type[name] = (begun, committed)."""
    d = {"requests": int(out[0]), "txns": int(out[1]), "committed": int(out[2]), "rounds": int(out[3])}
    names = TATP_TXN_NAMES if kind == TATP else SMALLBANK_TXN_NAMES
    d["by_type"] = {n: (int(out[4 + i]), int(out[11 + i])) for i, n in enumerate(names)}
    return d


def partition_by_shard(req, dst, n_shards, msg):
    """Stable partition of a round by destination shard: returns (order, counts, per-shard request arrays)."""
    order = np.argsort(dst, kind="stable")
    counts = np.bincount(dst, minlength=n_shards)[:n_shards]
    rows = np.ascontiguousarray(req).reshape(-1, msg)[order]
    parts, off = [], 0
    for c in counts:
        parts.append(rows[off:off + c].reshape(-1))
        off += c
    return order, counts, parts


class Cluster:
    """G independent shard servers (anything with .submit(req_bytes) -> resp_bytes): the reference's three
    `server_shard` processes.  Each shard sees its requests in trace order."""

    def __init__(self, servers, msg):
        self.servers, self.msg = servers, msg

    def submit(self, req, dst):
        order, counts, parts = partition_by_shard(req, dst, len(self.servers), self.msg)
        outs = [np.asarray(s(p)).reshape(-1) if p.size else p for s, p in zip(self.servers, parts)]
        merged = np.concatenate(outs).reshape(-1, self.msg)
        out = np.empty_like(merged)
        out[order] = merged
        return out.reshape(-1)
