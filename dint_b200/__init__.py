"""dint_b200 -- B200-resident batched implementation of DINT's per-request server hot path.

    from dint_b200 import Engine, wire
    eng = Engine(wire.FASST)            # stands in for `lock_fasst/udp/server 1`
    resp = eng.submit(requests)         # packed wire structs in, packed wire structs out
"""
from . import wire
from .engine import Engine, GpuCluster, GpuClients, GpuTxnClients, PinnedBuffer, DintError, default_cfg, lib

__all__ = ["Engine", "GpuCluster", "GpuClients", "GpuTxnClients", "PinnedBuffer", "DintError", "default_cfg", "lib", "wire"]
