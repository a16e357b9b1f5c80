"""-m gpu (ONE GPU is enough): the C-level multi-GPU server (dint_cluster_*, include/dint_b200.h) with all its shards
resident on device 0 -- shard-local indexing (slot / G), dispatch -> engines -> combine through the return buffers,
the host slice ring -- against ONE sequential oracle (lock kinds, store: SURVEY.md 8(e) "owner = slot % G") or against
G oracle shard servers (tatp / smallbank: the reference's placement, tatp/caladan/client_udp_shard.cc:187,490-531).
On a multi-GPU box the same tests also run with one shard per device (NVLink peer memory)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as O
import trace_gen as T
from dint_b200 import GpuCluster, wire
from golden_util import first_diff

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_gpus():
    import torch
    return torch.cuda.device_count()


def _placements(G):
    """shards all on device 0; plus one shard per device when the box has enough GPUs"""
    out = [("one_device", [0] * G)]
    if G > 1 and _n_gpus() >= G:
        out.append(("per_device", list(range(G))))
    return out


def _trace(kind, n, seed, skew=False):
    if kind == wire.FASST:
        return T.fasst_random(n, 4800 if skew else 60000, seed=seed), {}
    if kind == wire.LOCK2PL:
        return T.lock2pl_random(n, 3000 if skew else 50000, seed=seed), {}
    return T.store_random(n, 500, seed=seed), dict(subs_populate=500)


@pytest.mark.parametrize("G", [1, 2, 3, 8])
@pytest.mark.parametrize("kind", [wire.FASST, wire.LOCK2PL, wire.STORE])
def test_cluster_answers_like_one_server(kind, G):
    msg = wire.MSG_SIZE[kind]
    max_batch = 4096
    sizes = [1, G - 1 if G > 1 else 1, 777, G * max_batch, 3 * G * max_batch + 129, 50000]
    for name, devs in _placements(G):
        _, cfg = _trace(kind, 1, 0)
        ora = O.Oracle(kind, **cfg)
        with GpuCluster(kind, G, devices=devs, max_batch=max_batch, populate=True, **cfg) as cl:
            for i, n in enumerate(sizes):
                req, _ = _trace(kind, n, seed=100 + i, skew=(i % 2 == 1))
                want = ora.process(req)
                got = cl.submit(req)
                d = first_diff(got, want, msg)
                assert d is None, f"{name} G={G} call {i} (n={n}): {d}"
            # final state: a sample of slots / keys, asked of the shard that owns them
            rng = np.random.default_rng(7)
            if kind in (wire.FASST, wire.LOCK2PL):
                for lid in rng.integers(0, 3000, size=64):
                    slot = ora.lock_slot(0, int(lid))
                    assert cl.engine(slot % G).lock_state(0, slot) == ora.lock_state(0, slot)
            else:
                tot = sum(cl.engine(s).kv_count(0) for s in range(G))
                assert tot == ora.kv_count(0)


@pytest.mark.parametrize("G", [2, 8])
def test_cluster_survives_keys_that_all_hash_to_one_shard(G):
    """The exchange slabs hold mean + 25 % + 8 sigma records per (source, owner).  A batch whose keys all belong to ONE
    shard does not fit: the sources flag it, no shard serves that round (nor anything behind it), and the cluster serves
    it again in rounds that cannot overflow -- the replies must still be ONE sequential server's."""
    max_batch = 4096
    rng = np.random.default_rng(3)
    ora = O.Oracle(wire.FASST)
    with GpuCluster(wire.FASST, G, devices=[0] * G, max_batch=max_batch) as cl:
        calls = [T.fasst_random(2 * G * max_batch, 50000, seed=1),          # ordinary traffic
                 T.fasst_random(3 * G * max_batch + 77, 1, seed=2),         # every record on lock id 0
                 T.fasst_random(G * max_batch, 2, seed=3),                  # two ids
                 T.fasst_random(2 * G * max_batch, 50000, seed=4)]          # ordinary traffic again
        for i, req in enumerate(calls):
            want = ora.process(req)
            got = cl.submit(req)
            d = first_diff(got, want, 9)
            assert d is None, f"call {i}: {d}"
        assert cl.overflow_retries() >= 1


@pytest.mark.parametrize("kind,n,clients,G", [(wire.TATP, 3000, 1500, 3), (wire.TATP, 2500, 1200, 5),
                                              (wire.SMALLBANK, 5000, 1500, 3), (wire.SMALLBANK, 4000, 1000, 8)])
def test_cluster_serves_client_chosen_shards(kind, n, clients, G):
    """tatp / smallbank full transaction mixes, closed loop: the cluster must take the same commit / abort decisions,
    reply for reply, as G oracle shard servers (each holding the whole population, as the reference's do)."""
    from dint_b200.txn_workloads import TxnWorkload, Cluster
    cfg = dict(subs_populate=n) if kind == wire.TATP else dict(accts_populate=n)
    msg = wire.MSG_SIZE[kind]
    rounds = 60

    def run(submit):
        wl = TxnWorkload(kind, n_clients=clients, n_shards=G, subscribers=n)
        trace = []
        for _ in range(rounds):
            rq, dst = wl.next()
            rs = submit(rq, dst)
            wl.feed(rs)
            trace.append((rq.copy(), dst.copy(), np.array(rs, copy=True)))
        return trace, wl.stats()

    oras = [O.Oracle(kind, **cfg) for _ in range(G)]
    want, st_want = run(Cluster([o.process for o in oras], msg).submit)
    for name, devs in _placements(G):
        with GpuCluster(kind, G, devices=devs, max_batch=2048, populate=True, **cfg) as cl:
            got, st_got = run(lambda rq, dst: cl.submit(rq, dst))
            for r, ((q1, d1, s1), (q2, d2, s2)) in enumerate(zip(want, got)):
                assert np.array_equal(q1, q2) and np.array_equal(d1, d2), f"{name} round {r}: clients diverged"
                assert first_diff(s2, s1, msg) is None, f"{name} round {r}: {first_diff(s2, s1, msg)}"
            assert st_got == st_want and st_got["committed"] > 0
            for s in range(G):
                ring, appended = cl.engine(s).dump_log()
                assert appended == oras[s].log_appended() and np.array_equal(ring, oras[s].log_ring())
                if G == 3:                      # G > 3: a shard holds only the keys it is a replica of
                    for tb in range(5 if kind == wire.TATP else 2):
                        assert cl.engine(s).kv_count(tb) == oras[s].kv_count(tb)


def test_cluster_from_c():
    """A plain C caller (gcc, no Python, no torch): tests/c/cluster_check.c links libdint_b200.so and the oracle and
    compares dint_cluster_submit with ONE sequential server for lock_fasst (3 shards) and with 3 shard servers for
    smallbank -- the call sequence a C/C++ transport front-end makes (INTEGRATION.md).  The program is built in a
    temporary directory, so the test writes nothing into the source tree (which may be read-only or another user's)."""
    import tempfile
    from dint_b200 import _build
    src = os.path.join(ROOT, "tests", "c", "cluster_check.c")
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "cluster_check")
        subprocess.run(["gcc", "-O2", "-Wall", "-o", exe, src, "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "oracle"),
                        "-L" + _build.LIBDIR, "-ldint_b200", "-L" + os.path.join(ROOT, "oracle"), "-ldint_oracle",
                        "-Wl,-rpath," + _build.LIBDIR, "-Wl,-rpath," + os.path.join(ROOT, "oracle")], check=True)
        r = subprocess.run([exe], capture_output=True, timeout=300)
    sys.stdout.write(r.stdout.decode())
    assert r.returncode == 0, r.stdout.decode() + r.stderr.decode()
    assert b"cluster_check: OK" in r.stdout
