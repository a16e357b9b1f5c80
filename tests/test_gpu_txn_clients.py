"""-m gpu (one GPU): the TATP / SmallBank closed-loop clients resident on the GPU (dint_b200/csrc/txn_clients.cuh,
dint_txn_clients_*) must, round for round, put on the wire what the host clients (txn_workloads.cc, the same state machines
of txn_clients.h) put there, take the same decisions on the replies, and leave every shard in its oracle's state."""
import os

import numpy as np
import pytest

import oracle_lib as O
import trace_gen as T
from dint_b200 import DintError, Engine, GpuTxnClients, wire
from dint_b200.txn_workloads import Cluster, TxnWorkload
from golden_util import first_diff

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
_seen = {wire.TATP: {}, wire.SMALLBANK: {}}       # by_type totals over the parity cases, per kind


def _cfg(kind, n):
    return dict(subs_populate=n) if kind == wire.TATP else dict(accts_populate=n)


def _engines(kind, G, n, **over):
    place = [dict(txn_shards=G, txn_shard_id=i) if G > 3 else {} for i in range(G)]
    return [Engine(kind, populate=True, chunk=4096, **_cfg(kind, n), **place[i], **over) for i in range(G)]


def _populated_keys(kind, n):
    if kind == wire.TATP:
        return T.tatp_key_universe(n)
    return [(tb, k) for tb in (0, 1) for k in range(n)]


def _run_against_host(kind, G, n, clients, rounds, gid0=0, oracle=True):
    """Drive GpuTxnClients and TxnWorkload side by side.  oracle=False: the host clients are fed the GPU's replies."""
    msg = wire.MSG_SIZE[kind]
    engs = _engines(kind, G, n)
    oras = [O.Oracle(kind, **_cfg(kind, n)) for _ in range(G)] if oracle else None
    cl = Cluster([o.process for o in oras], msg) if oracle else None
    wl = TxnWorkload(kind, n_clients=clients, n_shards=G, subscribers=n, gid0=gid0)
    with GpuTxnClients(engs, clients, subscribers=n, gid0=gid0) as gc:
        for r in range(rounds):
            want_rq, want_dst = wl.next()
            got_rq, got_dst, _ = gc.peek()
            assert got_dst.size == want_dst.size, f"round {r}: {got_dst.size} records, host {want_dst.size}"
            assert np.array_equal(got_dst, want_dst), f"round {r}: destination shards differ"
            assert first_diff(got_rq, want_rq, msg) is None, f"round {r}: requests differ: {first_diff(got_rq, want_rq, msg)}"
            gc.run(1)
            _, _, got_rs = gc.peek()
            if oracle:
                want_rs = cl.submit(want_rq, want_dst)
                assert first_diff(got_rs, want_rs, msg) is None, f"round {r}: replies differ: {first_diff(got_rs, want_rs, msg)}"
            wl.feed(want_rs if oracle else got_rs)
        st = gc.stats()
        assert st == wl.stats(), (st, wl.stats())
        assert st["rounds"] == rounds and st["committed"] > 0
    if oracle:
        for s in range(G):
            ring, appended = engs[s].dump_log()
            assert appended == oras[s].log_appended() and np.array_equal(ring, oras[s].log_ring()), f"shard {s}: log differs"
            if G <= 3:                       # G > 3: a shard holds only the keys it is a replica of
                for tb in range(5 if kind == wire.TATP else 2):
                    assert engs[s].kv_count(tb) == oras[s].kv_count(tb), f"shard {s} table {tb}: kv_count"
            if G == 3:
                for tb, key in _populated_keys(kind, n):
                    assert engs[s].kv_get(tb, key) == oras[s].kv_get(tb, key), f"shard {s} table {tb} key {key:#x}"
    for e in engs:
        e.close()
    for name, (b, c) in st["by_type"].items():
        acc = _seen[kind].setdefault(name, [0, 0, 0])
        acc[0] += b
        acc[1] += c
        acc[2] += max(0, b - c - clients)  # transactions that certainly aborted: at most `clients` are still in flight
    return st


@pytest.mark.parametrize("G,n,clients,rounds", [(3, 3000, 1500, 120), (5, 2500, 1200, 100), (3, 50, 1000, 150)],
                         ids=["G3", "G5", "hot_50_subscribers"])
def test_tatp_gpu_clients_match_host_clients_and_oracle_shards(G, n, clients, rounds):
    _run_against_host(wire.TATP, G, n, clients, rounds, gid0=11)


def test_tatp_gpu_clients_match_host_clients_on_one_shard():
    """G = 1 sends both backups' DELETE_BCK to the one server; the reference server panics on the second (kvs_delete of
    a missing key), so there is no oracle for this deployment.  The host clients are fed the engine's replies: the
    clients must still agree round for round."""
    _run_against_host(wire.TATP, 1, 2000, 1500, 100, oracle=False)


@pytest.mark.parametrize("G,n,clients,rounds", [(1, 5000, 1500, 100), (3, 5000, 1500, 120), (8, 4000, 1000, 100),
                                                (3, 100, 1000, 150)],
                         ids=["G1", "G3", "G8", "hot_100_accounts"])
def test_smallbank_gpu_clients_match_host_clients_and_oracle_shards(G, n, clients, rounds):
    _run_against_host(wire.SMALLBANK, G, n, clients, rounds, gid0=5)


def test_every_transaction_type_commits_and_aborts():
    """Over the parity cases above: every type of both mixes committed, and aborted, at least once -- except
    get_subscriber_data, which has no abort path (one read, then commit: tatp/caladan/client_udp_shard.cc:177-199)."""
    if len(_seen[wire.TATP]) < 7 or len(_seen[wire.SMALLBANK]) < 6:
        pytest.skip("needs the parity cases of this module to have run")
    for kind, seen in _seen.items():
        for name, (begun, committed, aborted_lb) in seen.items():
            assert committed > 0, f"{name} never committed"
            if name != "get_subscriber_data":
                assert aborted_lb > 0, f"{name} never certainly aborted ({begun} begun, {committed} committed)"


@pytest.mark.parametrize("kind,name,n,clients,rounds", [(wire.TATP, "tatp_closed_shard0", 400, 150, 60),
                                                        (wire.SMALLBANK, "smallbank_closed_shard0", 3000, 300, 60)],
                         ids=["tatp", "smallbank"])
def test_gpu_clients_reproduce_the_recorded_shard0_stream(kind, name, n, clients, rounds):
    """tools/make_golden.py's closed loops (3 shards), whose replies came from the unmodified reference servers: the
    requests shard 0 receives from the GPU clients are the recorded ones."""
    msg = wire.MSG_SIZE[kind]
    want = np.load(os.path.join(GOLDEN, name + ".npz"))["req"]
    engs = _engines(kind, 3, n)
    got = []
    with GpuTxnClients(engs, clients, subscribers=n) as gc:
        for _ in range(rounds):
            rq, dst, _ = gc.peek()
            got.append(rq.reshape(-1, msg)[dst == 0].reshape(-1).copy())
            gc.run(1)
    got = np.concatenate(got)
    assert got.size == want.size and first_diff(got, want, msg) is None, first_diff(got, want, msg)
    for e in engs:
        e.close()


@pytest.mark.parametrize("kind", [wire.TATP, wire.SMALLBANK], ids=["tatp", "smallbank"])
def test_run_k_rounds_equals_k_single_rounds(kind):
    n = 20000
    a_eng, b_eng = _engines(kind, 3, n), _engines(kind, 3, n)
    with GpuTxnClients(a_eng, 30000, subscribers=n) as a, GpuTxnClients(b_eng, 30000, subscribers=n) as b:
        a.run(40)
        for _ in range(40):
            b.run(1)
        assert a.stats() == b.stats() and a.stats()["committed"] > 0
        for x, y in zip(a.peek(), b.peek()):
            assert np.array_equal(x, y)
    for e in a_eng + b_eng:
        e.close()


def test_create_rejects_bad_configurations():
    with Engine(wire.TATP, subs_populate=100) as t0, Engine(wire.TATP, subs_populate=100) as t1, \
            Engine(wire.TATP, subs_populate=100) as t2, Engine(wire.SMALLBANK, accts_populate=100) as s0:
        with Engine(wire.FASST) as f:
            with pytest.raises(DintError):
                GpuTxnClients([f], 10, subscribers=100)                   # not tatp / smallbank
        with pytest.raises(DintError):
            GpuTxnClients([t0, t1, s0], 10, subscribers=100)              # mixed kinds
        with pytest.raises(DintError):
            GpuTxnClients([t0, t1], 10, subscribers=100)                  # 2 shards
        with pytest.raises(DintError):
            GpuTxnClients([t0, t1, t2, t0, t1, t2, t0, t1, t2], 10, subscribers=100)   # 9 shards
        with pytest.raises(DintError):
            GpuTxnClients([t0, t1, t2], 0, subscribers=100)               # no clients
        with pytest.raises(DintError):
            GpuTxnClients([t0, t1, t2], 10, subscribers=2)                # subscribers < 3
        with pytest.raises(DintError):
            GpuTxnClients([t0, t1, t2, t0], 10, subscribers=100)          # G > 3 without txn_shards / txn_shard_id
        four = [Engine(wire.TATP, subs_populate=100, txn_shards=4, txn_shard_id=i) for i in (0, 1, 3, 2)]
        with pytest.raises(DintError):
            GpuTxnClients(four, 10, subscribers=100)                      # engine 2 says it is shard 3
        GpuTxnClients([four[0], four[1], four[3], four[2]], 10, subscribers=100).close()   # in shard order: accepted
        for e in four:
            e.close()
        import torch
        if torch.cuda.device_count() > 1:
            with Engine(wire.TATP, device=1, subs_populate=100) as t_other:
                with pytest.raises(DintError):
                    GpuTxnClients([t0, t1, t_other], 10, subscribers=100)   # engines on two devices
