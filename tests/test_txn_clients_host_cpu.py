"""No GPU: the host TATP / SmallBank clients (txn_workloads.cc around the state machines of txn_clients.h) driving three
oracle shard servers reproduce the request stream shard 0 received in tools/make_golden.py's closed loops, whose replies
came from the unmodified reference servers.  This pins the state machines the device driver shares to the reference."""
import os

import numpy as np
import pytest

import oracle_lib as O
from dint_b200 import wire
from dint_b200.txn_workloads import Cluster, TxnWorkload
from golden_util import first_diff

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("kind,name,n,clients,rounds,cfg", [
    (wire.TATP, "tatp_closed_shard0", 400, 150, 60, {"subs_populate": 400}),
    (wire.SMALLBANK, "smallbank_closed_shard0", 3000, 300, 60, {"accts_populate": 3000})], ids=["tatp", "smallbank"])
def test_host_clients_reproduce_the_recorded_shard0_stream(kind, name, n, clients, rounds, cfg):
    msg = wire.MSG_SIZE[kind]
    want = np.load(os.path.join(GOLDEN, name + ".npz"))["req"]
    oras = [O.Oracle(kind, **cfg) for _ in range(3)]
    wl = TxnWorkload(kind, n_clients=clients, n_shards=3, subscribers=n)
    cl = Cluster([o.process for o in oras], msg)
    shard0 = []
    for _ in range(rounds):
        rq, dst = wl.next()
        shard0.append(rq.reshape(-1, msg)[dst == 0].reshape(-1).copy())
        wl.feed(cl.submit(rq, dst))
    got = np.concatenate(shard0)
    assert got.size == want.size, (got.size // msg, want.size // msg)
    assert first_diff(got, want, msg) is None, first_diff(got, want, msg)
    assert wl.stats()["committed"] > 0
