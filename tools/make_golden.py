#!/usr/bin/env python
"""Generate tests/golden/*.npz from the UNMODIFIED reference servers (oracle/_ref, built in place from
/root/reference by `make -C oracle ref`).  Run in the build container only; the fixtures are committed.

Each fixture = {req: uint8[n*msg], resp: uint8[n*msg] as produced by `<server> 1` under the replay shim,
kind, cfg: the oracle/engine configuration under which the same replies must come out}.  KV traces only
touch subscribers / accounts below a small prefix N of the reference population, so that the oracle and
the engine can reproduce them with subs_populate = N (the reference's population streams are sequential
in s_id) while the table SIZING (hash sizes, lock-hash moduli) stays the reference's.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import golden_util as G         # noqa: E402
import oracle_lib as O          # noqa: E402
import trace_gen as T           # noqa: E402
from dint_b200 import wire      # noqa: E402
from dint_b200.workloads import Workload, record_trace, REF, HOT   # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def save(name, kind, req, cfg):
    ref, stats = O.run_ref(kind, req)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), req=req, resp=ref, kind=kind,
                        cfg_keys=np.array(list(cfg.keys())), cfg_vals=np.array(list(cfg.values()), dtype=np.int64))
    print(f"{name}: {req.size // wire.MSG_SIZE[kind]} requests, reference ran {stats['seconds']:.3f} s")


def closed_loop(kind, fam, clients, rounds, seed, **wl_kw):
    ora = O.Oracle(kind, **wl_kw.pop("oracle_cfg", {}))
    wl = Workload(kind, n_clients=clients, seed=seed, **fam, **wl_kw)
    req, _ = record_trace(wl, ora.process, rounds)
    return req


def main():
    os.makedirs(OUT, exist_ok=True)
    O.build_oracle(ref=True)
    assert O.ref_available(), "oracle/_ref is not built (is /root/reference mounted?)"
    # lock_fasst
    save("fasst_ref_closed", wire.FASST, closed_loop(wire.FASST, REF, 256, 40, 20230), {})
    save("fasst_hot_closed", wire.FASST, closed_loop(wire.FASST, HOT, 256, 40, 20231), {})
    save("fasst_random_collide", wire.FASST, T.fasst_random(8000, 40, seed=1), {})
    # lock_2pl
    save("lock2pl_ref_closed", wire.LOCK2PL, closed_loop(wire.LOCK2PL, REF, 256, 40, 20232), {})
    save("lock2pl_hot_closed", wire.LOCK2PL, closed_loop(wire.LOCK2PL, HOT, 256, 40, 20233), {})
    save("lock2pl_random_wrap", wire.LOCK2PL, T.lock2pl_random(8000, 25, seed=2), {})
    # log_server
    save("log_random", wire.LOG, T.log_random(3000, seed=3), {})
    # store: reads (hit + miss) and sets over the first 500 subscribers; closed-loop contention trace
    save("store_random", wire.STORE, T.store_random(4000, 500, seed=4), {"subs_populate": 500})
    # smallbank
    save("smallbank_random", wire.SMALLBANK, T.smallbank_random(8000, 200, seed=5), {"accts_populate": 200})
    # tatp: population sweep (every candidate key of the first 60 subscribers) + random valid traffic
    ora = O.Oracle(wire.TATP, subs_populate=60)
    u = T.tatp_key_universe(60)
    rd = np.zeros(len(u), dtype=wire.MSG_DTYPE[wire.TATP])
    rd["table"] = [x[0] for x in u]
    rd["key"] = [x[1] for x in u]
    req = np.concatenate([wire.as_bytes(rd), T.tatp_random(5000, 60, seed=6, oracle=ora)])
    save("tatp_sweep_random", wire.TATP, req, {"subs_populate": 60})
    # closed-loop transaction drivers (tatp 7 txn types / smallbank 6), 3 shards: the request stream shard 0 saw
    from dint_b200.txn_workloads import TxnWorkload, Cluster
    for kind, name, n, clients, rounds, cfg in [
            (wire.TATP, "tatp_closed_shard0", 400, 150, 60, {"subs_populate": 400}),
            (wire.SMALLBANK, "smallbank_closed_shard0", 3000, 300, 60, {"accts_populate": 3000})]:
        oras = [O.Oracle(kind, **cfg) for _ in range(3)]
        wl = TxnWorkload(kind, n_clients=clients, n_shards=3, subscribers=n)
        cl = Cluster([o.process for o in oras], wire.MSG_SIZE[kind])
        shard0 = []
        for _ in range(rounds):
            rq, dst = wl.next()
            shard0.append(rq.reshape(-1, wire.MSG_SIZE[kind])[dst == 0].reshape(-1).copy())
            wl.feed(cl.submit(rq, dst))
        save(name, kind, np.concatenate(shard0), cfg)
    # seeded trace_gen traces, replies only (golden_util.TRACES)
    for name, (kind, make) in G.TRACES.items():
        req = make()
        G.save_trace(name, req, O.run_ref(kind, req)[0])
        print(f"trace_gen/{name}: {req.size // wire.MSG_SIZE[kind]} requests")


if __name__ == "__main__":
    main()
