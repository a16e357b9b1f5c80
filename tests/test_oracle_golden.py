"""CPU tests: the oracle restatement (oracle/dint_oracle.c) against (a) the fasthash64 known-answer
table of SURVEY.md section 8(c), (b) the golden fixtures produced by the unmodified reference servers,
(c) the reference servers' recorded replies to seeded trace_gen.py traces; and, when oracle/_ref is
built, the unmodified reference server over loopback UDP."""
import os
import struct

import numpy as np
import pytest

import golden_util as G
import oracle_lib as O
import trace_gen as T
from dint_b200 import wire
from dint_b200.workloads import Workload, record_trace, REF, HOT

KAT = {  # (value, len) -> fasthash64(value, len, 0xdeadbeef); computed from lock_2pl/udp/utils.h
    (0, 4): 0xF1D9C3BC57488240, (1, 4): 0x2C13B74111C1F7E9, (7, 4): 0x90F120682C7CDD84,
    (9, 4): 0xA939C800026596A0, (4799, 4): 0x53250DB90DEF10A4, (23999999, 4): 0xB1CD0960FFA82E06,
    (0xFFFFFFFF, 4): 0x16BB2C2D42413085, (0, 8): 0x16C38EE185750EBC, (1, 8): 0xD7C65C9D6F0F512E,
    (7, 8): 0x3E1A03400272CDC3, (0x0000080100000005, 8): 0xA084F51D4BC4FB1A, (23999999, 8): 0x818C5A0000875647,
}
KAT_MOD = {(0, 4, 36000000): 28482624, (1, 4, 36000000): 33013481, (0xFFFFFFFF, 4, 36000000): 24026245,
           (0, 8, 9000000): 4819516, (0, 8, 36000000): 22819516, (0x0000080100000005, 8, 9000000): 4333594,
           (23999999, 8, 9000000): 5564871}


def test_fasthash_known_answers():
    for (x, ln), h in KAT.items():
        assert O.fasthash64(struct.pack("<I" if ln == 4 else "<Q", x)) == h
    for (x, ln, m), r in KAT_MOD.items():
        assert O.fasthash64(struct.pack("<I" if ln == 4 else "<Q", x)) % m == r


def test_fasthash_odd_lengths_follow_tail_switch():
    # lengths 1..7 and 9..15 exercise the fall-through tail (utils.h:44-54); cross-check with a
    # direct Python transcription of the published fasthash64
    def mix(h):
        h ^= h >> 23
        h = (h * 0x2127599BF4325C37) & (2**64 - 1)
        return h ^ (h >> 47)

    def ref(buf, seed=0xDEADBEEF):
        m = 0x880355F21E6D1965
        h = seed ^ ((len(buf) * m) & (2**64 - 1))
        nw = len(buf) // 8
        for i in range(nw):
            h ^= mix(int.from_bytes(buf[8 * i:8 * i + 8], "little"))
            h = (h * m) & (2**64 - 1)
        tail = buf[8 * nw:]
        if tail:
            h ^= mix(int.from_bytes(tail, "little"))
            h = (h * m) & (2**64 - 1)
        return mix(h)

    rng = np.random.default_rng(0)
    for ln in range(0, 24):
        b = rng.integers(0, 256, size=ln, dtype=np.uint8).tobytes()
        assert O.fasthash64(b) == ref(b)


@pytest.mark.parametrize("name", G.names())
def test_oracle_reproduces_reference_golden(name):
    kind, req, resp, cfg = G.load(name)
    ora = O.Oracle(kind, **cfg)
    ours = ora.process(req)
    assert G.mismatch(kind, ours, resp) is None, G.mismatch(kind, ours, resp)


def test_golden_fixtures_cover_every_server_kind():
    kinds = {G.load(n)[0] for n in G.names()}
    assert kinds == set(range(6))


def test_sequential_semantics_examples():
    """The survey's 7-request lock_fasst script (SURVEY.md section 8(c)) and its lock_2pl analogue."""
    rec = np.zeros(7, dtype=wire.MSG_DTYPE[wire.FASST])
    rec["type"] = [0, 1, 1, 3, 0, 2, 1]
    rec["lid"] = [9, 9, 9, 9, 9, 9, 7]
    out = wire.as_records(wire.FASST, O.Oracle(wire.FASST).process(wire.as_bytes(rec)))
    assert out["type"].tolist() == [4, 5, 6, 8, 4, 7, 5]
    assert out["ver"].tolist() == [0, 0, 0, 0, 1, 0, 0]
    rec = np.zeros(6, dtype=wire.MSG_DTYPE[wire.LOCK2PL])
    rec["action"] = [0, 0, 0, 1, 1, 0]
    rec["type"] = [0, 1, 0, 0, 0, 1]
    rec["lid"] = 5
    ora = O.Oracle(wire.LOCK2PL)
    out = wire.as_records(wire.LOCK2PL, ora.process(wire.as_bytes(rec)))
    assert out["action"].tolist() == [2, 3, 2, 5, 5, 2]      # S grant, X reject, S grant, rel, rel, X grant
    assert ora.lock_state(0, ora.lock_slot(0, 5)) == (1, 0)


def test_release_without_hold_wraps_like_the_reference():
    rec = np.zeros(2, dtype=wire.MSG_DTYPE[wire.LOCK2PL])
    rec["action"] = [1, 0]
    rec["type"] = [1, 0]
    rec["lid"] = 3
    ora = O.Oracle(wire.LOCK2PL)
    out = wire.as_records(wire.LOCK2PL, ora.process(wire.as_bytes(rec)))
    assert out["action"].tolist() == [5, 3]                  # num_ex wrapped to 0xffffffff -> S rejected
    assert ora.lock_state(0, ora.lock_slot(0, 3)) == (0xFFFFFFFF, 0)


def test_workload_drivers_are_deterministic_and_valid():
    for kind, fam in [(wire.FASST, REF), (wire.FASST, HOT), (wire.LOCK2PL, REF), (wire.LOCK2PL, HOT),
                      (wire.LOG, {}), (wire.STORE, dict(set_pct=50))]:
        runs = []
        for _ in range(2):
            ora = O.Oracle(kind, subs_populate=2000) if kind == wire.STORE else O.Oracle(kind)
            wl = Workload(kind, n_clients=128, seed=42, **({"store_subscribers": 2000} if kind == wire.STORE else {}), **fam)
            runs.append(record_trace(wl, ora.process, 30) + (wl.stats(),))
        assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])
        st = runs[0][2]
        assert st["requests"] == 128 * 30 and st["committed"] > 0


@pytest.mark.parametrize("name", sorted(G.TRACES))
def test_oracle_matches_recorded_reference_replies(name):
    kind, req, ref = G.load_trace(name)
    assert G.first_diff(O.Oracle(kind).process(req), ref, wire.MSG_SIZE[kind]) is None


def test_txn_drivers_run_valid_protocols_against_oracle_shards():
    """The TATP / SmallBank client state machines never send a request the reference would panic() on
    (kvs_set / kvs_delete of a missing row, unknown type), commit a sane share of transactions, and are
    deterministic."""
    from dint_b200.txn_workloads import TxnWorkload, Cluster
    for kind, n, cfg in [(wire.TATP, 2000, dict(subs_populate=2000)), (wire.SMALLBANK, 4000, dict(accts_populate=4000))]:
        runs = []
        for _ in range(2):
            oras = [O.Oracle(kind, **cfg) for _ in range(3)]
            wl = TxnWorkload(kind, n_clients=400, n_shards=3, subscribers=n)
            cl = Cluster([o.process for o in oras], wire.MSG_SIZE[kind])
            h = 0
            for _ in range(100):
                rq, dst = wl.next()
                rs = cl.submit(rq, dst)          # raises if an oracle shard hits a panic() path
                wl.feed(rs)
                h = hash((h, rs.tobytes()))
            runs.append((h, wl.stats()))
        assert runs[0] == runs[1]
        st = runs[0][1]
        assert st["committed"] > 0.2 * st["txns"]
        assert all(v[0] > 0 for v in st["by_type"].values())


@pytest.mark.skipif(not (O.ref_available() and os.path.exists(os.path.join(O.REF_DIR, "udp_blast"))),
                    reason="oracle/_ref not built (no /root/reference here)")
def test_reference_server_answers_over_loopback_udp():
    """The "as shipped" CPU baseline harness (oracle/udp_shim.c + udp_blast.c): the unmodified lock_fasst server
    with real sockets answers every datagram it is sent."""
    req = T.fasst_random(20000, 10**6, seed=2)
    try:
        r = O.run_ref_udp(O.FASST, req, server_threads=2, client_threads=2, window=8, seconds=1.0)
    except (OSError, RuntimeError) as ex:      # no loopback sockets in this sandbox
        pytest.skip(repr(ex))
    assert r["replies"] > 1000 and r["lost"] <= r["replies"] // 100
