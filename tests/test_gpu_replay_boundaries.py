"""-m gpu: the conflict-replay paths at their switch points, small group spaces, and state carried across chunks,
calls, streams and snapshots.

Every case compares the full reply stream with the oracle fed the same requests, compares the final state where the
API exposes it, and asserts the engine's `conflicted`, `max_run` and `fallback_chunks` equal tests/replay_model.py's
prediction: the counters are what shows that the intended replay path ran (test_replay_model_cpu.py shows, without
a GPU, that the traces have the shape they are named after)."""
import numpy as np
import pytest

import oracle_lib as O
import replay_model as M
import trace_gen as T
from dint_b200 import Engine, wire
from dint_b200.engine import DintError
from dint_b200.workloads import Workload, record_trace
from test_gpu_parity import first_diff

pytestmark = pytest.mark.gpu

KINDS = [wire.LOCK2PL, wire.FASST, wire.STORE, wire.TATP, wire.SMALLBANK]
IDS = [wire.KIND_NAMES[k] for k in KINDS]
VALSZ = {wire.STORE: 40, wire.TATP: 40, wire.SMALLBANK: 8}
MSG = wire.MSG_SIZE


def counters(eng):
    st = eng.stats()
    return dict(conflicted=st["conflicted"], max_run=st["max_run"], fallback_chunks=st["fallback_chunks"])


def expected(pr):
    return {k: pr[k] for k in ("conflicted", "max_run", "fallback_chunks")}


def probes(srv, kind, raw):
    """The server state the requests of `raw` can have touched: lock words / counters of their slots, KV rows,
    row counts and the commit log.  srv: an Engine or an oracle_lib.Oracle."""
    out = {}
    if kind != wire.LOG:
        mask, table, key = M.touches(kind, raw)
        pairs = sorted(set(zip(table[mask != 0].tolist(), key[mask != 0].tolist())))[:300]
        for t, k in pairs:
            if kind in (wire.LOCK2PL, wire.FASST, wire.TATP, wire.SMALLBANK):
                s = srv.lock_slot(t, k)
                ls = srv.lock_state(t, s)
                out["lock", t, s] = tuple(ls) if kind != wire.TATP else ls[0]
            if kind in VALSZ:
                r = srv.kv_get(t, k)
                out["kv", t, k] = None if r is None else (r[0][:VALSZ[kind]], r[1])
        for t in range({wire.STORE: 1, wire.TATP: 5, wire.SMALLBANK: 2}.get(kind, 0)):
            out["count", t] = int(srv.kv_count(t))
    if kind in (wire.LOG, wire.TATP, wire.SMALLBANK):
        if isinstance(srv, Engine):
            ring, appended = srv.dump_log()
        else:
            ring, appended = srv.log_ring(), srv.log_appended()
        out["log"] = (ring.tobytes(), int(appended))
    return out


def check_replies(got, want, msg, what):
    d = first_diff(np.asarray(got), np.asarray(want), msg)
    assert d is None, f"{what}: {d}"


# ---------------------------------------------------------------- (a) thresholds -------------------------------------
@pytest.mark.parametrize("chunk", [4096, 1 << 16])
@pytest.mark.parametrize("kind", KINDS, ids=IDS)
def test_replay_thresholds(kind, chunk):
    """A bucket at 128 / 129 listed pairs (bucket path / radix fallback), warp tasks of 32 / 33 / 128 / 129 pairs
    (rank sort / bitonic / one pass / bucket by bucket), two groups sharing a folded flag nibble, and a read-only chunk
    followed by a writer chunk on the same groups: replies, state and counters."""
    space, cfg, cases = M.threshold_cases(kind, chunk, seed=kind * 100 + chunk)
    kv = kind in VALSZ
    ora = O.Oracle(kind, populate=kv, **cfg)
    msg = wire.MSG_SIZE[kind]
    with Engine(kind, chunk=chunk, populate=kv, **cfg) as eng:
        for name, raw, _ in cases:
            eng.reset_stats()
            check_replies(eng.submit(raw), ora.process(raw), msg, name)
            want = expected(M.predict(space, [(raw, "host")]))
            assert counters(eng) == want, name
            if name == "bucket_129":
                assert want["fallback_chunks"] == 1 and want["max_run"] > 1
        every = np.concatenate([raw for _, raw, _ in cases])
        assert probes(eng, kind, every) == probes(ora, kind, every)


# ---------------------------------------------------------------- (b) small group spaces -----------------------------
LOCK_SLOTS = [1, 7, 256, 257, 65536, 65537, (1 << 24) + 1]


@pytest.mark.parametrize("slots", LOCK_SLOTS)
@pytest.mark.parametrize("kind", [wire.FASST, wire.LOCK2PL], ids=["lock_fasst", "lock_2pl"])
def test_small_lock_tables(kind, slots):
    """1 to 4 radix passes and the shrunken flag sets: a random trace in chunks of 4096 and a closed loop at the
    default chunk, both over more lock ids than slots."""
    n_keys = min(4 * slots + 64, 10**6)
    space = M.Space(kind, lock_slots=slots, chunk=4096)
    gen = T.fasst_random if kind == wire.FASST else T.lock2pl_random
    req = gen(40000, n_keys, seed=slots)
    rng = np.random.default_rng(slots)             # and one chunk that surely takes the radix fallback
    req = np.concatenate([req[:8 * 4096 * MSG[kind]], M.build_hot_bucket(space, M.default_pool(space, rng), 4096, rng)])
    pr = M.predict(space, [(req, "host")])
    assert pr["fallback_chunks"] >= 1
    ora = O.Oracle(kind, lock_slots=slots)
    want = ora.process(req)
    with Engine(kind, lock_slots=slots, chunk=4096) as eng:
        check_replies(eng.submit(req), want, eng.msg, "random trace")
        assert counters(eng) == expected(pr)
        assert probes(eng, kind, req) == probes(ora, kind, req)
    ora = O.Oracle(kind, lock_slots=slots)
    wl = Workload(kind, n_clients=2048, seed=slots, n_keys=4 * slots + 64, zipf_theta=0.5)
    req, want = record_trace(wl, ora.process, 20)
    with Engine(kind, lock_slots=slots) as eng:
        check_replies(eng.submit(req), want, eng.msg, "closed loop")
        assert counters(eng) == expected(M.predict(M.Space(kind, lock_slots=slots), [(req, "host")]))
        assert probes(eng, kind, req) == probes(ora, kind, req)


@pytest.mark.parametrize("kind,n", [(wire.FASST, 1 << 20), (wire.LOCK2PL, 1 << 18)], ids=["lock_fasst", "lock_2pl"])
def test_one_lock_slot_holds_the_whole_chunk(kind, n):
    """lock_slots = 1 at the default chunk: every request is in ONE run of the radix fallback (lock_fasst: the
    segmented scan, 2^20 requests; lock_2pl: one thread walks it)."""
    import torch
    space = M.Space(kind, lock_slots=1)
    rng = np.random.default_rng(11)
    req = M.build_one_group(space, M.default_pool(space, rng, n=16), n, rng)
    want = O.Oracle(kind, lock_slots=1).process(req)
    with Engine(kind, lock_slots=1) as eng:
        got = eng.submit_tensor(torch.from_numpy(req).cuda())
        torch.cuda.synchronize()
        check_replies(got.cpu().numpy(), want, eng.msg, "one slot")
        pr = M.predict(space, [(req, "device")])
        assert pr["max_run"] == n and pr["fallback_chunks"] == 1
        assert counters(eng) == expected(pr)


@pytest.mark.parametrize("small", [True, False], ids=["smallest", "over256"])
@pytest.mark.parametrize("kind", [wire.STORE, wire.TATP, wire.SMALLBANK], ids=["store", "tatp", "smallbank"])
def test_small_kv_tables(kind, small):
    """The smallest KV sizing the oracle and the engine accept (a handful of groups, so long runs in every chunk)
    and the first past 256 groups (two radix passes): random traces, a closed loop (store), and at the smallest
    sizing one key taking a whole 2^16-request chunk."""
    import torch
    cfg = M.KV_SIZINGS[kind][0 if small else 1]
    space = M.Space(kind, chunk=4096, **cfg)
    n_subs = cfg.get("subs_populate", cfg.get("accts_populate"))
    ora = O.Oracle(kind, **cfg)
    if kind == wire.STORE:
        req = T.store_random(30000, n_subs, seed=n_subs)
    elif kind == wire.TATP:
        req = T.tatp_random(20000, n_subs, seed=n_subs, oracle=ora)
    else:
        req = T.smallbank_random(30000, n_subs, seed=n_subs)
    want = ora.process(req)
    with Engine(kind, chunk=4096, populate=True, **cfg) as eng:
        check_replies(eng.submit(req), want, eng.msg, "random trace")
        assert counters(eng) == expected(M.predict(space, [(req, "host")]))
        assert probes(eng, kind, req) == probes(ora, kind, req)
        if kind == wire.STORE:
            eng.reset_stats()
            wl = Workload(wire.STORE, n_clients=1024, set_pct=50, store_subscribers=n_subs)
            req, want = record_trace(wl, ora.process, 20)
            check_replies(eng.submit(req), want, eng.msg, "closed loop")
            assert counters(eng) == expected(M.predict(space, [(req, "host")]))
    if small:
        space = M.Space(kind, chunk=1 << 16, **cfg)
        rng = np.random.default_rng(4)
        pool = M.Pool(space, [int(T.store_key(0, 1, 0))] if kind == wire.STORE else [0])
        req = M.build_one_group(space, pool, 1 << 16, rng)
        want = O.Oracle(kind, **cfg).process(req)
        with Engine(kind, chunk=1 << 16, populate=True, **cfg) as eng:
            got = eng.submit_tensor(torch.from_numpy(req).cuda())
            torch.cuda.synchronize()
            check_replies(got.cpu().numpy(), want, eng.msg, "one key")
            pr = M.predict(space, [(req, "device")])
            assert pr["max_run"] == 1 << 16
            assert counters(eng) == expected(pr)


# ---------------------------------------------------------------- (c) chunk, slice and call boundaries ---------------
ALL_KINDS = [wire.LOCK2PL, wire.FASST, wire.LOG, wire.STORE, wire.TATP, wire.SMALLBANK]
SMALL_CFG = {wire.LOG: dict(log_ring=7), wire.STORE: dict(subs_populate=20), wire.TATP: dict(subs_populate=3),
             wire.SMALLBANK: dict(accts_populate=40)}


def _trace(kind, n, seed):
    if kind == wire.FASST:
        return T.fasst_random(n, 60, seed)
    if kind == wire.LOCK2PL:
        return T.lock2pl_random(n, 60, seed)
    if kind == wire.LOG:
        return T.log_random(n, seed)
    if kind == wire.STORE:
        return T.store_random(n, 20, seed)
    if kind == wire.TATP:
        return T.tatp_random(n, 3, seed)
    return T.smallbank_random(n, 40, seed)


@pytest.mark.parametrize("kind", ALL_KINDS, ids=[wire.KIND_NAMES[k] for k in ALL_KINDS])
def test_call_boundaries_across_paths_and_streams(kind):
    """One seeded sequence of calls of 0, 1, 127, 128, 129, chunk - 1, chunk, chunk + 1 and 3 chunk + 5 requests,
    alternating the host path, the device path on the current stream and the device path on a second stream; the
    first requests of every call touch the groups of the last ones of the call before.  The replies, concatenated,
    are those of ONE oracle fed the concatenation."""
    import torch
    chunk = 4096
    msg = wire.MSG_SIZE[kind]
    cfg = SMALL_CFG.get(kind, {})
    rng = np.random.default_rng(kind)
    sizes = [int(x) for x in rng.permutation([0, 1, 127, 128, 129, chunk - 1, chunk, chunk + 1, 3 * chunk + 5] * 2)]
    req = _trace(kind, sum(sizes), seed=kind + 1)
    if kind not in (wire.LOG, wire.TATP):           # (tatp: a 3-subscriber universe, every key recurs anyway)
        rec = wire.as_records(kind, req).copy()
        for e in np.cumsum(sizes)[:-1]:
            k = min(8, e, len(rec) - e)
            for f in ("lid",) if kind in (wire.FASST, wire.LOCK2PL) else ("key", "table") if kind == wire.SMALLBANK else ("key",):
                rec[f][e:e + k] = rec[f][e - k:e]
        req = wire.as_bytes(rec)
    ora = O.Oracle(kind, **cfg)
    want = ora.process(req)
    space = M.Space(kind, chunk=chunk, **cfg)
    side = torch.cuda.Stream()
    cur = torch.cuda.current_stream()
    got, calls, off = [], [], 0
    with Engine(kind, chunk=chunk, populate=kind in VALSZ, **cfg) as eng:
        eng.reset_stats()
        for i, n in enumerate(sizes):
            part = req[off * msg:(off + n) * msg]
            off += n
            path = ("host", "device", "side")[i % 3]
            if path == "host":
                got.append(eng.submit(part))
            else:
                d = torch.from_numpy(part.copy()).cuda()
                if path == "side":
                    side.wait_stream(cur)                          # successive calls must be ordered
                    with torch.cuda.stream(side):
                        out = eng.submit_tensor(d, stream=side.cuda_stream)
                    cur.wait_stream(side)
                else:
                    out = eng.submit_tensor(d)
                got.append((out, d))
            calls.append((part, "host" if path == "host" else "device"))
        torch.cuda.synchronize()
        got = np.concatenate([g if isinstance(g, np.ndarray) else g[0].cpu().numpy() for g in got])
        check_replies(got, want, msg, f"calls {sizes}")
        if kind != wire.LOG:
            assert counters(eng) == expected(M.predict(space, calls))
        assert probes(eng, kind, req) == probes(ora, kind, req)


def test_host_path_pyramid_with_conflicts_at_every_slice_boundary():
    """One lock_fasst host-path call of ~2.5 M requests at the default chunk over 50 000 ids: more slices than the
    four-buffer ring, and every slice's listed replies become final only after the next slice's classify launch."""
    n = 2_500_003
    req = T.fasst_random(n, 50000, seed=77)
    space = M.Space(wire.FASST)
    slices = M.host_slices(n, space)
    assert len(slices) > 4 and max(slices) == 1 << 18
    ora = O.Oracle(wire.FASST)
    want = ora.process(req)
    with Engine(wire.FASST) as eng:
        check_replies(eng.submit(req), want, 9, "2.5 M requests")
        assert counters(eng) == expected(M.predict(space, [(req, "host")]))
        sample = req.reshape(-1, 9)[::997].reshape(-1)
        assert probes(eng, wire.FASST, sample) == probes(ora, wire.FASST, sample)


# ---------------------------------------------------------------- (d) snapshots --------------------------------------
@pytest.mark.parametrize("kind", ALL_KINDS, ids=[wire.KIND_NAMES[k] for k in ALL_KINDS])
def test_snapshot_restore_replays_exactly(kind):
    """Prefix P, snapshot, segment S, restore, S again (host path), and once more restored on a side stream and
    served by the device path on that stream with no host synchronisation in between: every replay of S answers
    like an oracle fed P + S, and leaves the same state."""
    import torch
    msg = wire.MSG_SIZE[kind]
    cfg = SMALL_CFG.get(kind, {})
    req = _trace(kind, 60000, seed=kind + 50)
    P, S = req[:20000 * msg], req[20000 * msg:]
    ora = O.Oracle(kind, **cfg)
    ora.process(P)
    want = ora.process(S)
    with Engine(kind, populate=kind in VALSZ, **cfg) as eng:
        eng.submit(P)
        snap = eng.snapshot()
        try:
            check_replies(eng.submit(S), want, msg, "first S")
            state = probes(eng, kind, req)
            assert state == probes(ora, kind, req)
            eng.restore(snap)
            check_replies(eng.submit(S), want, msg, "S after restore")
            assert probes(eng, kind, req) == state
            side = torch.cuda.Stream()
            d = torch.from_numpy(S.copy()).cuda()
            side.wait_stream(torch.cuda.current_stream())
            eng.restore(snap, side.cuda_stream)
            out = eng.submit_tensor(d, stream=side.cuda_stream)
            side.synchronize()
            check_replies(out.cpu().numpy(), want, msg, "S after restore on a side stream")
            assert probes(eng, kind, req) == state
        finally:
            eng.free_snapshot(snap)


def test_snapshot_restore_is_refused_after_the_table_doubled():
    """A TATP call-forwarding table of 1024 entries: net inserts past 35 % load, then insert / delete churn until the
    table is rehashed.  A doubled table makes restore fail with EINVAL and leaves the engine answering exactly; a
    same-capacity rehash lets restore succeed and the replay stay exact."""
    from dint_b200.wire import Tatp
    n_subs = 20
    cfg = dict(subs_populate=n_subs, kv_capacity_log2=[0, 0, 0, 0, 10])
    ora = O.Oracle(wire.TATP, subs_populate=n_subs)
    snap_ora = O.Oracle(wire.TATP, subs_populate=n_subs)        # the state at the snapshot: freshly populated
    rng = np.random.default_rng(9)
    next_sid = [1000]

    def calls(m, keep):
        keys = np.arange(next_sid[0], next_sid[0] + m, dtype=np.uint64) | (np.uint64(1) << np.uint64(32)) | (np.uint64(8) << np.uint64(40))
        next_sid[0] += m
        parts = [(Tatp.kInsertBck, keys), (Tatp.kRead, keys)] + ([] if keep else [(Tatp.kDeleteBck, keys)])
        rec = np.zeros(len(parts) * m, dtype=wire.MSG_DTYPE[wire.TATP])
        rec["table"] = Tatp.kCallForwarding
        rec["key"] = np.concatenate([k for _, k in parts])
        rec["type"] = np.concatenate([np.full(m, t) for t, _ in parts]).astype(np.uint8)
        rec["val"] = rng.integers(0, 256, size=(len(rec), 40))
        return wire.as_bytes(rec)

    probe_req = T.tatp_random(4000, n_subs, seed=3, oracle=snap_ora)
    with Engine(wire.TATP, populate=True, chunk=4096, **cfg) as eng:
        snap = eng.snapshot()
        try:
            r = calls(340, keep=True)                                      # net inserts: past 35 % of 1024
            check_replies(eng.submit(r), ora.process(r), 55, "net inserts")
            assert eng.kv_count(4) == ora.kv_count(4) > 0.35 * 1024
            for i in range(40):                                            # churn until the table is rehashed
                r = calls(256, keep=False)
                check_replies(eng.submit(r), ora.process(r), 55, f"churn call {i}")
                if eng.stats()["kv_rebuilds"]:
                    break
            assert eng.stats()["kv_rebuilds"] >= 1
            try:
                eng.restore(snap)
            except DintError as e:
                assert e.code == -22                                       # DINT_EINVAL: the table doubled
                r = calls(200, keep=False)
                check_replies(eng.submit(r), ora.process(r), 55, "after the refused restore")
                assert eng.kv_count(4) == ora.kv_count(4)
            else:                                                          # a same-capacity rehash: the restore stands
                check_replies(eng.submit(probe_req), snap_ora.process(probe_req), 55, "after the restore")
                assert eng.kv_count(4) == snap_ora.kv_count(4)
        finally:
            eng.free_snapshot(snap)
