"""CPU checks of tests/replay_model.py: its hashing agrees with the oracle, every trace builder produces the chunk
shape it is named after (so the GPU tests of test_gpu_replay_boundaries.py aim where they say), and its notion of
"listed" is sound: replaying the unlisted requests in any order and each group's listed requests in index order
gives the replies of the whole trace processed in order."""
import numpy as np
import pytest

import oracle_lib as O
import replay_model as M
import trace_gen as T
from dint_b200 import wire

KINDS = [wire.LOCK2PL, wire.FASST, wire.STORE, wire.TATP, wire.SMALLBANK]


def test_group_ids_agree_with_the_oracle():
    """Lock slots of the lock kinds and lock_hash of the TATP / SmallBank tables (store's group, its kvs bucket, is
    the same fasthash64 modulo the bucket count)."""
    rng = np.random.default_rng(1)
    for kind, cfg, tables in [(wire.FASST, dict(lock_slots=36000000), [0]), (wire.LOCK2PL, dict(lock_slots=65537), [0]),
                              (wire.TATP, dict(subs_sizing=3, subs_populate=1), range(5)),
                              (wire.SMALLBANK, dict(accts_sizing=24000000, accts_populate=1), range(2))]:
        ora = O.Oracle(kind, populate=False, **cfg)
        sp = M.Space(kind, **cfg)
        keys = rng.integers(0, 2**32 if kind in (wire.FASST, wire.LOCK2PL) else 2**63, size=200, dtype=np.uint64)
        for t in tables:
            g = sp.group(keys, t)
            assert [int(x) - sp.base[t] for x in g] == [ora.lock_slot(t, int(k)) for k in keys], (kind, t)
    for k in (0, 1, 2**32, 2**63 + 5):
        assert int(M.fasthash64_u64(np.uint64(k))) == O.fasthash64(int(k).to_bytes(8, "little"))


@pytest.mark.parametrize("slots,passes,flags_log2", [(1, 1, 12), (7, 1, 12), (256, 1, 12), (257, 2, 12), (65536, 2, 18),
                                                     (65537, 3, 18), ((1 << 24) + 1, 4, 25), (36000000, 4, 25)])
def test_lock_slots_cover_every_radix_pass_count(slots, passes, flags_log2):
    sp = M.Space(wire.FASST, lock_slots=slots)
    assert (sp.sort_passes, sp.flags_log2) == (passes, flags_log2)
    assert (sp.groups > sp.flags_mask + 1) == (slots == 36000000)     # only the reference size folds its flag nibbles


def test_small_kv_sizings():
    """The smallest sizes the oracle and the engine accept give a handful of groups (one radix pass); the second
    sizing of each kind is the first past 256 groups (two passes)."""
    for kind, (small, big) in M.KV_SIZINGS.items():
        a, b = M.Space(kind, **small), M.Space(kind, **big)
        assert a.sort_passes == 1 and a.groups <= 64, (kind, a.groups)
        assert b.sort_passes == 2 and 256 < b.groups <= 300, (kind, b.groups)
        key = "subs_sizing" if kind != wire.SMALLBANK else "accts_sizing"
        with pytest.raises(ValueError):
            M.Space(kind, **{key: small[key] - 1})        # one less and a table has no lock slot


@pytest.mark.parametrize("chunk", [4096, 1 << 16])
@pytest.mark.parametrize("kind", KINDS, ids=[wire.KIND_NAMES[k] for k in KINDS])
def test_builders_hit_their_target_shape(kind, chunk):
    space, cfg, cases = M.threshold_cases(kind, chunk, seed=kind * 100 + chunk)
    names = [c[0] for c in cases]
    assert names[:6] == ["bucket_128", "bucket_129", "task_32", "task_33", "task_128", "task_129"]
    assert ("nibble_alias" in names) == (kind != wire.STORE)            # store's 9 M groups fit 2^25 nibbles unfolded
    assert ("readonly_then_writer" in names) == (kind in (wire.FASST, wire.STORE, wire.TATP))
    msg = wire.MSG_SIZE[kind]
    for name, raw, want in cases:
        assert raw.size % (chunk * msg) == 0, name
        pr = M.predict(space, [(raw, "host")])
        cms = pr["chunks"]
        assert len(cms) == raw.size // (chunk * msg), name
        cm = cms[0]
        if "bucket" in want:
            assert sorted(cm["bucket_counts"])[-2:] == [0, want["bucket"]], name      # ONE bucket holds them all
            assert cm["nc"] == want["bucket"] and cm["overflow"] == (want["bucket"] > 128), name
            assert pr["fallback_chunks"] == int(want["bucket"] > 128)
            assert pr["max_run"] == min(40, want["bucket"])
        elif "task" in want:
            total = want["task"]
            assert cm["nc"] == total and not cm["overflow"] and cm["gsz"] >= 2, name
            tasks = np.flatnonzero(cm["task_totals"])
            assert len(tasks) == 1 and cm["task_totals"][tasks[0]] == total, name
            assert (cm["task_counts"][tasks[0]] > 0).sum() == 2, name         # spread over two buckets of the task
            mode, sorts = M.sort_modes(cm, tasks[0])
            if total <= 128:
                assert (mode, sorts) == ("one pass", ["rank" if total <= 32 else "bitonic"]), name
            else:
                assert (mode, sorts) == ("per bucket", ["bitonic", "bitonic"]), name
        elif "alias" in want:
            lg = cm["g"][cm["listed"]]
            assert cm["nc"] == 2 and lg[0] != lg[1] and (lg[0] - lg[1]) % (space.flags_mask + 1) == 0, name
            assert pr["max_run"] == 0 and pr["fallback_chunks"] == 0
        else:
            assert cms[0]["nc"] == 0 and not cms[0]["has_writer"], name
            assert cms[1]["nc"] == 40 * 6 and cms[1]["max_run"] == 6, name
            assert set(cms[0]["g"][cms[0]["mask"] == M.C_RA]) >= set(cms[1]["g"][cms[1]["listed"]])


def test_one_group_fills_a_chunk():
    space = M.Space(wire.FASST, lock_slots=1)
    rng = np.random.default_rng(3)
    raw = M.build_one_group(space, M.default_pool(space, rng, n=16), 1 << 12, rng)
    cm = M.chunk_model(space, raw)
    assert cm["nc"] == 1 << 12 and cm["max_run"] == 1 << 12 and cm["overflow"]


def _replay_by_group(kind, cfg, raw, space):
    """Replies of `raw` (one chunk) when the unlisted requests run first, LAST to first, and then every group's
    listed requests in index order, groups in a shuffled order."""
    msg = wire.MSG_SIZE[kind]
    rec = raw.reshape(-1, msg)
    cm = M.chunk_model(space, raw)
    ora = O.Oracle(kind, **cfg)
    out = np.empty_like(rec)
    for i in np.flatnonzero(~cm["listed"])[::-1]:
        out[i] = ora.process(rec[i]).reshape(msg)
    listed = np.flatnonzero(cm["listed"])
    groups = np.unique(cm["g"][listed])
    for grp in np.random.default_rng(0).permutation(groups):
        idx = listed[cm["g"][listed] == grp]
        out[idx] = ora.process(rec[idx].reshape(-1)).reshape(-1, msg)
    return out.reshape(-1), cm


@pytest.mark.parametrize("kind", KINDS, ids=[wire.KIND_NAMES[k] for k in KINDS])
def test_listed_requests_are_exactly_the_ones_that_need_index_order(kind):
    chunk = 2048
    cfg = {wire.STORE: dict(subs_populate=50), wire.TATP: dict(subs_populate=10),
           wire.SMALLBANK: dict(accts_populate=60)}.get(kind, {})
    space = M.Space(kind, chunk=chunk, **cfg)
    traces = []
    if kind == wire.FASST:
        traces.append(T.fasst_random(chunk, 3000, seed=1))
    elif kind == wire.LOCK2PL:
        traces.append(T.lock2pl_random(chunk, 3000, seed=1))
    elif kind == wire.STORE:
        traces.append(T.store_random(chunk, 50, seed=1))
    elif kind == wire.TATP:
        traces.append(T.tatp_random(chunk, 10, seed=1))
    else:
        traces.append(T.smallbank_random(chunk, 60, seed=1))
    traces = [(cfg, space, raw) for raw in traces]
    space2, cfg2, cases = M.threshold_cases(kind, chunk, seed=5)
    traces += [(cfg2, space2, raw[:chunk * wire.MSG_SIZE[kind]]) for name, raw, _ in cases if name in ("bucket_129", "nibble_alias")]
    for cf, sp, raw in traces:
        want = O.Oracle(kind, **cf).process(raw)
        got, cm = _replay_by_group(kind, cf, raw, sp)
        assert 0 < cm["nc"] < chunk
        assert np.array_equal(got, want)
