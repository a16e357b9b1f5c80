"""Plain-numpy model of how the engine classifies and replays one chunk (engine.cuh, kernels.cuh), and trace builders
that aim a chunk at a chosen replay path.

For one chunk the model restates K1 / K2: every request's group id and what it touches ({RA, WA, WL}), the folded
flag nibble of its group, whether it is listed for the ordered replay (kernels.cuh k_apply), which of the
`chunk / 64` hash buckets a listed request lands in, whether a bucket overflows its 128 pairs (radix fallback,
k_ordered) or not (bucket replay inside the next K1, ordered_buckets: warp tasks of `gsz` buckets, one pass or
bucket by bucket, rank sort up to 32 pairs, bitonic above).  From that it predicts the engine's counters:
`conflicted` (listed requests), `max_run` (longest same-group run of listed requests in one chunk) and
`fallback_chunks`.

The builders search lids / keys until the model reports the intended shape; tests/test_replay_model_cpu.py checks
that they do, tests/test_gpu_replay_boundaries.py runs them on the engine.
"""
import ctypes as C

import numpy as np

from dint_b200 import wire
from dint_b200.wire import Fasst, Lock2pl, Store, Tatp, Smallbank
from properties import _mix, fasthash64_u32

LOCK2PL, FASST, LOG, STORE, TATP, SMALLBANK = range(6)
NO_GROUP = 0xFFFFFFFF
C_RA, C_WA, C_WL = 1, 2, 4
F_R, F_WA, F_WL, F_W2 = 1, 2, 4, 8
TILE = 128
BUCKET_CAP = 128           # kBucketCap
BUCKET_FILL = 64           # kBucketFill
HOST_MIN_SLICE = 131072    # dint_create: host_min_slice
HOST_MAX_SLICE = 1 << 18   # dint_create: host_chunk = min(2^18, chunk)


def fasthash64_u64(x, seed=0xDEADBEEF):
    """Vectorised fasthash64(&x, 8, seed): one 8-byte block, no tail (store/udp/kvs.h:33-35)."""
    with np.errstate(over="ignore"):
        m = np.uint64(0x880355F21E6D1965)
        h = np.uint64(seed) ^ (np.uint64(8) * m)
        h = (h ^ _mix(np.asarray(x, dtype=np.uint64))) * m
        return _mix(h)


class Space:
    """The group space of one engine configuration (n_shards = 1): per-table group modulus and first group id
    (kv.cuh kv_create_tables), the flag-set size and radix passes (engine.cu create_impl), and the bucket count
    (chunk / 64, rounded up to a power of two)."""

    def __init__(self, kind, lock_slots=36000000, subs_sizing=None, accts_sizing=24000000, chunk=1 << 20, **_):
        self.kind = kind
        S = subs_sizing if subs_sizing is not None else (7000000 if kind == TATP else 2000000)
        A = accts_sizing
        if kind in (LOCK2PL, FASST):
            mods = [lock_slots]
        elif kind == STORE:
            mods = [S * 18 // 4]
        elif kind == TATP:
            mods = [4 * h for h in (S * 3 // 2 // 4, S * 3 // 2 // 4, S * 15 // 4 // 4, S * 15 // 4 // 4, S * 45 // 8 // 4)]
        elif kind == SMALLBANK:
            mods = [4 * (A * 3 // 2 // 4)] * 2
        else:
            mods = []
        if any(m == 0 for m in mods):
            raise ValueError("a table with no lock slots")
        self.mods = mods
        self.base = [int(x) for x in np.cumsum([0] + mods[:-1])] if mods else []
        self.groups = sum(mods)
        fl = 25
        while fl > 10 and (1 << (fl - 1)) >= self.groups * 2 + 2048:
            fl -= 1
        self.flags_log2 = fl
        self.flags_mask = (1 << fl) - 1
        bits = 1
        while (1 << bits) < self.groups:
            bits += 1
        self.sort_passes = (bits + 7) // 8
        self.chunk = (chunk + TILE - 1) // TILE * TILE
        lg = 0
        while (BUCKET_FILL << lg) < self.chunk:
            lg += 1
        self.bucket_log2 = lg
        self.n_buckets = 1 << lg
        self.host_chunk = min(HOST_MAX_SLICE, self.chunk)

    def group(self, keys, tables=0):
        """Group id of lock ids (lock kinds) or keys of `tables` (KV kinds)."""
        if self.kind in (LOCK2PL, FASST):
            return (fasthash64_u32(np.asarray(keys, dtype=np.uint32)) % np.uint64(self.mods[0])).astype(np.int64)
        t = np.broadcast_to(np.asarray(tables, dtype=np.int64), np.shape(keys))
        h = fasthash64_u64(keys)
        mod = np.asarray(self.mods, dtype=np.uint64)[t]
        return (h % mod).astype(np.int64) + np.asarray(self.base, dtype=np.int64)[t]

    def bucket(self, g):
        g = np.asarray(g, dtype=np.uint64)
        if self.bucket_log2 == 0:
            return np.zeros(g.shape, dtype=np.int64)
        return (((g * np.uint64(0x9E3779B1)) & np.uint64(0xFFFFFFFF)) >> np.uint64(32 - self.bucket_log2)).astype(np.int64)


def touches(kind, raw):
    """(mask, table, key) per request: what it touches inside its group (engine.cuh / kv.cuh type_info); mask 0 for
    requests that touch no group (log appends, would-panic requests)."""
    r = wire.as_records(kind, raw)
    n = len(r)
    mask = np.zeros(n, dtype=np.int64)
    table = np.zeros(n, dtype=np.int64)
    if kind == LOCK2PL:
        a, lt = r["action"].astype(np.int64), r["type"].astype(np.int64)
        mask[(a <= 1) & ~((a == 0) & (lt > 1))] = C_WL
        key = r["lid"]
    elif kind == FASST:
        t = r["type"]
        mask[t == 0] = C_RA
        mask[(t == 1) | (t == 2)] = C_WL
        mask[t == 3] = C_WA | C_WL
        key = r["lid"]
    elif kind == STORE:
        t = r["type"]
        mask[t == 0] = C_RA
        mask[(t == 1) | (t == 2)] = C_WA
        key = r["key"]
    elif kind == TATP:
        t, table = r["type"], r["table"].astype(np.int64)
        ok = table < 5
        mask[ok & (t == 0)] = C_RA
        mask[ok & ((t == 1) | (t == 2))] = C_WL
        mask[ok & np.isin(t, (12, 18, 22))] = C_WA | C_WL
        mask[ok & np.isin(t, (13, 19, 23))] = C_WA
        mask[(t == 14) | (t == 24)] = 0
        table = np.where(ok, table, 0)
        key = r["key"]
    elif kind == SMALLBANK:
        t, table = r["type"], r["table"].astype(np.int64)
        ok = table < 2
        mask[ok & (t <= 1)] = C_WL | C_RA
        mask[ok & ((t == 2) | (t == 3))] = C_WL
        mask[ok & ((t == 4) | (t == 5))] = C_WA
        table = np.where(ok, table, 0)
        key = r["key"]
    else:
        key = np.zeros(n, dtype=np.uint64)
    return mask, table, key


def chunk_model(space, raw):
    """What K1 / K2 decide for ONE chunk of wire records, and which replay path its listed requests take."""
    mask, table, key = touches(space.kind, raw)
    n = len(mask)
    act = mask != 0
    g = np.full(n, -1, dtype=np.int64)
    if act.any():
        g[act] = space.group(key[act], table[act])
    nib = np.where(act, g & space.flags_mask, -1)
    writer = act & (mask != C_RA)
    listed = np.zeros(n, dtype=bool)
    if writer.any():                                   # a chunk without a writer lists nothing (k_apply: chunk_has_writer)
        u, inv = np.unique(nib[act], return_inverse=True)
        m = mask[act]
        w = writer[act]
        fR = np.bincount(inv, weights=(m & C_RA) != 0, minlength=len(u)) > 0
        fWA = np.bincount(inv, weights=(m & C_WA) != 0, minlength=len(u)) > 0
        # W2: two writers of the nibble share WA or WL (whichever of them comes second sees the other's bit)
        nWA = np.bincount(inv, weights=w & ((m & C_WA) != 0), minlength=len(u))
        nWL = np.bincount(inv, weights=w & ((m & C_WL) != 0), minlength=len(u))
        fW2 = (nWA >= 2) | (nWL >= 2)
        fR, fWA, fW2 = fR[inv], fWA[inv], fW2[inv]
        listed[act] = (((m & C_RA) != 0) & fWA) | (((m & C_WA) != 0) & (fR | fW2)) | (((m & C_WL) != 0) & fW2)
    nc = int(listed.sum())
    P = space.n_buckets
    b = space.bucket(np.where(listed, g, 0))
    counts = np.bincount(b[listed], minlength=P)
    gsz = 1
    while gsz < 32 and nc * gsz * 2 <= 16 * P:
        gsz <<= 1
    n_tasks = (P + gsz - 1) // gsz
    task_counts = np.zeros(n_tasks * gsz, dtype=np.int64)
    task_counts[:P] = counts
    task_counts = task_counts.reshape(n_tasks, gsz)
    runs = np.unique(g[listed], return_counts=True)[1] if nc else np.zeros(0, dtype=np.int64)
    longest = int(runs.max()) if runs.size else 0
    return dict(n=n, g=g, nib=nib, mask=mask, listed=listed, nc=nc, bucket=b, bucket_counts=counts,
                overflow=bool((counts > BUCKET_CAP).any()), gsz=gsz, task_totals=task_counts.sum(axis=1),
                task_counts=task_counts, max_run=longest if longest > 1 else 0, has_writer=bool(writer.any()))


def sort_modes(cm, task):
    """How ordered_buckets sorts a warp task of the bucket path: one pass over all its pairs when they fit 128,
    else bucket by bucket; each pass by rank sort (m <= 32) or bitonic sort."""
    tc = cm["task_counts"][task]
    total = int(tc.sum())
    passes = [total] if total <= BUCKET_CAP else [int(x) for x in tc]
    return ("one pass" if total <= BUCKET_CAP else "per bucket",
            ["rank" if m <= 32 else "bitonic" for m in passes if m > 0])


def host_slices(n, space):
    """The slices dint_submit cuts a host-path call into (the engine's own schedule, through its test hook)."""
    from dint_b200 import engine as E
    if n == 0:
        return []
    L = E.lib()
    L.dint_test_host_slices.restype = C.c_uint32
    L.dint_test_host_slices.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_uint32), C.c_uint32]
    cap = 1 << 16
    buf = (C.c_uint32 * cap)()
    k = L.dint_test_host_slices(n, HOST_MIN_SLICE, space.host_chunk, 1, buf, cap)
    assert k <= cap
    return [int(x) for x in buf[:k]]


def chunks_of(n, space, path):
    """Chunk sizes of one call: the host path runs one chunk per slice, the device path cuts at `chunk`."""
    if path == "host":
        return host_slices(n, space)
    return [min(space.chunk, n - o) for o in range(0, n, space.chunk)]


def predict(space, calls):
    """calls: [(raw wire bytes, "host" | "device")].  Returns the counters the engine reports after them (from a
    reset) and the model of every chunk."""
    msg = wire.MSG_SIZE[space.kind]
    out = dict(conflicted=0, max_run=0, fallback_chunks=0, chunks=[])
    for raw, path in calls:
        raw = np.ascontiguousarray(raw).view(np.uint8).reshape(-1)
        off = 0
        for cn in chunks_of(raw.size // msg, space, path):
            cm = chunk_model(space, raw[off * msg:(off + cn) * msg])
            off += cn
            out["chunks"].append(cm)
            out["conflicted"] += cm["nc"]
            out["max_run"] = max(out["max_run"], cm["max_run"])
            out["fallback_chunks"] += int(cm["overflow"])
    return out


# ---------------------------------------------------------------------------------------------------------------
# wire records
def records(kind, keys, ops, rng, tables=0):
    """Wire records on `keys` with the request types `ops` (lock_2pl: action * 2 + lock type); random payloads."""
    n = len(keys)
    rec = np.zeros(n, dtype=wire.MSG_DTYPE[kind])
    ops = np.asarray(ops, dtype=np.int64)
    if kind == LOCK2PL:
        rec["action"], rec["type"], rec["lid"] = ops // 2, ops % 2, keys
    elif kind == FASST:
        rec["type"], rec["lid"] = ops, keys
        rec["ver"] = rng.integers(0, 2**32, size=n, dtype=np.uint64).astype(np.uint32)
    else:
        rec["type"], rec["key"] = ops, keys
        rec["val"] = rng.integers(0, 256, size=rec["val"].shape)
        rec["ver"] = rng.integers(0, 2**32, size=n, dtype=np.uint64).astype(np.uint32)
        if kind in (TATP, SMALLBANK):
            rec["table"] = tables
            rec["ord"] = rng.integers(0, 256, size=n)
    return wire.as_bytes(rec)


# request types by role: a WRITER conflicts with any other writer of its group (W2), so a group holding two or more
# of them has every one listed; a READER (RA only) alone never is; WA_WRITER: a writer of the versioned data (the
# TATP one needs an existing key).  Lock_2pl and SmallBank have no pure readers.
WRITERS = {LOCK2PL: [0, 1, 2, 3], FASST: [Fasst.kAcquireLock, Fasst.kAbort, Fasst.kCommit], STORE: [Store.kSet],
           TATP: [Tatp.kAcquireLock, Tatp.kAbort],
           SMALLBANK: [Smallbank.kAcquireShared, Smallbank.kAcquireExclusive, Smallbank.kReleaseShared,
                       Smallbank.kReleaseExclusive]}
KEYLESS_WRITERS = {**WRITERS, SMALLBANK: [Smallbank.kReleaseShared, Smallbank.kReleaseExclusive]}   # touch no row
READERS = {FASST: [Fasst.kRead], STORE: [Store.kRead], TATP: [Tatp.kRead]}
WA_WRITERS = {FASST: [Fasst.kCommit], STORE: [Store.kSet], TATP: [Tatp.kCommitBck]}


class Pool:
    """Candidate lids / keys (of one table) with their group, flag nibble and bucket."""

    def __init__(self, space, keys, table=0):
        self.space = space
        self.keys = np.asarray(keys)
        self.table = table
        self.g = space.group(self.keys, table)
        self.nib = self.g & space.flags_mask
        self.bucket = space.bucket(self.g)

    def distinct(self, sel=None, avoid_nib=()):
        """Indices of candidates with pairwise distinct nibbles, none in avoid_nib, in pool order."""
        idx = np.arange(len(self.keys)) if sel is None else np.flatnonzero(sel)
        _, first = np.unique(self.nib[idx], return_index=True)
        idx = idx[np.sort(first)]
        return idx[~np.isin(self.nib[idx], np.asarray(list(avoid_nib), dtype=np.int64))]


def default_pool(space, rng, n=1 << 20, existing=0):
    """lids (lock kinds) or keys of table 0 (KV kinds): the keys a populated engine holds first (`existing`
    subscribers / accounts; SmallBank's acquires and TATP's data writers need them), then random ones (not for
    SmallBank, whose every key must exist)."""
    if space.kind in (LOCK2PL, FASST):
        return Pool(space, rng.permutation(np.arange(n, dtype=np.uint64)).astype(np.uint32))
    s = np.arange(existing, dtype=np.uint64)
    if space.kind == STORE:
        s = np.concatenate([s | (np.uint64(sf) << np.uint64(32)) | (np.uint64(st) << np.uint64(40))
                            for sf in (1, 2, 3, 4) for st in (0, 8, 16)])
    extra = np.zeros(0, np.uint64) if space.kind == SMALLBANK else rng.integers(1 << 40, 1 << 62, size=n, dtype=np.uint64)
    return Pool(space, np.concatenate([rng.permutation(s), extra]))


def _run_sizes(total, rng, longest):
    """Run lengths >= 2 summing to `total`, the first of them `longest` (or total, when smaller)."""
    sizes = [min(longest, total)]
    left = total - sizes[0]
    while left:
        s = int(rng.integers(2, 6))
        if left - s < 2 and left != s:
            s = left if left <= 5 else 2
        sizes.append(s)
        left -= s
    assert all(s >= 2 for s in sizes) or total < 2
    return sizes


def _assemble(space, pool, groups, sizes, n, rng, writers=None, extra=None):
    """A chunk of n records: sizes[i] writers on pool candidate groups[i] (a listed run each), `extra` (keys, ops,
    tables) records, and solo singletons on fresh nibbles for the rest, in a seeded random order."""
    kind = space.kind
    writers = WRITERS[kind] if writers is None else writers
    keys = [np.repeat(pool.keys[groups], sizes)]
    ops = [rng.choice(writers, size=int(np.sum(sizes)))]
    tabs = [np.full(int(np.sum(sizes)), pool.table)]
    used = set(pool.nib[groups].tolist())
    if extra is not None:
        keys.append(extra[0]); ops.append(extra[1]); tabs.append(extra[2])
        used |= set(extra[3])
    n_fill = n - sum(len(k) for k in keys)
    fill = pool.distinct(avoid_nib=used)[:n_fill]
    if len(fill) < n_fill:
        raise ValueError("candidate pool too small for the filler")
    solo_ops = READERS.get(kind, []) + writers
    keys.append(pool.keys[fill]); ops.append(rng.choice(solo_ops, size=n_fill)); tabs.append(np.full(n_fill, pool.table))
    keys, ops, tabs = np.concatenate(keys), np.concatenate(ops), np.concatenate(tabs)
    order = rng.permutation(len(keys))
    return records(kind, keys[order], ops[order], rng, tabs[order])


def build_bucket(space, pool, n_listed, rng, bucket=None, longest=40, writers=None):
    """One full chunk whose listed requests all sit in ONE bucket, exactly n_listed of them (128: the bucket path's
    limit; 129: the radix fallback)."""
    b = int(np.argmax(np.bincount(pool.bucket, minlength=space.n_buckets))) if bucket is None else bucket
    sizes = _run_sizes(n_listed, rng, longest)
    cand = pool.distinct(pool.bucket == b)
    if len(cand) < len(sizes):
        raise ValueError("too few groups in the bucket")
    return _assemble(space, pool, cand[:len(sizes)], sizes, space.chunk, rng, writers)


def build_hot_bucket(space, pool, n, rng):
    """n writers on a few groups of ONE bucket: the bucket overflows whatever the size of the group space."""
    b = int(np.argmax(np.bincount(pool.bucket, minlength=space.n_buckets)))
    sel = np.flatnonzero(pool.bucket == b)[:64]
    return records(space.kind, pool.keys[rng.choice(sel, size=n)], rng.choice(WRITERS[space.kind], size=n), rng, pool.table)


def build_task(space, pool, total, rng, n_buckets=2, writers=None):
    """One full chunk whose listed requests (and nothing else) fill ONE warp task of the bucket path to `total`
    pairs, spread over n_buckets of its buckets (no bucket above 128)."""
    gsz = 1
    while gsz < 32 and total * gsz * 2 <= 16 * space.n_buckets:
        gsz <<= 1
    nb = min(n_buckets, gsz)
    task = int(rng.integers(0, max(1, space.n_buckets // gsz)))
    parts = [total // nb + (i < total % nb) for i in range(nb)]
    groups, sizes, used = [], [], set()
    for i, part in enumerate(parts):
        cand = pool.distinct(pool.bucket == task * gsz + i, avoid_nib=used)
        sz = _run_sizes(part, rng, 7)
        if len(cand) < len(sz):
            raise ValueError("too few groups in the bucket")
        groups += list(cand[:len(sz)]); sizes += sz
        used |= set(pool.nib[cand[:len(sz)]].tolist())
    return _assemble(space, pool, np.array(groups), sizes, space.chunk, rng, writers)


def find_alias(space, pools):
    """Two candidates (pool index, candidate index) of DIFFERENT groups that share a flag nibble, or None when the
    group space fits the flag set unfolded."""
    if space.groups <= space.flags_mask + 1:
        return None
    nib = np.concatenate([p.nib for p in pools])
    g = np.concatenate([p.g for p in pools])
    src = np.concatenate([np.stack([np.full(len(p.keys), i), np.arange(len(p.keys))], axis=1) for i, p in enumerate(pools)])
    order = np.lexsort((g, nib))
    hit = np.flatnonzero((nib[order][1:] == nib[order][:-1]) & (g[order][1:] != g[order][:-1]))
    if hit.size == 0:
        return None
    a, b = src[order[hit[0]]], src[order[hit[0] + 1]]
    return (int(a[0]), int(a[1])), (int(b[0]), int(b[1]))


def build_alias(space, pool, alias_pools, rng, writers):
    """One full chunk holding ONE writer on each of two different groups that share a flag nibble: folding makes
    both listed (as a run of one each), nothing else is listed."""
    hit = find_alias(space, alias_pools)
    if hit is None:
        return None
    (pa, ca), (pb, cb) = hit
    A, B = alias_pools[pa], alias_pools[pb]
    keys = np.array([A.keys[ca], B.keys[cb]], dtype=np.uint64)
    extra = (keys, rng.choice(writers, size=2), np.array([A.table, B.table]), [int(A.nib[ca])])
    return _assemble(space, pool, np.zeros(0, dtype=np.int64), [], space.chunk, rng, writers, extra=extra)


def build_readonly_then_writer(space, pool, rng, n_groups=40, reads=6):
    """Two full chunks on the same groups: the first only reads them (several reads per group, nothing listed:
    no writer in the chunk), the second reads them again with one data writer per group (everything on them listed)."""
    kind = space.kind
    cand = pool.distinct()[:n_groups]
    keys = np.repeat(pool.keys[cand], reads)
    nib = pool.nib[cand].tolist()
    rd = READERS[kind][0]
    ro = _assemble(space, pool, np.zeros(0, dtype=np.int64), [], space.chunk, rng, READERS[kind],
                   extra=(keys, np.full(len(keys), rd), np.full(len(keys), pool.table), nib))
    ops = np.full(len(keys), rd)
    ops[::reads] = WA_WRITERS[kind][0]
    wr = _assemble(space, pool, np.zeros(0, dtype=np.int64), [], space.chunk, rng, READERS[kind],
                   extra=(keys, ops, np.full(len(keys), pool.table), nib))
    return np.concatenate([ro, wr])


def build_one_group(space, pool, n, rng, writers=None, readers=True):
    """n requests on ONE key (so one group holds the whole chunk), writers and readers mixed (with a writer of the
    versioned data among them, every request is listed)."""
    kind = space.kind
    ops = list(WRITERS[kind] if writers is None else writers) + (READERS.get(kind, []) + WA_WRITERS.get(kind, []) if readers else [])
    return records(kind, np.full(n, pool.keys[0]), rng.choice(ops, size=n), rng, pool.table)


# KV sizings of the small-group-space tests: the smallest each kind accepts (every table has a lock slot), and the
# first that gives more than 256 groups (two radix passes)
KV_SIZINGS = {STORE: (dict(subs_sizing=1, subs_populate=1), dict(subs_sizing=58, subs_populate=58)),
              TATP: (dict(subs_sizing=3, subs_populate=3), dict(subs_sizing=17, subs_populate=17)),
              SMALLBANK: (dict(accts_sizing=3, accts_populate=3), dict(accts_sizing=88, accts_populate=88))}


# ---------------------------------------------------------------------------------------------------------------
# the threshold cases: reference table sizes, a small population
THRESHOLD_CFG = {LOCK2PL: {}, FASST: {}, STORE: dict(subs_populate=6000), TATP: dict(subs_populate=2000),
                 SMALLBANK: dict(accts_populate=200000)}


def threshold_cases(kind, chunk, seed):
    """(space, engine / oracle cfg, [(name, wire bytes, intended shape)]) for one kind and chunk size: a bucket at
    128 and at 129 listed pairs, warp tasks of 32 / 33 / 128 / 129 pairs, a flag-nibble alias pair (where the group
    space is folded at all), and a read-only chunk followed by a writer chunk on the same groups (kinds that have
    pure readers).  Every trace is a whole number of chunks."""
    rng = np.random.default_rng(seed)
    cfg = dict(THRESHOLD_CFG[kind])
    space = Space(kind, chunk=chunk, **cfg)
    existing = cfg.get("subs_populate", cfg.get("accts_populate", 0))
    pool = default_pool(space, rng, existing=existing)
    cases = [("bucket_128", build_bucket(space, pool, 128, rng), dict(bucket=128)),
             ("bucket_129", build_bucket(space, pool, 129, rng), dict(bucket=129))]
    for total in (32, 33, 128, 129):
        cases.append((f"task_{total}", build_task(space, pool, total, rng), dict(task=total)))
    alias_pools = [pool]
    if kind == TATP:
        alias_pools.append(Pool(space, rng.integers(1 << 40, 1 << 62, size=1 << 18, dtype=np.uint64), table=4))
    raw = build_alias(space, pool, alias_pools, rng, KEYLESS_WRITERS[kind])
    if raw is not None:
        cases.append(("nibble_alias", raw, dict(alias=True)))
    if kind in READERS:
        cases.append(("readonly_then_writer", build_readonly_then_writer(space, pool, rng), dict(readonly_then_writer=True)))
    return space, cfg, cases
