// engine.cuh -- device-side context, wire layouts and per-kind request semantics.
//
// Batch semantics.  dint_submit() must answer exactly as ONE reference server thread would have,
// taking the requests one by one in index order.  Two requests interact only if they touch the same
// "group" (a lock slot; for the KV kinds the lock slot of the key, which also pins the key), so a
// chunk of requests is processed in three launches:
//
//   K1 classify : stage the tile of wire records (TMA bulk copy), hash every key to its group id,
//                 record the id, and mark a 4-bit flag nibble per group.  A group has two resources:
//                 A (the versioned data: ver_table entry / KV rows) and L (the lock word / counters).
//                 A request is a reader of A (RA), a writer of A (WA) and/or a writer of L (WL); the
//                 nibble holds R (an RA exists), WA, WL and W2 (two or more writers of one class).
//                 The flag array is hash-folded to 2^25 nibbles (16 MB), so it stays in the 126 MB
//                 L2; folding can only add conflicts, never hide one.  Two flag sets alternate
//                 between chunks: K1 of chunk k also zeroes the words chunk k-1 touched.
//   K2 apply    : a request is SOLO when nothing else in the chunk can interact with it
//                 (RA: WA clear; WA: R and W2 clear; WL: W2 clear).  Solo requests are applied
//                 directly, one thread each, against the HBM-resident state and their tile is
//                 written back with one bulk store.  The others are listed, in index order, for K3.
//                 Persistent CTAs run a 3-stage TMA pipeline over the tiles.
//   ordered replay: K2 hashes the listed (group, index) pairs into buckets of <= 128.  The NEXT launch of
//                 K1 (or a flush launch at the end of a submit call) replays them while it classifies
//                 the next chunk: a warp gathers a few adjacent buckets into its slice of shared memory,
//                 sorts the pairs (rank sort by shuffles up to 32, bitonic above) and replays every
//                 same-group run in index order -- request fields fetched in parallel, the group's state
//                 walked in registers, replies written in parallel (lock servers), or request by request
//                 with the very same apply_one as K2 (KV servers).  No grid-wide barrier is involved.
//   K3 fallback : heavily skewed chunks that overflow a bucket (HOT: 4800 ids) are instead sorted whole
//                 by a stable LSD radix sort (cooperative launch, grid barriers) and replayed; the
//                 launch exits at once when no bucket overflowed.
//
// apply_one<KIND>() below is therefore the single statement of each server's request semantics.
#pragma once
#include "common.cuh"

namespace dint {

enum Kind { K_LOCK2PL = 0, K_FASST = 1, K_LOG = 2, K_STORE = 3, K_TATP = 4, K_SMALLBANK = 5 };

constexpr int kTile = 128;       // wire records per tile = threads per CTA in K1/K2 (16 CTAs, i.e. 16 independent
                                 // latency chains, per SM)
constexpr int kThreads = 256;    // threads per CTA of the other kernels (K3's radix passes rely on 256)
constexpr int kMaxTables = 5;
constexpr uint32_t kBucketCap = 128;    // ordered replay: bucket capacity (sorted in a warp's slice of shared memory)
constexpr uint32_t kBucketFill = 64;    // K3: chunk / kBucketFill buckets (mean occupancy 64 if EVERY request were listed)
constexpr int kStages = 3;              // TMA pipeline depth of the persistent K1/K2 CTAs

// what a request touches inside its group (conflict detection)
enum : uint32_t { C_RA = 1, C_WA = 2, C_WL = 4 };
// flag nibble bits
enum : uint32_t { F_R = 1, F_WA = 2, F_WL = 4, F_W2 = 8 };

// ---- wire layouts (packed structs of the reference) ----------------------------------------------
template <int KIND> struct Wire;
template <> struct Wire<K_LOCK2PL> {   // lock_2pl/udp/net.h:25-31 {u8 action; u32 lid; u8 type}
  static constexpr int MSG = 6, TYPE = 0, KEY = 1, LTYPE = 5;
};
template <> struct Wire<K_FASST> {     // lock_fasst/udp/net.h:25-31 {u8 type; u32 lid; u32 ver}
  static constexpr int MSG = 9, TYPE = 0, KEY = 1, VER = 5;
};
template <> struct Wire<K_LOG> {       // log_server/udp/net.h:23-30 {u8 type; u64 key; u8 val[40]; u32 ver}
  static constexpr int MSG = 53, TYPE = 0, KEY = 1, VAL = 9, VER = 49, VALSZ = 40, LOGENT = 56;
};
template <> struct Wire<K_STORE> {     // store/udp/net.h:34-41 (same shape)
  static constexpr int MSG = 53, TYPE = 0, KEY = 1, VAL = 9, VER = 49, VALSZ = 40;
};
template <> struct Wire<K_TATP> {      // tatp/udp/net.h:57-65 {u8 ord; u8 type; u8 table; u64 key; u8 val[40]; u32 ver}
  static constexpr int MSG = 55, TYPE = 1, TABLE = 2, KEY = 3, VAL = 11, VER = 51, VALSZ = 40, LOGENT = 64;
};
template <> struct Wire<K_SMALLBANK> { // smallbank/udp/net.h:43-52 {u8 ord; u8 type; u8 table; u64 key; u8 val[8]; u32 ver}
  static constexpr int MSG = 23, TYPE = 1, TABLE = 2, KEY = 3, VAL = 11, VER = 19, VALSZ = 8, LOGENT = 32;
};

// ---- KV table: open addressing, one 64-byte (val 40) or 32-byte (val 8) entry per key -------------
// entry = { u64 key; u32 ver; u32 meta; u8 val[VALSZ]; pad } -- a GET that hits on its first probe
// costs exactly one aligned 64-byte (32-byte) HBM access.
enum : uint32_t { ENT_EMPTY = 0, ENT_FULL = 1, ENT_TOMB = 2, ENT_BUSY = 3 };
struct KvTable {
  uint8_t* entries;
  uint64_t cap_mask;       // capacity - 1 (power of two)
  uint32_t cap_log2;
  uint32_t ent_shift;      // log2(entry bytes): 6 or 5
  FastMod lock_mod;        // kKeysPerEntry * hash_size of the reference (tatp.h:12-14, smallbank.h:12-14)
  uint32_t grp_base;       // first group id of this table
  uint32_t n_groups;       // local groups of this table
  unsigned long long* live;  // [0] live keys, [1] entries that have left EMPTY (FULL + TOMB)
};

struct Ctx {
  // chunk
  const uint8_t* req;      // n wire records, 16-byte aligned
  uint8_t* resp;           // n wire records, 16-byte aligned (may equal req)
  uint32_t n;
  uint32_t n_tiles;
  // conflict detection
  uint32_t* grp;           // [chunk] group id per request of THIS chunk (0xffffffff: none)
  const uint32_t* grp_prev;  // [prev_n] group ids of the previous chunk (its flags are cleared by this K1)
  uint32_t prev_n;
  uint32_t* flags;         // this chunk's flag set: 2^flags_log2 nibbles
  uint32_t* flags_prev;    // the previous chunk's flag set
  uint32_t flags_mask;     // 2^flags_log2 - 1
  uint32_t* clist;         // [n_tiles][kTile] indices of listed requests, tile-segmented
  uint32_t* ccnt;          // [n_tiles] listed requests per tile
  uint32_t* cprefix;       // [n_tiles+1] exclusive prefix of ccnt (K3 general path)
  uint32_t* nc_cur;        // of THIS chunk: [0] listed requests, [1] bucket overflows (K1 resets, K2 counts),
                           //                [2] a writer exists (K1 sets; the NEXT launch's K1 clears it)
  uint32_t* nc_ord;        // same, of the chunk whose listed requests are replayed by this launch
  uint8_t* ord_resp;       // reply array of that chunk (K2 left the listed requests' bytes there)
  uint32_t ord_pending;    // 1: a previous chunk still has listed requests to replay (done inside K1)
  uint64_t* buckets;       // [2^bucket_log2][kBucketCap] (group << 32 | index), filled by K2
  uint32_t* bcnt;          // [2^bucket_log2]
  uint32_t bucket_log2;
  uint64_t* sortA;         // [chunk] (group << 32 | index)
  uint64_t* sortB;
  uint32_t* ghist;         // [256][sort tiles]
  uint32_t* rowtot;        // [256]
  uint32_t sort_passes;    // 8-bit digits covering the group-id bits
  // sharding of the group space
  FastMod shard_div;       // n_shards
  uint32_t n_shards, shard_id;
  // lock tables (lock_2pl / lock_fasst)
  FastMod slot_mod;        // kLockHashSize
  uint32_t* lockbits;      // fasst / tatp: 1 bit per group
  uint32_t* ver;           // fasst: u32 per slot
  uint2* cnt2;             // lock_2pl / smallbank: {num_ex, num_sh} per group
  // KV
  KvTable tbl[kMaxTables];
  uint32_t n_tables;
  // log
  uint8_t* ring;
  uint32_t ring_n;
  uint32_t* log_tilecnt;   // [n_tiles] log appends per tile (K1)
  unsigned long long* log_tilebase;  // [n_tiles] absolute append ordinal of the tile's first append (K1b)
  unsigned long long* log_total;     // [2]: [0] appends before this chunk ... running total, [1] this chunk's total
  // bookkeeping
  unsigned long long* counters;   // [0] errors [1] conflicted [2] max_run [3] chunks replayed by the radix fallback
  uint32_t* gbar;                 // k_ordered's grid barrier when it is not launched cooperatively
  uint32_t coop_launch;           // 1: k_ordered was launched cooperatively
  // where the replies go.  Default: `resp`, one contiguous array.  Inside the multi-GPU step the batch is W source
  // slabs of seg_tiles tiles each and the replies of slab s are stored straight into source s's return buffer over
  // NVLink (seg_resp[s]; posted stores), so no separate push / pull pass exists.
  const uint8_t* ord_req;         // request array of the chunk being replayed (replies may live in remote memory)
  uint32_t seg_tiles;             // tiles per source slab; 0 = contiguous replies
  uint32_t tile0, ord_tile0;      // index, inside the batch, of the first tile of this chunk / of the replayed chunk
  uint32_t pad_ok;                // 1 inside the multi-GPU step: type 0xFE records are slab padding (else: invalid)
  uint64_t seg_resp[8];           // reply slab of source s (device address, possibly peer memory)
  const uint32_t* skip;           // multi-GPU step: non-zero = a slab overflowed, serve nothing more (see k_p2p_wait)
};

// address of tile T's replies (T counted from the start of the batch) when the replies are segmented by source
template <int MSG> DINT_D uint8_t* seg_tile_ptr(const Ctx& c, uint32_t T) {
  const uint32_t s = T / c.seg_tiles;
  return (uint8_t*)c.seg_resp[s] + (size_t)(T - s * c.seg_tiles) * (kTile * MSG);
}
// address of the reply of record `idx` of the chunk being replayed
template <int MSG> DINT_D uint8_t* ord_out_ptr(const Ctx& c, uint32_t idx) {
  if (c.seg_tiles) return seg_tile_ptr<MSG>(c, c.ord_tile0 + idx / kTile) + (size_t)(idx % kTile) * MSG;
  return c.ord_resp + (size_t)idx * MSG;
}

// ---- bitmap helpers -------------------------------------------------------------------------------
DINT_D bool bm_test(const uint32_t* bm, uint32_t g) { return (bm[g >> 5] >> (g & 31)) & 1u; }
DINT_D void bm_set(uint32_t* bm, uint32_t g) { atomicOr(&bm[g >> 5], 1u << (g & 31)); }
DINT_D uint32_t bm_fetch_set(uint32_t* bm, uint32_t g) {
  uint32_t bit = 1u << (g & 31);
  return atomicOr(&bm[g >> 5], bit) & bit;
}
DINT_D void bm_clear_bit(uint32_t* bm, uint32_t g) { atomicAnd(&bm[g >> 5], ~(1u << (g & 31))); }

// flag nibble of group g inside a flag set
DINT_D uint32_t flag_word(const Ctx& c, uint32_t g) { return (g & c.flags_mask) >> 3; }
DINT_D uint32_t flag_shift(uint32_t g) { return (g & 7u) * 4u; }

// global group id -> local group id of this shard (owner = global % n_shards)
DINT_D bool to_local_group(const Ctx& c, uint32_t gglobal, uint32_t& glocal) {
  if (c.n_shards == 1) { glocal = gglobal; return true; }
  uint32_t q = (uint32_t)fast_div(gglobal, c.shard_div);
  glocal = q;
  return gglobal - q * c.n_shards == c.shard_id;
}

// ---- decode: what a wire record touches (type_info, cheap) and where (key_info, hashes) -----------
struct TypeInfo {
  uint32_t mask;    // C_RA | C_WA | C_WL
  bool invalid;     // the reference would panic() on this record
  bool is_log;      // appends to the commit log
};
struct KeyInfo {
  uint64_t key;     // lock id / KV key
  uint64_t h;       // fasthash64 of it (KV kinds: also picks the table entry)
  uint32_t grp;     // local group id, kNoGroup when the record is not this shard's
};
constexpr uint32_t kNoGroup = 0xffffffffu;
// Padding record of the fixed-capacity multi-GPU exchange (shard.py): type byte 0xFE, no reference server
// ever sees it.  It touches nothing, is answered unchanged, and is not an error.
constexpr uint8_t kPadType = 0xFE;

template <int KIND> DINT_D TypeInfo type_info(const uint8_t* rec);
template <int KIND> DINT_D KeyInfo key_info(const Ctx& c, const uint8_t* rec);

// State fetched BEFORE the conflict decision is known, so that its HBM latency overlaps the flag
// lookup instead of following it (see k_apply).  Never trusted across a write to the same group:
// K3 re-fetches immediately before every replayed request.
template <int KIND> struct Pre;
template <int KIND> DINT_D Pre<KIND> prefetch(const Ctx& c, const uint8_t* rec, const KeyInfo& ki, const TypeInfo& ti);
// Warp-wide variant used by k_apply: called by all 32 lanes (`active` = this lane has a request to fetch
// for).  The KV kinds fetch table entries with several adjacent lanes per entry, so that an entry is ONE
// 64-byte memory request instead of four 16-byte ones: random-access throughput on this chip is bounded
// by outstanding requests per SM, not by bytes (tools/ubench.cu).
template <int KIND>
DINT_D Pre<KIND> prefetch_coop(const Ctx& c, const uint8_t* rec, const KeyInfo& ki, const TypeInfo& ti, bool active);

// apply_one: the request semantics, in place on the wire record.  `rec` holds the request and becomes
// the reply (the reference mutates the received buffer and sends it back: lock_fasst/udp/server.cc:87-89).
// The caller guarantees that nothing else touches the same resource of the group concurrently.
// log_ord: absolute append ordinal for log requests (ring index = ord % ring_n); log_keep: false when a
// later append of the same chunk lands on the same ring entry.
template <int KIND>
DINT_D void apply_one(const Ctx& c, uint8_t* rec, const KeyInfo& ki, const Pre<KIND>& pf, unsigned long long log_ord,
                      bool log_keep);

// marks a record as "the reference would panic() here" (SURVEY.md section 8(b), errors row)
template <int KIND> DINT_D void mark_invalid(const Ctx& c, uint8_t* rec) {
  rec[Wire<KIND>::TYPE] = 0xFF;
  atomicAdd(&c.counters[0], 1ULL);
}

// Register-resident replay of a same-group run (K3).  For the lock servers a group's whole state is a
// couple of words, so a run need not be replayed request by request against memory: every request's
// fields are fetched up front IN PARALLEL (load_op), the run's owner walks the ops with the state in
// registers (step), and the replies are written back IN PARALLEL (write_result) -- three memory round
// trips per run instead of three per request.
template <int KIND> struct FastReplay { static constexpr bool ok = false; };

// =================================== lock_2pl =========================================================
template <> DINT_D TypeInfo type_info<K_LOCK2PL>(const uint8_t* rec) {
  using W = Wire<K_LOCK2PL>;
  uint8_t action = rec[W::TYPE], lt = rec[W::LTYPE];
  // lock_2pl/udp/server.cc:82,109,112,121: acquire needs a valid lock type, release accepts any
  if (action > 1 || (action == 0 && lt > 1)) return TypeInfo{0, true, false};
  return TypeInfo{C_WL, false, false};   // every lock_2pl request reads or changes the slot's counters
}
template <> DINT_D KeyInfo key_info<K_LOCK2PL>(const Ctx& c, const uint8_t* rec) {
  KeyInfo k;
  k.key = ld_u32_unaligned(rec + Wire<K_LOCK2PL>::KEY);
  k.h = fasthash64_u32((uint32_t)k.key);                                  // server.cc:71
  if (!to_local_group(c, fast_mod(k.h, c.slot_mod), k.grp)) k.grp = kNoGroup;   // :72
  return k;
}
template <> struct Pre<K_LOCK2PL> { uint2 s; };
template <> DINT_D Pre<K_LOCK2PL> prefetch<K_LOCK2PL>(const Ctx& c, const uint8_t*, const KeyInfo& ki, const TypeInfo&) {
  return Pre<K_LOCK2PL>{__ldcg(&c.cnt2[ki.grp])};
}
template <> DINT_D Pre<K_LOCK2PL> prefetch_coop<K_LOCK2PL>(const Ctx& c, const uint8_t* rec, const KeyInfo& ki, const TypeInfo& ti, bool active) {
  return active ? prefetch<K_LOCK2PL>(c, rec, ki, ti) : Pre<K_LOCK2PL>{make_uint2(0, 0)};
}
template <>
DINT_D void apply_one<K_LOCK2PL>(const Ctx& c, uint8_t* rec, const KeyInfo& ki, const Pre<K_LOCK2PL>& pf,
                                 unsigned long long, bool) {
  using W = Wire<K_LOCK2PL>;
  const uint32_t g = ki.grp;
  uint8_t action = rec[W::TYPE], lt = rec[W::LTYPE];
  uint2 s = pf.s;                          // x = num_ex, y = num_sh
  if (action == 0) {                       // kAcquireLock, lock_2pl/udp/server.cc:82-110
    if (lt == 0) {                         // kShared :83-93
      if (s.x == 0) { s.y++; c.cnt2[g] = s; rec[W::TYPE] = 2; } else rec[W::TYPE] = 3;
    } else {                               // kExclusive :96-107
      if (s.x == 0 && s.y == 0) { s.x++; c.cnt2[g] = s; rec[W::TYPE] = 2; } else rec[W::TYPE] = 3;
    }
  } else {                                 // kReleaseLock :112-119 (u32 wrap-around preserved)
    if (lt == 0) { s.y--; c.cnt2[g] = s; }
    else if (lt == 1) { s.x--; c.cnt2[g] = s; }
    rec[W::TYPE] = 5;                      // kReleaseAck
  }
}

template <> struct FastReplay<K_LOCK2PL> {
  static constexpr bool ok = true;
  using W = Wire<K_LOCK2PL>;
  struct State { uint2 s; };
  static DINT_D uint32_t load_op(const uint8_t* rec) { return (uint32_t)rec[W::TYPE] | ((uint32_t)rec[W::LTYPE] << 8); }
  static DINT_D State load_state(const Ctx& c, uint32_t g) { return State{__ldcg(&c.cnt2[g])}; }
  static DINT_D void store_state(const Ctx& c, uint32_t g, const State& st) { c.cnt2[g] = st.s; }
  static DINT_D uint64_t step(State& st, uint32_t op) {             // lock_2pl/udp/server.cc:82-119
    const uint32_t action = op & 255u, lt = op >> 8;
    if (action == 0) {
      if (lt == 0) { if (st.s.x == 0) { st.s.y++; return 2; } return 3; }
      if (st.s.x == 0 && st.s.y == 0) { st.s.x++; return 2; }
      return 3;
    }
    if (lt == 0) st.s.y--; else if (lt == 1) st.s.x--;
    return 5;
  }
  static DINT_D void write_result(uint8_t* rec, uint64_t r) { rec[W::TYPE] = (uint8_t)r; }
};

// =================================== lock_fasst =======================================================
template <> DINT_D TypeInfo type_info<K_FASST>(const uint8_t* rec) {
  uint8_t t = rec[Wire<K_FASST>::TYPE];
  if (t > 3) return TypeInfo{0, true, false};               // lock_fasst/udp/server.cc:116-117
  // kRead reads ver_table; kAcquireLock / kAbort CAS the lock word; kCommit does ver++ and the CAS
  return TypeInfo{(t == 0) ? C_RA : (t == 3) ? (C_WA | C_WL) : C_WL, false, false};
}
template <> DINT_D KeyInfo key_info<K_FASST>(const Ctx& c, const uint8_t* rec) {
  KeyInfo k;
  k.key = ld_u32_unaligned(rec + Wire<K_FASST>::KEY);
  k.h = fasthash64_u32((uint32_t)k.key);                                  // server.cc:81
  if (!to_local_group(c, fast_mod(k.h, c.slot_mod), k.grp)) k.grp = kNoGroup;   // :82
  return k;
}
// The version of a lock_fasst slot: `ver` u32 per slot (144 MB at 36 M slots -- every READ costs one 64-byte HBM burst
// for 4 bytes used).  A 16-bit hot array + cold high bits was measured (round 2, profiles/r02_variants.md): K2 -6 %,
// step -2.4 %, and it degenerates to two accesses once a slot has seen 32768 commits (minutes of service): dropped.
DINT_D uint32_t ver_load(const Ctx& c, uint32_t g) { return __ldcg(&c.ver[g]); }
DINT_D void ver_store(const Ctx& c, uint32_t g, uint32_t v) { c.ver[g] = v; }
template <> struct Pre<K_FASST> { uint32_t ver; };
template <> DINT_D Pre<K_FASST> prefetch<K_FASST>(const Ctx& c, const uint8_t*, const KeyInfo& ki, const TypeInfo& ti) {
  return Pre<K_FASST>{(ti.mask & (C_RA | C_WA)) ? ver_load(c, ki.grp) : 0u};
}
template <> DINT_D Pre<K_FASST> prefetch_coop<K_FASST>(const Ctx& c, const uint8_t* rec, const KeyInfo& ki, const TypeInfo& ti, bool active) {
  return active ? prefetch<K_FASST>(c, rec, ki, ti) : Pre<K_FASST>{0u};
}
template <>
DINT_D void apply_one<K_FASST>(const Ctx& c, uint8_t* rec, const KeyInfo& ki, const Pre<K_FASST>& pf,
                               unsigned long long, bool) {
  using W = Wire<K_FASST>;
  const uint32_t g = ki.grp;
  uint8_t t = rec[W::TYPE];
  if (t == 0) {                            // kRead, lock_fasst/udp/server.cc:86-90
    st_u32_unaligned(rec + W::VER, pf.ver);
    rec[W::TYPE] = 4;
  } else if (t == 1) {                     // kAcquireLock :92-101  CAS(0 -> 1)
    rec[W::TYPE] = bm_fetch_set(c.lockbits, g) ? 6 : 5;
  } else if (t == 2) {                     // kAbort :103-107       CAS(1 -> 0)
    bm_clear_bit(c.lockbits, g);
    rec[W::TYPE] = 7;
  } else {                                 // kCommit :109-114      ver++, CAS(1 -> 0)
    ver_store(c, g, pf.ver + 1);
    bm_clear_bit(c.lockbits, g);
    rec[W::TYPE] = 8;
  }
}

template <> struct FastReplay<K_FASST> {
  static constexpr bool ok = true;
  using W = Wire<K_FASST>;
  struct State { uint32_t ver, lock, g; bool dirty_ver; };
  static DINT_D uint32_t load_op(const uint8_t* rec) { return rec[W::TYPE]; }
  static DINT_D State load_state(const Ctx& c, uint32_t g) {
    return State{ver_load(c, g), (__ldcg(&c.lockbits[g >> 5]) >> (g & 31)) & 1u, g, false};
  }
  static DINT_D void store_state(const Ctx& c, uint32_t g, const State& st) {
    if (st.dirty_ver) ver_store(c, g, st.ver);
    if (st.lock) bm_set(c.lockbits, g); else bm_clear_bit(c.lockbits, g);   // neighbours share the word: atomics
  }
  static DINT_D uint64_t step(State& st, uint32_t t) {               // lock_fasst/udp/server.cc:86-114
    if (t == 0) return 4ull | ((uint64_t)st.ver << 8);
    if (t == 1) { if (st.lock) return 6; st.lock = 1; return 5; }
    if (t == 2) { st.lock = 0; return 7; }
    st.ver++; st.dirty_ver = true; st.lock = 0;
    return 8;
  }
  static DINT_D void write_result(uint8_t* rec, uint64_t r) {
    rec[W::TYPE] = (uint8_t)r;
    if ((uint8_t)r == 4) st_u32_unaligned(rec + W::VER, (uint32_t)(r >> 8));
  }
};

// =================================== log_server =======================================================
template <> DINT_D TypeInfo type_info<K_LOG>(const uint8_t* rec) {
  if (rec[Wire<K_LOG>::TYPE] != 0) return TypeInfo{0, true, false};   // log_server/udp/server.cc:76-77
  return TypeInfo{0, false, true};
}
template <> DINT_D KeyInfo key_info<K_LOG>(const Ctx&, const uint8_t*) { return KeyInfo{0, 0, kNoGroup}; }
template <> struct Pre<K_LOG> {};
template <> DINT_D Pre<K_LOG> prefetch<K_LOG>(const Ctx&, const uint8_t*, const KeyInfo&, const TypeInfo&) { return {}; }
template <> DINT_D Pre<K_LOG> prefetch_coop<K_LOG>(const Ctx&, const uint8_t*, const KeyInfo&, const TypeInfo&, bool) { return {}; }
template <>
DINT_D void apply_one<K_LOG>(const Ctx& c, uint8_t* rec, const KeyInfo&, const Pre<K_LOG>&, unsigned long long ord,
                             bool keep) {
  using W = Wire<K_LOG>;
  if (keep) {                              // log_server/udp/server.cc:79-84; entry {key@0 val@8 ver@48}
    uint8_t* e = c.ring + (size_t)(ord % c.ring_n) * W::LOGENT;
    uint32_t w[13];                        // key(2) + val(10) + ver(1) are contiguous on the wire
    ld_words_unaligned<13>(rec + W::KEY, w);
    uint2* e8 = (uint2*)e;
#pragma unroll
    for (int i = 0; i < 6; i++) e8[i] = make_uint2(w[2 * i], w[2 * i + 1]);
    *(uint32_t*)(e + 48) = w[12];
  }
  rec[W::TYPE] = 1;                        // kAck :86
}

}  // namespace dint
