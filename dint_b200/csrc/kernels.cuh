// kernels.cuh -- the three launches of a chunk (see engine.cuh for the scheme).
#pragma once
#include <cooperative_groups.h>
#include "engine.cuh"

namespace dint {
namespace cg = cooperative_groups;

DINT_D uint32_t lane_id() { return threadIdx.x & 31; }
DINT_D uint32_t warp_id() { return threadIdx.x >> 5; }

// In-tile exclusive rank of `flag` in thread order; returns rank, writes the tile total to `total`.
// `scratch` is kTile/32 words of shared memory.  Contains __syncthreads().  (K1/K2 only: kTile threads)
DINT_D uint32_t tile_rank(bool flag, uint32_t* scratch, uint32_t& total) {
  uint32_t bal = __ballot_sync(0xffffffffu, flag);
  uint32_t in_warp = __popc(bal & ((1u << lane_id()) - 1u));
  if (lane_id() == 0) scratch[warp_id()] = __popc(bal);
  __syncthreads();
  uint32_t off = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kTile / 32; w++) {
    uint32_t v = scratch[w];
    if (w < (int)warp_id()) off += v;
    tot += v;
  }
  __syncthreads();
  total = tot;
  return off + in_warp;
}

// Two ranks with ONE barrier (flag a in the low half-word of the per-warp counts, b in the high).
DINT_D void tile_rank2(bool a, bool b, uint32_t* scratch, uint32_t& ra, uint32_t& rb, uint32_t& ta, uint32_t& tb) {
  const uint32_t ba = __ballot_sync(0xffffffffu, a), bb = __ballot_sync(0xffffffffu, b);
  const uint32_t lt = (1u << lane_id()) - 1u;
  if (lane_id() == 0) scratch[warp_id()] = __popc(ba) | (__popc(bb) << 16);
  __syncthreads();
  uint32_t off = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < kTile / 32; w++) {
    uint32_t v = scratch[w];
    if (w < (int)warp_id()) off += v;
    tot += v;
  }
  // no trailing barrier: the caller alternates between two scratch arrays and has a CTA barrier per tile
  ra = (off & 0xffffu) + __popc(ba & lt);
  rb = (off >> 16) + __popc(bb & lt);
  ta = tot & 0xffffu;
  tb = tot >> 16;
}

DINT_D uint32_t bucket_of(uint32_t g, uint32_t log2p) { return log2p ? (g * 0x9E3779B1u) >> (32 - log2p) : 0; }

// bytes of one pipeline stage: a tile of wire records, padded so every stage stays 128-byte aligned
template <int MSG> struct Stage {
  static constexpr uint32_t BYTES = ((kTile * MSG + 16 + 127) / 128) * 128;
  // pipeline depth: big records get 2 stages so that 8 CTAs (2048 threads) still fit in one SM's shared memory
  static constexpr uint32_t N = (BYTES > 8192) ? 2 : kStages;
};

// Persistent-CTA tile pipeline: CTA b owns tiles b, b + gridDim.x, ...; thread 0 keeps kStages - 1 TMA bulk loads in
// flight ahead of the tile being processed.  (Dynamic assignment by a ticket counter was built and measured in round 2,
// profiles/r02_variants.md: +17 % with the ticket drawn at the point of use, +5-7 % with the draw one iteration ahead,
// and NO gain inside the multi-GPU step it was meant for -- 145.7 vs 144.5 us per batch at N = 2 -- because the kernels
// of the step compete for the memory system, not for SM slots.  Dropped.)
struct TileIter {
  uint32_t n_my;        // tiles owned by this CTA
  DINT_D uint32_t tile(uint32_t i) const { return blockIdx.x + i * gridDim.x; }
  DINT_D bool has(uint32_t i) const { return i < n_my; }
};
DINT_D TileIter tile_iter(uint32_t n_tiles) {
  TileIter it;
  it.n_my = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  return it;
}
template <int MSG>
DINT_D void issue_tile_load(const Ctx& c, uint8_t* smem, uint64_t* full, const TileIter& it, uint32_t i) {
  const uint32_t t = it.tile(i), first = t * kTile;
  const uint32_t cnt = min((uint32_t)kTile, c.n - first);
  const uint32_t body = (cnt * MSG) & ~15u;
  const uint32_t buf = i % Stage<MSG>::N;
  if (body) {
    mbar_expect_tx(&full[buf], body);
    tma_load_1d(smem + buf * Stage<MSG>::BYTES, c.req + (size_t)first * MSG, body, &full[buf]);
  }
}
// all threads: wait for tile i's bulk load, fetch the (<16-byte) tail of the very last tile by hand
template <int MSG>
DINT_D uint8_t* acquire_tile(const Ctx& c, uint8_t* smem, uint64_t* full, const TileIter& it, uint32_t i,
                             uint32_t& first, uint32_t& cnt) {
  const uint32_t t = it.tile(i);
  first = t * kTile;
  cnt = min((uint32_t)kTile, c.n - first);
  const uint32_t bytes = cnt * MSG, body = bytes & ~15u;
  uint8_t* tile = smem + (i % Stage<MSG>::N) * Stage<MSG>::BYTES;
  if (body) mbar_wait(&full[i % Stage<MSG>::N], (i / Stage<MSG>::N) & 1u);
  if (body != bytes) {
    const uint8_t* src = c.req + (size_t)first * MSG;
    for (uint32_t b = body + threadIdx.x; b < bytes; b += blockDim.x) tile[b] = src[b];
    __syncthreads();
  }
  return tile;
}

// the shard that owns a request: the slot / bucket / lock_hash ONE server would compute, modulo the shard count
template <int KIND>
DINT_D uint32_t route_owner_of(const Ctx& c, const uint8_t* rec) {
  using W = Wire<KIND>;
  const TypeInfo ti = type_info<KIND>(rec);
  if (ti.invalid || !ti.mask) return c.shard_id;         // no per-key state touched: serve it where it arrived
  uint32_t gglobal = 0;
  if constexpr (KIND == K_LOCK2PL || KIND == K_FASST) gglobal = fast_mod(fasthash64_u32(ld_u32_unaligned(rec + W::KEY)), c.slot_mod);
  else if constexpr (KIND == K_STORE) gglobal = fast_mod(fasthash64_u64(ld_u64_unaligned(rec + W::KEY)), c.tbl[0].lock_mod);
  else if constexpr (KIND == K_TATP || KIND == K_SMALLBANK) gglobal = fast_mod(fasthash64_u64(ld_u64_unaligned(rec + W::KEY)), c.tbl[rec[W::TABLE]].lock_mod);
  else return c.shard_id;
  return gglobal - (uint32_t)fast_div(gglobal, c.shard_div) * c.n_shards;
}
// owner shard of every request (multi-GPU routing; see dint_route_owner)
template <int KIND>
__global__ void __launch_bounds__(kThreads) k_route_owner(const Ctx c, const uint8_t* req, uint32_t n, uint8_t* owner) {
  const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
  if (i < n) owner[i] = (uint8_t)route_owner_of<KIND>(c, req + (size_t)i * Wire<KIND>::MSG);
}

// ---- multi-GPU dispatch: stable partition of a batch by owner shard -------------------------------------
// (1) k_route_count: per 256-record tile, how many records go to each shard;  (2) k_exact_scan (one CTA):
// exclusive offsets -- shard-major, then tile order -- and the per-shard totals;  (3) k_route_scatter: every
// record is copied to its slot (stable inside a shard: tile order, then thread order) and the inverse
// permutation is recorded.  Afterwards the wire records sit grouped by destination, ready for the exchange.
constexpr int kMaxShards = 8;
__global__ void __launch_bounds__(kThreads) k_exact_count(const uint8_t* owner, uint32_t n, uint32_t world, uint32_t* tilecnt) {
  __shared__ uint32_t cnt[kMaxShards];
  if (threadIdx.x < kMaxShards) cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
  const uint32_t o = i < n ? owner[i] : 0xffu;
  const uint32_t peers = __match_any_sync(0xffffffffu, o);
  if (o < world && (int)lane_id() == __ffs(peers) - 1) atomicAdd(&cnt[o], (uint32_t)__popc(peers));
  __syncthreads();
  if (threadIdx.x < world) tilecnt[(size_t)threadIdx.x * gridDim.x + blockIdx.x] = cnt[threadIdx.x];   // shard-major
}
__global__ void __launch_bounds__(kThreads) k_exact_scan(uint32_t* tilecnt, uint32_t n_tiles, uint32_t* totals) {
  // one CTA per shard: exclusive scan of that shard's row of per-tile counts, row total -> totals[shard]
  __shared__ uint32_t wsum[kThreads / 32];
  __shared__ uint32_t carry;
  uint32_t* row = tilecnt + (size_t)blockIdx.x * n_tiles;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (uint32_t base = 0; base < n_tiles; base += kThreads) {
    const uint32_t i = base + threadIdx.x;
    const uint32_t v = i < n_tiles ? row[i] : 0;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
      if ((int)lane_id() >= o) x += y;
    }
    if (lane_id() == 31) wsum[warp_id()] = x;
    __syncthreads();
    uint32_t woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; w++) {
      if (w < (int)warp_id()) woff += wsum[w];
      tot += wsum[w];
    }
    if (i < n_tiles) row[i] = carry + woff + (x - v);
    __syncthreads();
    if (threadIdx.x == 0) carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) totals[blockIdx.x] = carry;
}
template <int MSG>
__global__ void __launch_bounds__(kThreads) k_exact_scatter(const uint8_t* req, const uint8_t* owner, uint32_t n, uint32_t world,
                                                            const uint32_t* tilebase, const uint32_t* totals, uint8_t* out,
                                                            uint32_t* perm) {
  __shared__ uint32_t wcnt[kThreads / 32][kMaxShards];
  const uint32_t i = blockIdx.x * kThreads + threadIdx.x;
  if (threadIdx.x < (kThreads / 32) * kMaxShards) ((uint32_t*)wcnt)[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t o = i < n ? owner[i] : 0xffu;
  const uint32_t peers = __match_any_sync(0xffffffffu, o);
  const uint32_t before = __popc(peers & ((1u << lane_id()) - 1u));
  if (o < world && before == 0) wcnt[warp_id()][o] = __popc(peers);
  __syncthreads();
  if (o < world) {
    uint32_t pos = tilebase[(size_t)o * gridDim.x + blockIdx.x] + before;
    for (uint32_t w = 0; w < warp_id(); w++) pos += wcnt[w][o];
    for (uint32_t q = 0; q < o; q++) pos += totals[q];                 // start of shard o's segment
    copy_record<MSG>(out + (size_t)pos * MSG, req + (size_t)i * MSG);
    perm[pos] = i;
  }
}
// ---- exchange over NVLink peer memory: epoch flags ---------------------------------------------------------
// Every rank owns a buffer {inbox[world][cap], return buffer[world][cap], signals} that its peers map (torch symmetric
// memory / CUDA IPC / peer access).  The dispatch kernel (route.cuh) stores each record straight into the OWNER's inbox
// slab for this source, the owner's k_apply stores each reply tile straight into the SOURCE's return buffer.
// Ordering across GPUs: epoch counters written with system-scope release stores after the data and polled
// with acquire loads.
struct PeerPtrs { uint64_t p[kMaxShards]; };

// after the data: tell every peer that epoch `e` of this rank's slab is complete
__global__ void k_p2p_signal(PeerPtrs sig, uint32_t world, uint32_t me, uint32_t epoch) {
  if (threadIdx.x < world) {
    __threadfence_system();
    volatile uint32_t* flag = (volatile uint32_t*)sig.p[threadIdx.x] + me;
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
  }
}
// before consuming: wait until every peer has signalled epoch `e` (bounded spin: ~4 s, then *timeout = 1).
// Bit 31 of a request flag = "this source could not fit one of its slabs": the first epoch for which any source says so
// is recorded in *bad (0 = none), and from then on every engine launch of the step returns at once (Ctx::skip): the
// batch and everything behind it is left unserved on EVERY shard -- all owners see all sources' flags -- so the server
// state stays consistent and the host can serve those records again in smaller rounds.
constexpr uint32_t kSigOverflow = 0x80000000u;
__global__ void k_p2p_wait(const uint32_t* my_sig, uint32_t world, uint32_t epoch, uint32_t* timeout, uint32_t* bad) {
  if (threadIdx.x < world) {
    const long long t0 = clock64();
    uint32_t v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(my_sig + threadIdx.x) : "memory");
      if (clock64() - t0 > 8000000000LL) { atomicExch(timeout, 1u); break; }
    } while ((int32_t)((v & ~kSigOverflow) - epoch) < 0);
    if (bad && (v & kSigOverflow) && (v & ~kSigOverflow) == epoch) atomicCAS(bad, 0u, epoch);
  }
  __syncthreads();
  __threadfence_system();
}

// combine: replies arrive in partition order; put each back at its original index
template <int MSG>
__global__ void __launch_bounds__(kThreads) k_exact_unpermute(const uint8_t* sorted, const uint32_t* perm, uint32_t n, uint8_t* out) {
  const uint32_t pos = blockIdx.x * kThreads + threadIdx.x;
  if (pos >= n) return;
  const uint32_t idx = perm[pos];
  if (idx == 0xffffffffu) return;                        // padding slot of a slab
  copy_record<MSG>(out + (size_t)idx * MSG, sorted + (size_t)pos * MSG);
}

// ordered replay (defined below): per-warp shared-memory slice and the replay itself
template <int KIND> struct OrdSlice {
  static constexpr uint32_t BYTES = kBucketCap * (FastReplay<KIND>::ok ? (8 + 8 + 4) : 8);
};
template <int KIND> DINT_D void ordered_buckets(const Ctx& c, uint8_t* scratch);

// ---------------------------------------------------------------------------------------------------
// K1 classify (+ clears the flag words of the previous chunk)
// ---------------------------------------------------------------------------------------------------
template <int KIND, bool HAS_LOG>
__global__ void __launch_bounds__(kTile) k_classify(const Ctx c) {
  using W = Wire<KIND>;
  constexpr uint32_t NS = Stage<W::MSG>::N;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t full[kStages];
  __shared__ uint32_t scratch[kTile / 32];
  if (c.skip && __ldcg(c.skip)) return;                  // the multi-GPU step is draining after a slab overflow (k_p2p_wait)
  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; s++) mbar_init(&full[s], 1);
    // [2] (a writer exists) is OR-ed by any CTA of this launch, so it is cleared one launch early: each K1
    // clears the slot of the chunk it replays, which is the slot the NEXT chunk will use
    if (blockIdx.x == 0) { c.nc_cur[0] = 0; c.nc_cur[1] = 0; c.nc_ord[2] = 0; }
  }
  __syncthreads();
  // The previous chunk's listed requests are replayed by this launch too (their buckets were filled by its
  // K2; a bucket overflow was already handled by the fallback launch).  Odd CTAs replay first and classify
  // afterwards, even CTAs the other way round, so the latency-bound replay overlaps classification.
  const bool do_ord = c.ord_pending && c.nc_ord[0] != 0 && c.nc_ord[1] == 0;
  const bool ord_first = (blockIdx.x & 1u) != 0;
  if (do_ord && ord_first) {
    ordered_buckets<KIND>(c, smem);
    __syncthreads();
  }
  const TileIter it = tile_iter(c.n_tiles);
  if (threadIdx.x == 0)
    for (uint32_t i = 0; i < NS && i < it.n_my; i++) issue_tile_load<W::MSG>(c, smem, full, it, i);

  // retire the previous chunk's flags: every word it touched is zeroed (all of that set's nibbles
  // were written by that chunk, so whole-word stores are exact).  Loads are batched four deep so that
  // the kernel start pays one memory latency, not one per element.
  for (uint32_t i = blockIdx.x * kTile + threadIdx.x; i < c.prev_n; i += 4 * gridDim.x * kTile) {
    uint32_t g[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const uint32_t j = i + u * gridDim.x * kTile;
      g[u] = j < c.prev_n ? __ldcg(&c.grp_prev[j]) : kNoGroup;
    }
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (g[u] != kNoGroup) c.flags_prev[flag_word(c, g[u])] = 0;
  }

  // A writer needs the OLD nibble to learn whether it is the second writer of its class (-> W2).  Waiting
  // for the atomic's return value would expose one L2 round trip per tile; the check is deferred by one
  // tile instead (the value is consumed after the NEXT tile's atomics have been issued).
  uint32_t pend_old = 0, pend_test = 0, pend_sh = 0;
  uint32_t* pend_w = nullptr;
  bool saw_writer = false;          // any request of this CTA's tiles that writes A or L
  for (uint32_t i = 0; it.has(i); i++) {
    // the stage that held tile i-1 is free (barrier at the end of iteration i-1): refill it now
    if (threadIdx.x == 0 && i && i + NS - 1 < it.n_my) issue_tile_load<W::MSG>(c, smem, full, it, i + NS - 1);
    uint32_t first, cnt;
    const uint8_t* tile = acquire_tile<W::MSG>(c, smem, full, it, i, first, cnt);
    const bool valid = threadIdx.x < cnt;
    bool is_log = false;
    uint32_t new_old = 0, new_test = 0, new_sh = 0;
    uint32_t* new_w = nullptr;
    if (valid) {
      const uint8_t* rec = tile + threadIdx.x * W::MSG;
      TypeInfo ti = (c.pad_ok && rec[W::TYPE] == kPadType) ? TypeInfo{0, false, false} : type_info<KIND>(rec);
      uint32_t g = kNoGroup;
      if (!ti.invalid && ti.mask) {
        g = key_info<KIND>(c, rec).grp;
        if (g != kNoGroup) {
          uint32_t* w = &c.flags[flag_word(c, g)];
          const uint32_t sh = flag_shift(g);
          if (ti.mask == C_RA) {
            atomicOr(w, F_R << sh);                      // no return value: a fire-and-forget RED
          } else {
            const uint32_t bits = ((ti.mask & C_RA) ? F_R : 0u) | ((ti.mask & C_WA) ? F_WA : 0u) | ((ti.mask & C_WL) ? F_WL : 0u);
            saw_writer = true;
            new_old = atomicOr(w, bits << sh);
            new_test = ((ti.mask & C_WA) ? F_WA : 0u) | ((ti.mask & C_WL) ? F_WL : 0u);
            new_w = w;
            new_sh = sh;
          }
        }
      }
      c.grp[first + threadIdx.x] = g;
      is_log = !ti.invalid && ti.is_log;
    }
    if (pend_w && ((pend_old >> pend_sh) & pend_test)) atomicOr(pend_w, F_W2 << pend_sh);
    pend_old = new_old; pend_test = new_test; pend_sh = new_sh; pend_w = new_w;
    if (HAS_LOG) {
      uint32_t total;
      (void)tile_rank(is_log, scratch, total);          // contains the CTA barriers that free the stage
      if (threadIdx.x == 0) c.log_tilecnt[it.tile(i)] = total;
    } else {
      __syncthreads();                                   // everyone is done reading this stage
    }
  }
  if (pend_w && ((pend_old >> pend_sh) & pend_test)) atomicOr(pend_w, F_W2 << pend_sh);
  // a chunk without a single writer cannot hold a conflict: K2 then skips the flag lookups altogether
  if (__syncthreads_or(saw_writer ? 1 : 0) && threadIdx.x == 0) atomicOr(&c.nc_cur[2], 1u);
  if (do_ord && !ord_first) {
    __syncthreads();                                     // the stages double as the replay's scratch
    ordered_buckets<KIND>(c, smem);
  }
}

// K1b: absolute append ordinal of every tile's first log append (single CTA).
__global__ void __launch_bounds__(kThreads) k_log_scan(const Ctx c) {
  if (c.skip && __ldcg(c.skip)) return;
  __shared__ unsigned long long carry;
  __shared__ uint32_t wsum[kThreads / 32];
  if (threadIdx.x == 0) carry = c.log_total[0];
  __syncthreads();
  for (uint32_t base = 0; base < c.n_tiles; base += kThreads) {
    uint32_t i = base + threadIdx.x;
    uint32_t v = i < c.n_tiles ? c.log_tilecnt[i] : 0;
    uint32_t x = v;                       // inclusive warp scan
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
      if ((int)lane_id() >= o) x += y;
    }
    if (lane_id() == 31) wsum[warp_id()] = x;
    __syncthreads();
    uint32_t woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; w++) {
      if (w < (int)warp_id()) woff += wsum[w];
      tot += wsum[w];
    }
    if (i < c.n_tiles) c.log_tilebase[i] = carry + woff + (x - v);
    __syncthreads();
    if (threadIdx.x == 0) carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    c.log_total[1] = carry;               // end ordinal of this chunk
    c.log_total[0] = carry;               // base of the next chunk
  }
}

// ---------------------------------------------------------------------------------------------------
// K2 apply
// ---------------------------------------------------------------------------------------------------
// (register caps were tried for the KV servers: 48 registers / 10 CTAs per SM measured 10 % slower than the
// compiler's own 62 registers / 8 CTAs, and more registers / fewer CTAs slower still)
template <int KIND, bool HAS_LOG>
__global__ void __launch_bounds__(kTile) k_apply(const Ctx c) {
  using W = Wire<KIND>;
  constexpr uint32_t NS = Stage<W::MSG>::N;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ uint64_t full[kStages];
  __shared__ uint32_t scratch2[2][kTile / 32];
  // lock servers: the group id K1 stored is all K2 needs of the key -- fetch it (coalesced, independent of
  // the TMA stage) instead of re-hashing; KV servers need the hash itself to find the table entry
  constexpr bool kGrpFromK1 = (KIND == K_LOCK2PL || KIND == K_FASST);
  if (c.skip && __ldcg(c.skip)) return;
  if (threadIdx.x == 0)
    for (int s = 0; s < kStages; s++) mbar_init(&full[s], 1);
  __syncthreads();
  const TileIter it = tile_iter(c.n_tiles);
  if (threadIdx.x == 0)
    for (uint32_t i = 0; i < NS && i < it.n_my; i++) issue_tile_load<W::MSG>(c, smem, full, it, i);
  const bool chunk_has_writer = c.nc_cur[2] != 0;      // set by K1; false = nothing in this chunk can conflict

  for (uint32_t i = 0; it.has(i); i++) {
    uint32_t* scratch = scratch2[i & 1];
    uint32_t g_k1 = kNoGroup;
    if (kGrpFromK1) {
      const uint32_t idx = it.tile(i) * kTile + threadIdx.x;
      if (idx < c.n) g_k1 = __ldcg(&c.grp[idx]);
    }
    if (threadIdx.x == 0 && i && i + NS - 1 < it.n_my) {
      // the stage that held tile i-1 is refilled as soon as its bulk store has finished READING it
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
      issue_tile_load<W::MSG>(c, smem, full, it, i + NS - 1);
    }
    uint32_t first, cnt;
    uint8_t* tile = acquire_tile<W::MSG>(c, smem, full, it, i, first, cnt);
    const uint32_t t = it.tile(i);
    const bool valid = threadIdx.x < cnt;
    uint8_t* rec = tile + threadIdx.x * W::MSG;
    TypeInfo ti{0, false, false};
    KeyInfo ki{0, 0, kNoGroup};
    Pre<KIND> pf;
    bool listed = false;
    const bool pad = valid && c.pad_ok && rec[W::TYPE] == kPadType;
    if (valid && !pad) {
      ti = type_info<KIND>(rec);
      if (!ti.invalid && ti.mask) {
        if (kGrpFromK1) ki.grp = g_k1; else ki = key_info<KIND>(c, rec);
        if (ki.grp == kNoGroup) ti.invalid = true;   // not this shard's / bad table
      }
    }
    {
      // issue the state fetch and the flag lookup back to back: one HBM latency, not two
      const bool active = valid && !ti.invalid && ti.mask;
      pf = prefetch_coop<KIND>(c, rec, ki, ti, active);
      if (active && chunk_has_writer) {
        const uint32_t f = (__ldcg(&c.flags[flag_word(c, ki.grp)]) >> flag_shift(ki.grp)) & 15u;
        listed = ((ti.mask & C_RA) && (f & F_WA)) || ((ti.mask & C_WA) && (f & (F_R | F_W2))) ||
                 ((ti.mask & C_WL) && (f & F_W2));
      }
    }
    unsigned long long log_ord = 0;
    bool log_keep = false;
    {
      // listed requests: (a) the tile-segmented, index-ordered list (radix fallback of K3),
      //                  (b) the hash bucket K3 sorts in shared memory
      const bool lg = HAS_LOG && valid && !ti.invalid && ti.is_log;
      uint32_t r_list, r_log, n_list, n_log;
      tile_rank2(listed, lg, scratch, r_list, r_log, n_list, n_log);
      if (lg) {
        log_ord = c.log_tilebase[t] + r_log;
        log_keep = log_ord + c.ring_n >= c.log_total[1];   // no later append of this chunk overwrites it
      }
      if (listed) {
        const uint32_t idx = first + threadIdx.x;
        c.clist[(size_t)t * kTile + r_list] = idx;
        const uint32_t b = bucket_of(ki.grp, c.bucket_log2);
        const uint32_t pos = atomicAdd(&c.bcnt[b], 1u);
        if (pos < kBucketCap) c.buckets[(size_t)b * kBucketCap + pos] = ((uint64_t)ki.grp << 32) | idx;
        else atomicAdd(&c.nc_cur[1], 1u);
      }
      if (threadIdx.x == 0) {
        c.ccnt[t] = n_list;
        if (n_list) atomicAdd(&c.nc_cur[0], n_list);
      }
    }
    if (valid && !pad) {
      if (ti.invalid) mark_invalid<KIND>(c, rec);
      else if (!listed) apply_one<KIND>(c, rec, ki, pf, log_ord, log_keep);
      // listed: the record leaves this kernel unchanged; K3 rewrites it in place in resp
    }
    // ---- write the tile back; keep the load pipeline kStages - 1 tiles ahead ----
    const uint32_t bytes = cnt * W::MSG, body = bytes & ~15u;
    uint8_t* gdst = c.seg_tiles ? seg_tile_ptr<W::MSG>(c, c.tile0 + t) : c.resp + (size_t)first * W::MSG;
    fence_proxy_async_smem();
    __syncthreads();
    for (uint32_t b = body + threadIdx.x; b < bytes; b += blockDim.x) gdst[b] = tile[b];
    if (threadIdx.x == 0) {
      if (body) tma_store_1d(gdst, tile, body);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
  }
  if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---------------------------------------------------------------------------------------------------
// K3 ordered replay (cooperative launch: the whole grid is co-resident and uses grid-wide barriers)
// ---------------------------------------------------------------------------------------------------
constexpr int kSortItems = 8;                         // items per thread per radix tile
constexpr int kSortTile = kThreads * kSortItems;      // 2048

template <int KIND>
DINT_D void replay_run(const Ctx& c, const uint64_t* sorted, uint32_t p, uint32_t nc) {
  using W = Wire<KIND>;
  const uint32_t g = (uint32_t)(sorted[p] >> 32);
  uint32_t len = 0;
  for (uint32_t q = p; q < nc; q++) {
    uint64_t e = sorted[q];
    if ((uint32_t)(e >> 32) != g) break;
    // the request is applied on a private copy and leaves with word-wide stores: the reply array may be peer memory
    __align__(4) uint8_t rec[(W::MSG + 3) / 4 * 4];
    copy_record<W::MSG>(rec, c.ord_req + (size_t)(uint32_t)e * W::MSG);
    const TypeInfo ti = type_info<KIND>(rec);
    const KeyInfo ki = key_info<KIND>(c, rec);
    const Pre<KIND> pf = prefetch<KIND>(c, rec, ki, ti);      // fetched AFTER the previous request of the run
    apply_one<KIND>(c, rec, ki, pf, 0, false);
    copy_record<W::MSG>(ord_out_ptr<W::MSG>(c, (uint32_t)e), rec);
    len++;
  }
  if (len > 1) atomicMax(&c.counters[2], (unsigned long long)len);
}

// Ordered replay of the listed requests of a finished chunk (see engine.cuh).  Called by every warp of the
// grid; `scratch` = blockDim.x/32 slices of OrdSlice<KIND>::BYTES.
template <int KIND>
DINT_D void ordered_buckets(const Ctx& c, uint8_t* scratch) {
    // K2 already hashed every listed (group, index) pair into a bucket.  Warps work
    // independently (no CTA or grid barrier).  A warp task = `gsz` adjacent buckets (a power of two chosen
    // so that a task holds ~16 pairs: with few listed requests most buckets hold 0-2 pairs and one latency
    // chain per bucket would dominate).  The task's pairs are gathered into the warp's 256-key slice of
    // shared memory, sorted (rank sort by shuffles up to 32 keys, bitonic above; the keys carry the group
    // id in their high half, so pairs of different buckets may be sorted together) and replayed.
    uint64_t* wkeys = (uint64_t*)(scratch + (size_t)warp_id() * OrdSlice<KIND>::BYTES);
    uint64_t* wres = wkeys + kBucketCap;                       // fast replay only
    uint32_t* wops = (uint32_t*)(wkeys + 2 * kBucketCap);      // fast replay only
    const uint32_t lane = lane_id();
    const uint32_t warps_per_cta = blockDim.x / 32;
    const uint32_t n_warps = gridDim.x * warps_per_cta;
    const uint32_t P = 1u << c.bucket_log2;
    const uint32_t nc = c.nc_ord[0];
    uint32_t gsz = 1;
    while (gsz < 32 && (uint64_t)nc * gsz * 2 <= (uint64_t)16 * P) gsz <<= 1;      // mean pairs per task <= ~16
    const uint32_t n_tasks = (P + gsz - 1) / gsz;
    for (uint32_t task = blockIdx.x * warps_per_cta + warp_id(); task < n_tasks; task += n_warps) {
      const uint32_t b0 = task * gsz;
      const uint32_t myb = b0 + lane;
      const uint32_t cnt = (lane < gsz && myb < P) ? c.bcnt[myb] : 0;
      uint32_t incl = cnt;                                   // inclusive prefix over the task's buckets
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
        if ((int)lane >= o) incl += y;
      }
      const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
      if (total == 0) continue;
      // one pass when everything fits the slice, else bucket by bucket (each bucket alone always fits)
      const uint32_t n_pass = total <= kBucketCap ? 1 : gsz;
      for (uint32_t pass = 0; pass < n_pass; pass++) {
        uint32_t m;
        if (n_pass == 1) {
          m = total;
          for (uint32_t k = 0; k < gsz; k++) {               // gather bucket k at offset excl(k)
            const uint32_t ck = __shfl_sync(0xffffffffu, cnt, k);
            const uint32_t ek = __shfl_sync(0xffffffffu, incl, k) - ck;
            const uint64_t* src = c.buckets + (size_t)(b0 + k) * kBucketCap;
            for (uint32_t i = lane; i < ck; i += 32) wkeys[ek + i] = src[i];
          }
        } else {
          m = __shfl_sync(0xffffffffu, cnt, pass);
          const uint64_t* src = c.buckets + (size_t)(b0 + pass) * kBucketCap;
          for (uint32_t i = lane; i < m; i += 32) wkeys[i] = src[i];
        }
        __syncwarp();
        if (m == 0) continue;
        if (m <= 32) {
          const uint64_t key = lane < m ? wkeys[lane] : ~0ULL;
          uint32_t rank = 0;
#pragma unroll
          for (int j = 0; j < 32; j++) rank += (__shfl_sync(0xffffffffu, key, j) < key) ? 1u : 0u;   // keys are distinct
          __syncwarp();
          if (lane < m) wkeys[rank] = key;
        } else {
          uint32_t npow = 64;
          while (npow < m) npow <<= 1;
          for (uint32_t i = m + lane; i < npow; i += 32) wkeys[i] = ~0ULL;
          __syncwarp();
          for (uint32_t kk = 2; kk <= npow; kk <<= 1)
            for (uint32_t j = kk >> 1; j > 0; j >>= 1) {
              for (uint32_t i = lane; i < npow; i += 32) {
                const uint32_t ixj = i ^ j;
                if (ixj > i) {
                  const uint64_t a = wkeys[i], bb = wkeys[ixj];
                  const bool up = (i & kk) == 0;
                  if ((a > bb) == up) { wkeys[i] = bb; wkeys[ixj] = a; }
                }
              }
              __syncwarp();
            }
        }
        __syncwarp();
        if constexpr (FastReplay<KIND>::ok) {
          using FR = FastReplay<KIND>;
          using Wq = Wire<KIND>;
          for (uint32_t p = lane; p < m; p += 32) wops[p] = FR::load_op(c.ord_req + (size_t)(uint32_t)wkeys[p] * Wq::MSG);
          __syncwarp();
          for (uint32_t p = lane; p < m; p += 32)
            if (p == 0 || (uint32_t)(wkeys[p - 1] >> 32) != (uint32_t)(wkeys[p] >> 32)) {
              const uint32_t g = (uint32_t)(wkeys[p] >> 32);
              typename FR::State st = FR::load_state(c, g);
              uint32_t q = p;
              for (; q < m && (uint32_t)(wkeys[q] >> 32) == g; q++) wres[q] = FR::step(st, wops[q]);
              FR::store_state(c, g, st);
              if (q - p > 1) atomicMax(&c.counters[2], (unsigned long long)(q - p));
            }
          __syncwarp();
          for (uint32_t p = lane; p < m; p += 32) FR::write_result(ord_out_ptr<Wq::MSG>(c, (uint32_t)wkeys[p]), wres[p]);
        } else {
          for (uint32_t p = lane; p < m; p += 32)
            if (p == 0 || (uint32_t)(wkeys[p - 1] >> 32) != (uint32_t)(wkeys[p] >> 32)) replay_run<KIND>(c, wkeys, p, m);
        }
        __syncwarp();
      }
      if (lane < gsz && myb < P && cnt) c.bcnt[myb] = 0;
    }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&c.counters[1], (unsigned long long)c.nc_ord[0]);
}

// ---- parallel replay of lock_fasst runs (fallback path) ------------------------------------------------
// A lock_fasst request acts on its slot's (lock, ver) as  lock' in {lock, 0, 1},  ver' = ver + d :
//   kRead (id, +0)   kAcquireLock (set 1, +0)   kAbort (set 0, +0)   kCommit (set 0, +1)
// (lock_fasst/udp/server.cc:86-114).  Such maps compose associatively, so the state every request of a run
// SEES is an exclusive segmented scan over the sorted list -- a run of tens of thousands of requests on one
// hot slot (HOT: 4800 ids, Zipf) is then replayed by the whole grid instead of by one thread.
// Encoding: bits 0-31 d, bits 32-33 lock map (0 id, 1 set 0, 2 set 1), bit 34 segment head, bits 35-63 the number
// of requests composed since the segment head (so the inclusive value at a run's last entry holds the run length;
// exact for runs shorter than 2^29 requests, so for chunks of up to 2^29).
DINT_D uint64_t fx_of(uint32_t type, bool head) {
  const uint64_t lt = (type == 0) ? 0ull : (type == 1) ? 2ull : 1ull;
  return (uint64_t)(type == 3 ? 1u : 0u) | (lt << 32) | ((uint64_t)(head ? 1u : 0u) << 34) | (1ull << 35);
}
DINT_D uint64_t fx_compose(uint64_t a, uint64_t b) {        // a then b, segment-aware
  if ((b >> 34) & 1ull) return b;
  const uint64_t lt = ((b >> 32) & 3ull) ? ((b >> 32) & 3ull) : ((a >> 32) & 3ull);
  return (uint64_t)((uint32_t)a + (uint32_t)b) | (lt << 32) | (a & (1ull << 34)) | (((a >> 35) + (b >> 35)) << 35);
}
constexpr uint64_t kFxId = 0ull;

// inclusive scan of `x` over the CTA in thread order (fx_compose); returns the inclusive value and leaves the
// CTA total in *total.  sh: 8 words of shared memory.
DINT_D uint64_t fx_block_scan(uint64_t x, uint64_t* sh, uint64_t* total) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if ((int)lane_id() >= o) x = fx_compose(y, x);
  }
  if (lane_id() == 31) sh[warp_id()] = x;
  __syncthreads();
  uint64_t pre = kFxId;
  bool have = false;
  uint64_t tot = kFxId;
  for (int w = 0; w < kThreads / 32; w++) {
    const uint64_t v = sh[w];
    if (w < (int)warp_id()) { pre = have ? fx_compose(pre, v) : v; have = true; }
    tot = w ? fx_compose(tot, v) : v;
  }
  __syncthreads();
  *total = tot;
  return have ? fx_compose(pre, x) : x;
}

// Grid-wide barrier of k_ordered.  Stand-alone engines launch it cooperatively (cg grid sync).  Inside the
// multi-GPU step other streams hold flag-polling kernels that wait for PEERS, and a cooperative launch is not
// started while another kernel is resident -- it would wait for a kernel that waits for it.  There the
// launch is a plain one (the grid is sized to be co-resident next to those one-warp kernels) and the barrier is
// a generation counter in global memory.
struct GridBar {
  cg::grid_group g;
  uint32_t* bar;            // [0] arrivals, [1] generation
  bool coop;
  DINT_D void sync() {
    if (coop) { g.sync(); return; }
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t gen;
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(gen) : "l"(bar + 1) : "memory");
      __threadfence();
      if (atomicAdd(bar, 1u) == gridDim.x - 1) {
        bar[0] = 0;
        __threadfence();
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(bar + 1), "r"(gen + 1) : "memory");
      } else {
        uint32_t now;
        do {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(now) : "l"(bar + 1) : "memory");
        } while (now == gen);
      }
      __threadfence();
    }
    __syncthreads();
  }
};

template <int KIND>
__global__ void __launch_bounds__(kThreads) k_ordered(const Ctx c) {
  if (c.skip && __ldcg(c.skip)) return;
  const uint32_t nc = c.nc_ord[0];
  const uint32_t overflow = c.nc_ord[1];
  if (nc == 0 || overflow == 0) return;               // the bucket path (inside the next K1) handles this chunk
  GridBar grid{cg::this_grid(), c.gbar, c.coop_launch != 0};
  __shared__ uint64_t skeys[2048];                    // radix counters
  __shared__ uint32_t wsum[kThreads / 32];
  __shared__ uint32_t s_carry;
  const uint32_t tid = threadIdx.x;
  const uint32_t P = 1u << c.bucket_log2;
  {
    // ---- fallback (skewed chunk): stable LSD radix sort of the whole list by group id --------------
    for (uint32_t b = blockIdx.x * kThreads + tid; b < P; b += gridDim.x * kThreads) c.bcnt[b] = 0;
    // (0) exclusive prefix of the per-tile list lengths (CTA 0)
    if (blockIdx.x == 0) {
      if (tid == 0) s_carry = 0;
      __syncthreads();
      for (uint32_t base = 0; base < c.n_tiles; base += kThreads) {
        uint32_t i = base + tid;
        uint32_t v = i < c.n_tiles ? c.ccnt[i] : 0;
        uint32_t x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
          if ((int)lane_id() >= o) x += y;
        }
        if (lane_id() == 31) wsum[warp_id()] = x;
        __syncthreads();
        uint32_t woff = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < kThreads / 32; w++) {
          if (w < (int)warp_id()) woff += wsum[w];
          tot += wsum[w];
        }
        if (i < c.n_tiles) c.cprefix[i] = s_carry + woff + (x - v);
        __syncthreads();
        if (tid == 0) s_carry += tot;
        __syncthreads();
      }
    }
    grid.sync();
    // (1) densify the tile-segmented list into (group << 32 | index), index-ascending
    for (uint32_t t = blockIdx.x; t < c.n_tiles; t += gridDim.x) {
      uint32_t m = c.ccnt[t];
      if (tid < m) {
        uint32_t idx = c.clist[(size_t)t * kTile + tid];
        c.sortA[c.cprefix[t] + tid] = ((uint64_t)c.grp[idx] << 32) | idx;
      }
    }
    grid.sync();
    uint64_t* src = c.sortA;
    uint64_t* dst = c.sortB;
    const uint32_t n_st = (nc + kSortTile - 1) / kSortTile;
    uint32_t* s_hist = (uint32_t*)skeys;                       // [256]
    uint32_t* s_wcnt = (uint32_t*)skeys + 256;                 // [8 warps][256]
    for (uint32_t pass = 0; pass < c.sort_passes; pass++) {
      const uint32_t shift = 32 + 8 * pass;
      // (a) per-tile digit histograms
      for (uint32_t T = blockIdx.x; T < n_st; T += gridDim.x) {
        s_hist[tid] = 0;
        __syncthreads();
        uint32_t base = T * kSortTile;
#pragma unroll
        for (int k = 0; k < kSortItems; k++) {
          uint32_t i = base + k * kThreads + tid;
          if (i < nc) atomicAdd(&s_hist[(uint32_t)(src[i] >> shift) & 255u], 1u);
        }
        __syncthreads();
        c.ghist[(size_t)tid * n_st + T] = s_hist[tid];
        __syncthreads();
      }
      grid.sync();
      // (b) row totals
      for (uint32_t d = blockIdx.x; d < 256; d += gridDim.x) {
        uint32_t s = 0;
        for (uint32_t T = tid; T < n_st; T += kThreads) s += c.ghist[(size_t)d * n_st + T];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane_id() == 0) wsum[warp_id()] = s;
        __syncthreads();
        if (tid == 0) {
          uint32_t tot = 0;
          for (int w = 0; w < kThreads / 32; w++) tot += wsum[w];
          c.rowtot[d] = tot;
        }
        __syncthreads();
      }
      grid.sync();
      // (c) rows -> global exclusive offsets (digit-major, tile-minor)
      for (uint32_t d = blockIdx.x; d < 256; d += gridDim.x) {
        uint32_t part = (tid < d) ? c.rowtot[tid] : 0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (lane_id() == 0) wsum[warp_id()] = part;
        __syncthreads();
        if (tid == 0) {
          uint32_t b = 0;
          for (int w = 0; w < kThreads / 32; w++) b += wsum[w];
          s_carry = b;
        }
        __syncthreads();
        for (uint32_t base = 0; base < n_st; base += kThreads) {
          uint32_t T = base + tid;
          uint32_t v = T < n_st ? c.ghist[(size_t)d * n_st + T] : 0;
          uint32_t x = v;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if ((int)lane_id() >= o) x += y;
          }
          if (lane_id() == 31) wsum[warp_id()] = x;
          __syncthreads();
          uint32_t woff = 0, tot = 0;
#pragma unroll
          for (int w = 0; w < kThreads / 32; w++) {
            if (w < (int)warp_id()) woff += wsum[w];
            tot += wsum[w];
          }
          if (T < n_st) c.ghist[(size_t)d * n_st + T] = s_carry + woff + (x - v);
          __syncthreads();
          if (tid == 0) s_carry += tot;
          __syncthreads();
        }
      }
      grid.sync();
      // (d) stable scatter: warp w owns items [w*256, w*256+256) of the tile, in 8 rounds of 32
      for (uint32_t T = blockIdx.x; T < n_st; T += gridDim.x) {
        for (uint32_t i = tid; i < 8 * 256; i += kThreads) s_wcnt[i] = 0;
        __syncthreads();
        const uint32_t wbase = T * kSortTile + warp_id() * (kSortItems * 32);
        uint64_t key[kSortItems];
        uint32_t rank[kSortItems];
#pragma unroll
        for (int k = 0; k < kSortItems; k++) {
          uint32_t i = wbase + k * 32 + lane_id();
          bool ok = i < nc;
          key[k] = ok ? src[i] : 0;
          uint32_t dgt = ok ? ((uint32_t)(key[k] >> shift) & 255u) : 256u + lane_id();  // inactive lanes never match
          uint32_t peers = __match_any_sync(0xffffffffu, dgt);
          uint32_t before = __popc(peers & ((1u << lane_id()) - 1u));
          uint32_t basec = 0;
          if (ok) {
            uint32_t* cptr = &s_wcnt[warp_id() * 256 + dgt];
            if (before == 0) { basec = *cptr; *cptr = basec + __popc(peers); }
            basec = __shfl_sync(peers, basec, __ffs(peers) - 1);
          }
          rank[k] = basec + before;
          __syncwarp();
        }
        __syncthreads();
        {                                   // exclusive scan over warps for digit = tid
          uint32_t run = c.ghist[(size_t)tid * n_st + T];
#pragma unroll
          for (int w = 0; w < kThreads / 32; w++) {
            uint32_t v = s_wcnt[w * 256 + tid];
            s_wcnt[w * 256 + tid] = run;
            run += v;
          }
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kSortItems; k++) {
          uint32_t i = wbase + k * 32 + lane_id();
          if (i < nc) {
            uint32_t dgt = (uint32_t)(key[k] >> shift) & 255u;
            dst[s_wcnt[warp_id() * 256 + dgt] + rank[k]] = key[k];
          }
        }
        __syncthreads();
      }
      grid.sync();
      uint64_t* tmp = src; src = dst; dst = tmp;
    }
    if constexpr (KIND == K_FASST) {
      // parallel replay by segmented scan (see fx_of): tile aggregates -> carries -> replies
      using FR = FastReplay<K_FASST>;
      using Wq = Wire<K_FASST>;
      uint64_t* tile_agg = (uint64_t*)c.ghist;                 // [n_st], free after the sort
      uint64_t* sh_scan = skeys;                               // 8 words
      auto load8 = [&](uint32_t T, uint64_t (&f)[kSortItems], uint32_t (&ty)[kSortItems], uint32_t& cnt) {
        const uint32_t base = T * kSortTile + tid * kSortItems;   // blocked: thread t owns 8 consecutive entries
        cnt = base < nc ? min((uint32_t)kSortItems, nc - base) : 0;
#pragma unroll
        for (int k = 0; k < kSortItems; k++) {
          if ((uint32_t)k < cnt) {
            const uint32_t p = base + k;
            const uint64_t e = src[p];
            ty[k] = FR::load_op(c.ord_req + (size_t)(uint32_t)e * Wq::MSG);
            const bool head = p == 0 || (uint32_t)(src[p - 1] >> 32) != (uint32_t)(e >> 32);
            f[k] = fx_of(ty[k], head);
          } else { ty[k] = 0; f[k] = kFxId; }
        }
      };
      // (1) per-tile aggregates
      for (uint32_t T = blockIdx.x; T < n_st; T += gridDim.x) {
        uint64_t f[kSortItems]; uint32_t ty[kSortItems]; uint32_t cnt;
        load8(T, f, ty, cnt);
        uint64_t agg = f[0];
#pragma unroll
        for (int k = 1; k < kSortItems; k++) if ((uint32_t)k < cnt) agg = fx_compose(agg, f[k]);
        uint64_t total;
        (void)fx_block_scan(agg, sh_scan, &total);
        if (tid == 0) tile_agg[T] = total;
      }
      grid.sync();
      // (2) exclusive scan of the tile aggregates (CTA 0, sequential over <= a few hundred tiles per thread-chunk)
      if (blockIdx.x == 0 && tid == 0) {
        uint64_t run = kFxId;
        bool have = false;
        for (uint32_t T = 0; T < n_st; T++) {
          const uint64_t a = tile_agg[T];
          tile_agg[T] = have ? run : (1ull << 34);           // "nothing before": behaves as a segment head
          run = have ? fx_compose(run, a) : a;
          have = true;
        }
      }
      grid.sync();
      // (3) replies: every entry derives the state it sees from its exclusive prefix
      uint32_t run_max = 0;                                    // longest run ending in this thread's entries
      for (uint32_t T = blockIdx.x; T < n_st; T += gridDim.x) {
        uint64_t f[kSortItems]; uint32_t ty[kSortItems]; uint32_t cnt;
        load8(T, f, ty, cnt);
        uint64_t agg = f[0];
#pragma unroll
        for (int k = 1; k < kSortItems; k++) if ((uint32_t)k < cnt) agg = fx_compose(agg, f[k]);
        uint64_t total;
        const uint64_t incl = fx_block_scan(agg, sh_scan, &total);
        // exclusive prefix of this thread's first entry = carry(tile) o (inclusive of the previous thread)
        uint64_t prev_thread = __shfl_up_sync(0xffffffffu, incl, 1);
        if (lane_id() == 0) prev_thread = kFxId;               // patched below from shared memory
        __shared__ uint64_t s_warp_last[kThreads / 32];
        if (lane_id() == 31) s_warp_last[warp_id()] = incl;
        __syncthreads();
        const uint64_t carry = tile_agg[T];
        uint64_t pre;
        if (tid == 0) pre = carry;
        else {
          const uint64_t before = lane_id() == 0 ? s_warp_last[warp_id() - 1] : prev_thread;
          pre = ((carry >> 34) & 1ull) && carry == (1ull << 34) ? before : fx_compose(carry, before);
        }
        __syncthreads();
        const uint32_t base = T * kSortTile + tid * kSortItems;
#pragma unroll
        for (int k = 0; k < kSortItems; k++) {
          if ((uint32_t)k < cnt) {
            const uint32_t p = base + k;
            const uint64_t e = src[p];
            const uint32_t g = (uint32_t)(e >> 32);
            const bool head = (f[k] >> 34) & 1ull;
            const uint64_t ex = head ? kFxId : pre;            // exclusive prefix inside the run
            typename FR::State st = FR::load_state(c, g);
            const uint32_t lt = (uint32_t)(ex >> 32) & 3u;
            if (!head) {
              if (lt) st.lock = (lt == 2u);
              st.ver += (uint32_t)ex;
              st.dirty_ver = (uint32_t)ex != 0;
            }
            const uint64_t r = FR::step(st, ty[k]);
            FR::write_result(ord_out_ptr<Wq::MSG>(c, (uint32_t)e), r);
            // the run's final state is written only after EVERY entry has read the initial one (next pass)
            const bool last = p + 1 == nc || (uint32_t)(src[p + 1] >> 32) != g;
            if (last) dst[p] = (uint64_t)st.ver | ((uint64_t)st.lock << 32) | ((uint64_t)(st.dirty_ver ? 1u : 0u) << 33);
            pre = head ? f[k] : fx_compose(pre, f[k]);
            if (last) run_max = max(run_max, (uint32_t)(pre >> 35));   // inclusive prefix of a run's last entry: its length
          }
        }
      }
      run_max = __reduce_max_sync(0xffffffffu, run_max);        // the loop above is uniform per CTA: every lane is here
      if (lane_id() == 0 && run_max > 1) atomicMax(&c.counters[2], (unsigned long long)run_max);
      grid.sync();
      // (4) final state of every run
      for (uint32_t p = blockIdx.x * kThreads + tid; p < nc; p += gridDim.x * kThreads) {
        const uint32_t g = (uint32_t)(src[p] >> 32);
        if (p + 1 == nc || (uint32_t)(src[p + 1] >> 32) != g) {
          const uint64_t v = dst[p];
          typename FR::State st{(uint32_t)v, (uint32_t)(v >> 32) & 1u, g, ((v >> 33) & 1ull) != 0};
          FR::store_state(c, g, st);
        }
      }
    } else if constexpr (FastReplay<KIND>::ok) {
      // replay in three passes: request fields of ALL listed requests (parallel) -> per-run walk with the
      // group state in registers -> replies (parallel).  ops live in the (now free) clist, replies in `dst`.
      using FR = FastReplay<KIND>;
      using Wq = Wire<KIND>;
      uint32_t* ops_g = c.clist;
      uint64_t* res_g = dst;
      for (uint32_t p = blockIdx.x * kThreads + tid; p < nc; p += gridDim.x * kThreads)
        ops_g[p] = FR::load_op(c.ord_req + (size_t)(uint32_t)src[p] * Wq::MSG);
      grid.sync();
      for (uint32_t p = blockIdx.x * kThreads + tid; p < nc; p += gridDim.x * kThreads)
        if (p == 0 || (uint32_t)(src[p - 1] >> 32) != (uint32_t)(src[p] >> 32)) {
          const uint32_t g = (uint32_t)(src[p] >> 32);
          typename FR::State st = FR::load_state(c, g);
          uint32_t q = p;
          for (; q < nc && (uint32_t)(src[q] >> 32) == g; q++) res_g[q] = FR::step(st, ops_g[q]);
          FR::store_state(c, g, st);
          if (q - p > 1) atomicMax(&c.counters[2], (unsigned long long)(q - p));
        }
      grid.sync();
      for (uint32_t p = blockIdx.x * kThreads + tid; p < nc; p += gridDim.x * kThreads)
        FR::write_result(ord_out_ptr<Wq::MSG>(c, (uint32_t)src[p]), res_g[p]);
    } else {
      // replay: one thread per same-group run
      for (uint32_t p = blockIdx.x * kThreads + tid; p < nc; p += gridDim.x * kThreads)
        if (p == 0 || (uint32_t)(src[p - 1] >> 32) != (uint32_t)(src[p] >> 32)) replay_run<KIND>(c, src, p, nc);
    }
  }
  if (blockIdx.x == 0 && tid == 0) {
    atomicAdd(&c.counters[1], (unsigned long long)nc);
    atomicAdd(&c.counters[3], 1ull);                   // chunks that took this fallback
  }
}

}  // namespace dint
