// engine.cu -- host side of libdint_b200.so: state allocation in HBM, the per-chunk launch sequence,
// host<->device pipelining for dint_submit(), state inspection, and the extern "C" ABI of
// include/dint_b200.h.  No CPU implementation of the request path exists here: without a CUDA
// device every compute entry point returns DINT_ENODEV.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <chrono>
#include <vector>

#include "../../include/dint_b200.h"
#include "kernels.cuh"
#include "route.cuh"
#include "kv.cuh"
#include "clients.cuh"
#include "txn_clients.cuh"

using namespace dint;

static thread_local std::string g_last_error;
static int set_err(int code, const char* what, cudaError_t ce = cudaSuccess) {
  char buf[512];
  if (ce != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(ce));
  else snprintf(buf, sizeof buf, "%s", what);
  g_last_error = buf;
  return code;
}
#define CU(call)                                                              \
  do {                                                                        \
    cudaError_t _e = (call);                                                  \
    if (_e != cudaSuccess) return set_err(_e == cudaErrorMemoryAllocation ? DINT_ENOMEM : DINT_EIO, #call, _e); \
  } while (0)

static const uint32_t kMsgSize[DINT_NUM_KINDS] = {6, 9, 53, 53, 55, 23};
static const uint32_t kLogEntry[DINT_NUM_KINDS] = {0, 0, 56, 0, 64, 32};
static const uint32_t kValSize[DINT_NUM_KINDS] = {0, 0, 0, 40, 40, 8};

enum { KT_CLASSIFY = 0, KT_LOGSCAN, KT_APPLY, KT_ORDERED, KT_LOAD, KT_NUM };
static const char* kKernelNames[KT_NUM] = {"k_classify", "k_log_scan", "k_apply", "k_ordered", "k_kv_load"};

struct EvPair { cudaEvent_t a, b; int which; };
constexpr int kHostBufs = 4;      // device staging buffers of the host path (dint_submit)

struct dint_engine {
  int kind = 0;
  int device = 0;
  dint_cfg cfg{};
  uint32_t msg = 0;
  uint32_t chunk = 0;
  uint32_t max_tiles = 0;
  bool has_log = false;
  Ctx ctx{};                       // device pointers + constants; per-launch fields filled per chunk
  std::vector<void*> allocs;       // everything to cudaFree
  cudaStream_t stream = nullptr, s_in = nullptr, s_out = nullptr;
  uint8_t* d_req[kHostBufs] = {nullptr};
  uint8_t* d_resp[kHostBufs] = {nullptr};
  cudaEvent_t ev_in[kHostBufs]{}, ev_comp[kHostBufs]{}, ev_out[kHostBufs]{};
  uint32_t host_chunk = 0;                   // requests per host-path slice
  bool plain_launches = false;               // inside the multi-GPU step: no cooperative launches (see GridBar)
  uint32_t host_min_slice = 0;               // smallest slice of the pyramid a host-path call is cut into
  bool host_ramp_up = true;
  unsigned long long* h_counters = nullptr;  // pinned mirror of ctx.counters (host path reads it without a blocking copy)
  unsigned long long* h_kvcnt = nullptr;     // pinned mirror of every table's {live, used} (kv_maintain)
  cudaEvent_t ev_kvcnt = nullptr;
  int coop_grid = 0;
  int sms = 0;
  int grid_classify = 0, grid_apply = 0;     // persistent CTAs (SMs x resident CTAs per SM)
  uint32_t smem_stage = 0;                   // dynamic shared memory of K1/K2: kStages staged tiles
  uint64_t total_groups = 0;
  uint32_t* d_flags[2] = {nullptr, nullptr}; // flag-nibble sets, alternating per chunk
  uint32_t* d_grp[2] = {nullptr, nullptr};   // group ids of the current / previous chunk
  uint64_t chunk_seq = 0;
  uint32_t prev_n = 0;                       // requests of the previous chunk whose flags are still set
  bool ord_pending = false;                  // the previous chunk's listed requests await their replay
  uint8_t* ord_resp = nullptr;               //   ... and live in this reply array
  const uint8_t* ord_req = nullptr;          //   ... their request bytes in this one
  uint32_t ord_tile0 = 0;                    //   ... which starts at this tile of its batch
  // segmented replies (multi-GPU step): set around run_device by the sharded step, zero otherwise
  uint32_t seg_tiles = 0;
  uint64_t seg_resp[kMaxShards]{};
  bool pad_ok = false;
  const uint32_t* skip = nullptr;
  uint32_t smem_classify = 0;                // K1: max(stages, ordered-replay slices)
  uint32_t* d_nc = nullptr;                  // [2 chunks][2]: listed / overflow counters
  uint32_t* d_route = nullptr;               // multi-GPU dispatch scratch (per-tile per-shard counts)
  uint32_t route_tiles = 0;
  uint32_t* d_route2 = nullptr;              // dispatch scratch: counters, totals, look-back descriptors
  uint32_t route_desc_tiles = 0, route_seq = 0;
  int grid_route = 148 * 4;                  // CTAs of k_route_dispatch: 4 per SM are resident (64 registers x 256 threads); 2^20 small
                                             // records = 512 tiles = ONE wave (tiles are drawn by ticket, so any grid is correct)
  // L2 persistence: the flag sets (+ lock_fasst lock bits) live in one arena that every launch maps
  // with a persisting access-policy window, so the streaming request/reply traffic cannot evict it
  uint8_t* hot_arena = nullptr;
  size_t hot_bytes = 0;
  bool use_window = false;
  cudaAccessPolicyWindow window{};
  // stats
  dint_stats stats{};
  // profiling
  uint32_t profiling = 0;          // bit k set: bracket launches of kernel k (KT_*) with CUDA events
  std::vector<EvPair> ev_pool;
  size_t ev_used = 0;
  double kt_ms[KT_NUM] = {0};
  uint64_t kt_n[KT_NUM] = {0};
  // KV host mirrors
  KvHost kv[kMaxTables];
};

template <typename T>
static int dalloc(dint_engine* e, T** p, size_t count, bool zero = true) {
  size_t bytes = count * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  void* q = nullptr;
  CU(cudaMalloc(&q, bytes));
  e->allocs.push_back(q);
  if (zero) CU(cudaMemsetAsync(q, 0, bytes, e->stream));
  *p = (T*)q;
  return DINT_OK;
}

// ---- profiling helpers ------------------------------------------------------------------------------
static int prof_flush(dint_engine* e) {
  for (size_t i = 0; i < e->ev_used; i++) {
    float ms = 0;
    CU(cudaEventSynchronize(e->ev_pool[i].b));
    CU(cudaEventElapsedTime(&ms, e->ev_pool[i].a, e->ev_pool[i].b));
    e->kt_ms[e->ev_pool[i].which] += ms;
    e->kt_n[e->ev_pool[i].which]++;
  }
  e->ev_used = 0;
  return DINT_OK;
}
struct ProfScope {
  dint_engine* e; cudaStream_t s; EvPair* p = nullptr;
  ProfScope(dint_engine* e_, cudaStream_t s_, int which) : e(e_), s(s_) {
    e->stats.kernel_launches++;
    if (!((e->profiling >> which) & 1u)) return;
    if (e->ev_used == e->ev_pool.size()) {
      if (e->ev_pool.size() >= 8192) { prof_flush(e); }
      else {
        EvPair np{}; cudaEventCreate(&np.a); cudaEventCreate(&np.b);
        e->ev_pool.push_back(np);
      }
    }
    p = &e->ev_pool[e->ev_used++];
    p->which = which;
    cudaEventRecord(p->a, s);
  }
  ~ProfScope() { if (p) cudaEventRecord(p->b, s); }
};

// ---- per-chunk launch sequence ------------------------------------------------------------------------
template <typename... Args>
static cudaError_t launch_ex(dint_engine* e, void (*kern)(Args...), int grid, int block, size_t smem, cudaStream_t s,
                             bool coop, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid < 1 ? 1 : grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute at[3];
  int na = 0;
  if (coop) { at[na].id = cudaLaunchAttributeCooperative; at[na].val.cooperative = 1; na++; }
  if (e->use_window) { at[na].id = cudaLaunchAttributeAccessPolicyWindow; at[na].val.accessPolicyWindow = e->window; na++; }
  cfg.attrs = at;
  cfg.numAttrs = na;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

// One chunk: K1 (classify this chunk + replay the previous chunk's listed requests), K2 (apply), and the
// fallback launch that only does work when one of THIS chunk's buckets overflowed.  c.n == 0 = flush: K1
// alone, replaying the last chunk's listed requests.
template <int KIND, bool HAS_LOG>
static int launch_chunk_t(dint_engine* e, const Ctx& c, cudaStream_t s) {
  {
    ProfScope ps(e, s, KT_CLASSIFY);
    int want = (int)c.n_tiles, clr = (int)((c.prev_n + 4 * kTile - 1) / (4 * kTile));
    if (clr > want) want = clr;
    int grid = (want < e->grid_classify && !c.ord_pending) ? want : e->grid_classify;
    if (c.n == 0 && e->sms > 0 && grid > 8 * e->sms) grid = 8 * e->sms;     // a flush launch only replays: 32 warps per SM are plenty
    CU(launch_ex(e, k_classify<KIND, HAS_LOG>, grid, kTile, e->smem_classify, s, false, c));
  }
  if (c.n == 0) { CU(cudaGetLastError()); return DINT_OK; }
  if (HAS_LOG) {
    ProfScope ps(e, s, KT_LOGSCAN);
    k_log_scan<<<1, kThreads, 0, s>>>(c);
  }
  {
    ProfScope ps(e, s, KT_APPLY);
    int grid = (int)c.n_tiles < e->grid_apply ? (int)c.n_tiles : e->grid_apply;
    CU(launch_ex(e, k_apply<KIND, HAS_LOG>, grid, kTile, e->smem_stage, s, false, c));
  }
  if (KIND != K_LOG) {   // the log server has no per-key state: nothing to order
    ProfScope ps(e, s, KT_ORDERED);
    Ctx f = c;           // this chunk's own counters / replies
    f.nc_ord = c.nc_cur;
    f.ord_resp = c.resp;
    f.ord_req = c.req;
    f.ord_tile0 = c.tile0;
    f.coop_launch = e->plain_launches ? 0u : 1u;
    int g3 = e->coop_grid;
    if (e->plain_launches && e->sms > 0) {             // leave room for the one-warp flag-polling kernels of the other streams
      const int per = g3 / e->sms;
      g3 = (per > 1 ? per - 1 : 1) * e->sms;
    }
    CU(launch_ex(e, k_ordered<KIND>, g3, kThreads, 0, s, !e->plain_launches, f));
  }
  CU(cudaGetLastError());
  return DINT_OK;
}

static int launch_chunk(dint_engine* e, const Ctx& c, cudaStream_t s) {
  switch (e->kind) {
    case DINT_LOCK2PL: return launch_chunk_t<K_LOCK2PL, false>(e, c, s);
    case DINT_FASST: return launch_chunk_t<K_FASST, false>(e, c, s);
    case DINT_LOG: return launch_chunk_t<K_LOG, true>(e, c, s);
    case DINT_STORE: return launch_chunk_t<K_STORE, false>(e, c, s);
    case DINT_TATP: return launch_chunk_t<K_TATP, true>(e, c, s);
    case DINT_SMALLBANK: return launch_chunk_t<K_SMALLBANK, true>(e, c, s);
  }
  return DINT_EINVAL;
}

template <int KIND, bool HAS_LOG>
static int grids_for(dint_engine* e) {
  int per_sm = 0, sms = 0;
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->device));
  e->smem_stage = Stage<Wire<KIND>::MSG>::N * Stage<Wire<KIND>::MSG>::BYTES;
  if (e->smem_stage > 48 * 1024) {
    CU(cudaFuncSetAttribute(k_classify<KIND, HAS_LOG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->smem_stage));
    CU(cudaFuncSetAttribute(k_apply<KIND, HAS_LOG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->smem_stage));
  }
  e->smem_classify = e->smem_stage;
  if (KIND != K_LOG && (kTile / 32) * OrdSlice<KIND>::BYTES > e->smem_classify) e->smem_classify = (kTile / 32) * OrdSlice<KIND>::BYTES;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_classify<KIND, HAS_LOG>, kTile, e->smem_classify));
  if (per_sm < 1) return set_err(DINT_EIO, "k_classify cannot be resident");
  e->grid_classify = per_sm * sms;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_apply<KIND, HAS_LOG>, kTile, e->smem_stage));
  if (per_sm < 1) return set_err(DINT_EIO, "k_apply cannot be resident");
  e->grid_apply = per_sm * sms;
  if (KIND == K_LOG) { e->coop_grid = 1; return DINT_OK; }
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_ordered<KIND>, kThreads, 0));
  if (per_sm < 1) return set_err(DINT_EIO, "k_ordered cannot be resident");
  if (per_sm > 4) per_sm = 4;
  e->coop_grid = per_sm * sms;
  e->sms = sms;
  return DINT_OK;
}

static void fill_chunk_ctx(dint_engine* e, Ctx& c) {
  const int cur = (int)(e->chunk_seq & 1);
  c.grp = e->d_grp[cur];
  c.grp_prev = e->d_grp[cur ^ 1];
  c.flags = e->d_flags[cur];
  c.flags_prev = e->d_flags[cur ^ 1];
  c.prev_n = e->prev_n;
  c.nc_cur = e->d_nc + 4 * cur;          // {listed, overflow, a writer exists, -}
  c.nc_ord = e->d_nc + 4 * (cur ^ 1);
  c.ord_pending = e->ord_pending ? 1u : 0u;
  c.ord_resp = e->ord_resp;
  c.ord_req = e->ord_req;
  c.ord_tile0 = e->ord_tile0;
  c.seg_tiles = e->seg_tiles;
  c.pad_ok = e->pad_ok ? 1u : 0u;
  c.skip = e->skip;
  for (int i = 0; i < kMaxShards; i++) c.seg_resp[i] = e->seg_resp[i];
}

// one chunk (n <= e->chunk); leaves its listed requests pending until the next chunk or flush_ordered()
static int submit_chunk(dint_engine* e, const uint8_t* req, uint32_t n, uint8_t* resp, cudaStream_t s, uint32_t tile0 = 0) {
  Ctx c = e->ctx;
  c.n = n;
  c.n_tiles = (n + kTile - 1) / kTile;
  c.req = req;
  c.resp = resp;
  c.tile0 = tile0;
  fill_chunk_ctx(e, c);
  int rc = launch_chunk(e, c, s);
  if (rc) return rc;
  e->chunk_seq++;
  e->prev_n = n;
  e->ord_pending = e->kind != DINT_LOG;
  e->ord_resp = resp;
  e->ord_req = req;
  e->ord_tile0 = tile0;
  e->stats.chunks++;
  e->stats.requests += n;
  return DINT_OK;
}

// replays the last chunk's listed requests (and retires its flags); after this every reply is final
static int flush_ordered(dint_engine* e, cudaStream_t s) {
  if (!e->ord_pending) return DINT_OK;
  Ctx c = e->ctx;
  c.n = 0;
  c.n_tiles = 0;
  c.req = nullptr;
  c.resp = nullptr;
  fill_chunk_ctx(e, c);
  c.prev_n = 0;                  // replay only: that chunk's flags are retired by the NEXT chunk's K1 as usual (next to its tile
                                 // loads), not by this launch, which a caller is waiting for
  int rc = launch_chunk(e, c, s);
  if (rc) return rc;
  e->ord_pending = false;
  return DINT_OK;
}

// Tombstone reclamation (kv.cuh): after every call the per-table {live, used} counters travel to a pinned mirror;
// before the next call a table whose FULL + TOMB entries exceed 70 % of its capacity is rehashed into a fresh
// array (doubled when the live keys alone exceed 35 %).  Synchronous and rare: at load <= 0.5 it takes an
// insert / delete churn of 20 % of the capacity to get there.
static int kv_maintain(dint_engine* e, cudaStream_t s) {
  if (e->ctx.n_tables == 0) return DINT_OK;
  if (!e->h_kvcnt) {
    CU(cudaHostAlloc((void**)&e->h_kvcnt, 2 * kMaxTables * sizeof(unsigned long long), cudaHostAllocDefault));
    memset(e->h_kvcnt, 0, 2 * kMaxTables * sizeof(unsigned long long));
    CU(cudaEventCreateWithFlags(&e->ev_kvcnt, cudaEventDisableTiming));
    return DINT_OK;
  }
  if (cudaEventQuery(e->ev_kvcnt) != cudaSuccess) { cudaGetLastError(); return DINT_OK; }   // mirror not refreshed yet
  for (uint32_t t = 0; t < e->ctx.n_tables; t++) {
    KvTable& T = e->ctx.tbl[t];
    const unsigned long long live = e->h_kvcnt[2 * t], used = e->h_kvcnt[2 * t + 1];
    const unsigned long long cap = T.cap_mask + 1;
    if (used * 10 < cap * 7) continue;
    KvTable N = T;
    if (live * 20 > cap * 7) { N.cap_log2++; N.cap_mask = (1ULL << N.cap_log2) - 1; }
    void* fresh = nullptr;
    const size_t bytes = (size_t)(N.cap_mask + 1) << N.ent_shift;
    CU(cudaMalloc(&fresh, bytes));
    CU(cudaMemsetAsync(fresh, 0, bytes, s));
    CU(cudaMemsetAsync(T.live, 0, 16, s));                   // the rehash re-counts both
    N.entries = (uint8_t*)fresh;
    {
      ProfScope ps(e, s, KT_LOAD);
      if (e->kind == DINT_SMALLBANK) k_kv_rehash<8><<<148 * 8, 256, 0, s>>>(T, N);
      else k_kv_rehash<40><<<148 * 8, 256, 0, s>>>(T, N);
    }
    CU(cudaStreamSynchronize(s));
    for (auto& p : e->allocs) if (p == (void*)T.entries) p = fresh;
    CU(cudaFree(T.entries));
    T = N;
    e->kv[t].capacity = N.cap_mask + 1;
    e->h_kvcnt[2 * t + 1] = live;
    e->stats.kv_rebuilds++;
  }
  return DINT_OK;
}
static int kv_publish_counts(dint_engine* e, cudaStream_t s) {
  if (e->ctx.n_tables == 0 || !e->h_kvcnt) return DINT_OK;
  CU(cudaMemcpyAsync(e->h_kvcnt, e->ctx.tbl[0].live, 16 * e->ctx.n_tables, cudaMemcpyDeviceToHost, s));   // (the tables' counters are contiguous)
  CU(cudaEventRecord(e->ev_kvcnt, s));
  return DINT_OK;
}

static int run_device(dint_engine* e, const uint8_t* req, uint64_t n, uint8_t* resp, cudaStream_t s) {
  { int rc = kv_maintain(e, s); if (rc) return rc; }
  for (uint64_t off = 0; off < n; off += e->chunk) {
    uint32_t cn = (uint32_t)((n - off < e->chunk) ? (n - off) : e->chunk);
    int rc = submit_chunk(e, req + off * e->msg, cn, resp ? resp + off * e->msg : nullptr, s, (uint32_t)(off / kTile));
    if (rc) return rc;
  }
  int rc = flush_ordered(e, s);
  return rc ? rc : kv_publish_counts(e, s);
}

static int pull_counters(dint_engine* e) {
  unsigned long long h[4];
  CU(cudaMemcpy(h, e->ctx.counters, sizeof h, cudaMemcpyDeviceToHost));
  e->stats.errors = h[0];
  e->stats.conflicted = h[1];
  e->stats.max_run = h[2];
  e->stats.fallback_chunks = h[3];
  return DINT_OK;
}

template <int MSG>
static void route_scatter_t(const uint8_t* rq, const uint8_t* ow, uint32_t n, uint32_t world, const uint32_t* tb,
                            const uint32_t* totals, uint8_t* out, uint32_t* perm, uint32_t tiles, cudaStream_t s) {
  k_exact_scatter<MSG><<<tiles, kThreads, 0, s>>>(rq, ow, n, world, tb, totals, out, perm);
}
template <int MSG>
static void route_unpermute_t(const uint8_t* sorted, const uint32_t* perm, uint32_t n, uint8_t* out, cudaStream_t s) {
  k_exact_unpermute<MSG><<<(n + kThreads - 1) / kThreads, kThreads, 0, s>>>(sorted, perm, n, out);
}

// Host-path slice sizes for a call of n requests (see dint_submit): slices double from `mn` up to the plateau
// `mx`, the body moves in plateau slices (a remainder first), and the end halves back down to `mn`.
struct HostSlices {
  uint32_t lvl[32];          // pyramid levels below the plateau, smallest first
  uint32_t n_lvl = 0, i_up = 0, i_down = 0;
  uint64_t body = 0, plateau = 0, pending = 0;
  bool ramp_up;
  HostSlices(uint64_t n, uint32_t mn, uint32_t mx, bool ramp_up_) : ramp_up(ramp_up_) {
    if (mn > mx) mn = mx;
    uint64_t used = 0;
    for (uint64_t s = mn; s < mx && n_lvl < 32; s <<= 1) {
      const uint64_t cost = ramp_up ? 2 * s : s;
      if (used + cost > n) break;
      lvl[n_lvl++] = (uint32_t)s;
      used += cost;
    }
    body = n - used;
    plateau = n_lvl ? (uint64_t)lvl[n_lvl - 1] * 2 : mx;
    if (plateau > mx) plateau = mx;
    i_down = n_lvl;
    if (!ramp_up) i_up = n_lvl;
  }
  uint32_t next() {          // 0 = done
    if (i_up < n_lvl) return lvl[i_up++];
    if (body) {
      const uint64_t rem = body % plateau;
      uint64_t c = rem ? rem : plateau;
      if (pending) { c = pending; pending = 0; }
      else if (rem && body > rem) {                        // a remainder is shared with one plateau slice: two
        c = (plateau + rem + 1) / 2;                       // mid-size slices instead of a tiny one and a full one
        pending = plateau + rem - c;
      }
      body -= c;
      return (uint32_t)c;
    }
    if (i_down) return lvl[--i_down];
    return 0;
  }
};

// ---- fused dispatch / combine (route.cuh) ---------------------------------------------------------------
template <int KIND>
static int route_dispatch_t(dint_engine* e, const RouteArgs& a, cudaStream_t s) {
  using RT = RTile<Wire<KIND>::MSG>;
  // scratch: [0] finished-CTA counter, [1] the dispatch tile ticket, [4..12] totals + valid word, then the look-back descriptors
  if (!e->d_route2 || a.n_tiles > e->route_desc_tiles) {
    if (e->d_route2) { CU(cudaStreamSynchronize(s)); CU(cudaFree(e->d_route2)); e->d_route2 = nullptr; }
    e->route_desc_tiles = a.n_tiles + a.n_tiles / 2 + 64;
    const size_t bytes = 64 + (size_t)(e->route_desc_tiles + e->route_desc_tiles / 32 + 1) * 4 * sizeof(unsigned long long);
    CU(cudaMalloc(&e->d_route2, bytes));
    CU(cudaMemsetAsync(e->d_route2, 0, bytes, s));
    e->route_seq = 0;
  }
  e->route_seq = e->route_seq % 255u + 1u;              // 1..255; when the number wraps every descriptor is cleared, so a word
  if (e->route_seq == 1)                                 // left by an earlier launch can never carry the current number
    CU(cudaMemsetAsync(e->d_route2, 0, 64 + (size_t)(e->route_desc_tiles + e->route_desc_tiles / 32 + 1) * 4 * sizeof(unsigned long long), s));
  RouteArgs b = a;
  b.done = e->d_route2;
  b.ticket = e->d_route2 + 1;
  b.totals = e->d_route2 + 4;
  b.desc = (unsigned long long*)(e->d_route2 + 16);
  b.gdesc = b.desc + (size_t)e->route_desc_tiles * 4;
  b.seq = e->route_seq;
  if (CUDART_VERSION >= 11000 && RT::SMEM > 48 * 1024) CU(cudaFuncSetAttribute(k_route_dispatch<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RT::SMEM));
  int grid = (int)b.n_tiles < e->grid_route ? (int)b.n_tiles : e->grid_route;
  if (grid < 1) grid = 1;
  k_route_dispatch<KIND><<<grid, kThreads, RT::SMEM, s>>>(e->ctx, b);
  CU(cudaGetLastError());
  return DINT_OK;
}
template <int MSG>
static int route_combine_t(dint_engine* e, const RouteArgs& a, cudaStream_t s) {
  using RT = RTile<MSG>;
  int grid = (int)a.n_tiles;
  if (grid > 148 * 4) grid = 148 * 4;
  k_route_combine<MSG><<<grid, kThreads, RT::SMEM, s>>>(a);
  CU(cudaGetLastError());
  return DINT_OK;
}
static uint32_t route_tile_records(const dint_engine* e) { return e->msg <= 12 ? kThreads * 8u : (uint32_t)kThreads; }

// ======================================================================================================
extern "C" {

uint32_t dint_msg_size(int kind) { return (kind >= 0 && kind < DINT_NUM_KINDS) ? kMsgSize[kind] : 0; }
uint32_t dint_log_entry_size(int kind) { return (kind >= 0 && kind < DINT_NUM_KINDS) ? kLogEntry[kind] : 0; }
const char* dint_last_error(void) { return g_last_error.c_str(); }
uint64_t dint_test_fasthash64(uint64_t x, int len) { return len == 4 ? fasthash64_u32((uint32_t)x) : fasthash64_u64(x); }
uint32_t dint_test_fastmod(uint64_t n, uint32_t d) { FastMod f = make_fastmod(d); return fast_mod(n, f); }
uint32_t dint_test_host_slices(uint64_t n, uint32_t min_slice, uint32_t max_slice, int ramp_up, uint32_t* out, uint32_t cap) {
  HostSlices sched(n, min_slice, max_slice, ramp_up != 0);
  uint32_t k = 0;
  for (uint32_t cn; (cn = sched.next()) != 0; k++)
    if (k < cap) out[k] = cn;
  return k;
}

void dint_default_cfg(int kind, dint_cfg* cfg) {
  memset(cfg, 0, sizeof *cfg);
  cfg->lock_slots = 36000000u;
  cfg->log_ring = 1000000u;
  cfg->subs_sizing = (kind == DINT_TATP) ? 7000000u : 2000000u;
  cfg->subs_populate = cfg->subs_sizing;
  cfg->accts_sizing = 24000000u;
  cfg->accts_populate = cfg->accts_sizing;
  cfg->n_shards = 1;
  cfg->shard_id = 0;
  cfg->chunk = 1u << 20;
}

void* dint_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void dint_host_free(void* p) { if (p) cudaFreeHost(p); }

void dint_destroy(dint_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  for (void* p : e->allocs) cudaFree(p);
  if (e->d_route) cudaFree(e->d_route);
  if (e->d_route2) cudaFree(e->d_route2);
  if (e->h_counters) cudaFreeHost(e->h_counters);
  if (e->h_kvcnt) cudaFreeHost(e->h_kvcnt);
  if (e->ev_kvcnt) cudaEventDestroy(e->ev_kvcnt);
  for (auto& ep : e->ev_pool) { cudaEventDestroy(ep.a); cudaEventDestroy(ep.b); }
  for (int i = 0; i < kHostBufs; i++) {
    if (e->ev_in[i]) cudaEventDestroy(e->ev_in[i]);
    if (e->ev_comp[i]) cudaEventDestroy(e->ev_comp[i]);
    if (e->ev_out[i]) cudaEventDestroy(e->ev_out[i]);
  }
  if (e->stream) cudaStreamDestroy(e->stream);
  if (e->s_in) cudaStreamDestroy(e->s_in);
  if (e->s_out) cudaStreamDestroy(e->s_out);
  delete e;
}

static int create_impl(dint_engine* e) {
  const dint_cfg& cf = e->cfg;
  Ctx& c = e->ctx;
  CU(cudaSetDevice(e->device));
  CU(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&e->s_in, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&e->s_out, cudaStreamNonBlocking));
  for (int i = 0; i < kHostBufs; i++) {
    CU(cudaEventCreateWithFlags(&e->ev_in[i], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_comp[i], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&e->ev_out[i], cudaEventDisableTiming));
  }
  c.n_shards = cf.n_shards;
  c.shard_id = cf.shard_id;
  c.shard_div = make_fastmod(cf.n_shards);
  c.slot_mod = make_fastmod(cf.lock_slots);
  c.ring_n = cf.log_ring ? cf.log_ring : 1;

  // ---- per-kind state in HBM ----
  uint64_t groups = 0;
  auto local_groups = [&](uint64_t global) { return (global + cf.n_shards - 1) / cf.n_shards; };
  int rc;
  switch (e->kind) {
    case DINT_LOCK2PL:
      groups = local_groups(cf.lock_slots);
      if ((rc = dalloc(e, &c.cnt2, groups))) return rc;
      break;
    case DINT_FASST:
      groups = local_groups(cf.lock_slots);
      if ((rc = dalloc(e, &c.ver, groups))) return rc;     // lock bits: in the hot arena, below
      break;
    case DINT_LOG:
      groups = 0;
      break;
    default:
      if ((rc = kv_create_tables(e->kind, cf, c, e->kv, &groups,
                                 [&](void** p, size_t bytes) -> int {
                                   uint8_t* q = nullptr;
                                   int r = dalloc(e, &q, bytes);
                                   *p = q;
                                   return r;
                                 })))
        return rc == DINT_EINVAL ? set_err(rc, "bad KV configuration") : rc;
      break;
  }
  e->total_groups = groups;
  if (groups >= 0xffffffffULL) return set_err(DINT_EINVAL, "too many groups");
  {
    uint32_t fl = 25;                                  // 2^25 nibbles = 16 MB per set: L2-resident
    while (fl > 10 && (1ULL << (fl - 1)) >= groups * 2 + 2048) fl--;   // tiny group spaces need less
    c.flags_mask = (1u << fl) - 1;
    const size_t set_bytes = (size_t)4 << (fl - 3);
    const size_t lock_bytes = (e->kind == DINT_FASST) ? (((groups + 31) / 32) * 4 + 255) / 256 * 256 : 0;
    e->hot_bytes = 2 * set_bytes + lock_bytes;
    if ((rc = dalloc(e, &e->hot_arena, e->hot_bytes))) return rc;
    e->d_flags[0] = (uint32_t*)e->hot_arena;
    e->d_flags[1] = (uint32_t*)(e->hot_arena + set_bytes);
    if (lock_bytes) c.lockbits = (uint32_t*)(e->hot_arena + 2 * set_bytes);
    // reserve L2 for it
    int max_persist = 0, max_win = 0;
    cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, e->device);
    cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, e->device);
    if (max_persist > 0 && max_win > 0) {
      size_t want = e->hot_bytes < (size_t)max_persist ? e->hot_bytes : (size_t)max_persist;
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want) == cudaSuccess) {
        e->window.base_ptr = e->hot_arena;
        e->window.num_bytes = e->hot_bytes < (size_t)max_win ? e->hot_bytes : (size_t)max_win;
        e->window.hitRatio = (float)((double)want / (double)e->window.num_bytes > 1.0 ? 1.0 : (double)want / (double)e->window.num_bytes);
        e->window.hitProp = cudaAccessPropertyPersisting;
        e->window.missProp = cudaAccessPropertyStreaming;
        e->use_window = true;
      } else cudaGetLastError();
    }
  }
  uint32_t bits = 1;
  while ((1ULL << bits) < groups) bits++;
  c.sort_passes = (bits + 7) / 8;

  if (e->has_log) {
    if ((rc = dalloc(e, &c.ring, (size_t)c.ring_n * kLogEntry[e->kind]))) return rc;
  }
  // ---- chunk scratch ----
  const uint32_t ch = e->chunk;
  e->max_tiles = (ch + kTile - 1) / kTile;
  for (int i = 0; i < 2; i++)
    if ((rc = dalloc(e, &e->d_grp[i], ch))) return rc;
  if ((rc = dalloc(e, &c.clist, (size_t)e->max_tiles * kTile))) return rc;
  if ((rc = dalloc(e, &c.ccnt, e->max_tiles))) return rc;
  if ((rc = dalloc(e, &c.cprefix, e->max_tiles + 1))) return rc;
  if ((rc = dalloc(e, &e->d_nc, 8))) return rc;
  {
    uint32_t lg = 0;
    while (((uint64_t)kBucketFill << lg) < ch) lg++;
    c.bucket_log2 = lg;
    if ((rc = dalloc(e, &c.buckets, ((size_t)1 << lg) * kBucketCap, false))) return rc;
    if ((rc = dalloc(e, &c.bcnt, (size_t)1 << lg))) return rc;
  }
  if ((rc = dalloc(e, &c.sortA, ch))) return rc;
  if ((rc = dalloc(e, &c.sortB, ch))) return rc;
  if ((rc = dalloc(e, &c.ghist, (size_t)256 * ((ch + kSortTile - 1) / kSortTile)))) return rc;
  if ((rc = dalloc(e, &c.rowtot, 256))) return rc;
  if ((rc = dalloc(e, &c.log_tilecnt, e->max_tiles))) return rc;
  if ((rc = dalloc(e, &c.log_tilebase, e->max_tiles))) return rc;
  if ((rc = dalloc(e, &c.log_total, 2))) return rc;
  if ((rc = dalloc(e, &c.counters, 4))) return rc;
  if ((rc = dalloc(e, &c.gbar, 4))) return rc;

  switch (e->kind) {
    case DINT_LOCK2PL: rc = grids_for<K_LOCK2PL, false>(e); break;
    case DINT_FASST: rc = grids_for<K_FASST, false>(e); break;
    case DINT_LOG: rc = grids_for<K_LOG, true>(e); break;
    case DINT_STORE: rc = grids_for<K_STORE, false>(e); break;
    case DINT_TATP: rc = grids_for<K_TATP, true>(e); break;
    default: rc = grids_for<K_SMALLBANK, true>(e); break;
  }
  if (rc) return rc;
  int coop = 0;
  CU(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, e->device));
  if (!coop) return set_err(DINT_ENODEV, "device lacks cooperative launch");
  CU(cudaStreamSynchronize(e->stream));
  return DINT_OK;
}

int dint_create(int kind, const dint_cfg* cfg, int device, dint_engine** out) {
  if (!out || kind < 0 || kind >= DINT_NUM_KINDS) return set_err(DINT_EINVAL, "bad kind/out");
  *out = nullptr;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return set_err(DINT_ENODEV, "no CUDA device: dint_b200 has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return set_err(DINT_EINVAL, "bad device ordinal");
  dint_engine* e = new dint_engine();
  e->kind = kind;
  e->device = device;
  if (cfg) e->cfg = *cfg; else dint_default_cfg(kind, &e->cfg);
  dint_cfg& cf = e->cfg;
  if (cf.n_shards == 0) cf.n_shards = 1;
  if (cf.shard_id >= cf.n_shards || cf.lock_slots == 0) { delete e; return set_err(DINT_EINVAL, "bad shard/lock_slots"); }
  if (cf.chunk == 0) cf.chunk = 1u << 20;
  e->chunk = (cf.chunk + kTile - 1) / kTile * kTile;
  {
    // host-path slice schedule (measured, tools/e2e_probe.py round 1: every schedule between 128 K and 1 M lands within 5 %)
    const uint32_t want = 1u << 18;
    e->host_chunk = want < e->chunk ? want : e->chunk;
    e->host_min_slice = 131072u;
    e->host_ramp_up = true;
  }
  e->msg = kMsgSize[kind];
  e->has_log = kLogEntry[kind] != 0;
  int rc = create_impl(e);
  if (rc) { dint_destroy(e); return rc; }
  *out = e;
  return DINT_OK;
}

int dint_route_owner(dint_engine* e, const void* req_dev, uint64_t n, uint8_t* owner_dev, void* cuda_stream) {
  if (!e || (n && (!req_dev || !owner_dev)) || n > 0xffffffffULL) return set_err(DINT_EINVAL, "bad argument");
  if (n == 0) return DINT_OK;
  CU(cudaSetDevice(e->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const uint32_t blocks = (uint32_t)((n + kThreads - 1) / kThreads);
  const uint8_t* rq = (const uint8_t*)req_dev;
  e->stats.kernel_launches++;
  switch (e->kind) {
    case DINT_LOCK2PL: k_route_owner<K_LOCK2PL><<<blocks, kThreads, 0, s>>>(e->ctx, rq, (uint32_t)n, owner_dev); break;
    case DINT_FASST: k_route_owner<K_FASST><<<blocks, kThreads, 0, s>>>(e->ctx, rq, (uint32_t)n, owner_dev); break;
    case DINT_LOG: k_route_owner<K_LOG><<<blocks, kThreads, 0, s>>>(e->ctx, rq, (uint32_t)n, owner_dev); break;
    case DINT_STORE: k_route_owner<K_STORE><<<blocks, kThreads, 0, s>>>(e->ctx, rq, (uint32_t)n, owner_dev); break;
    case DINT_TATP: k_route_owner<K_TATP><<<blocks, kThreads, 0, s>>>(e->ctx, rq, (uint32_t)n, owner_dev); break;
    default: k_route_owner<K_SMALLBANK><<<blocks, kThreads, 0, s>>>(e->ctx, rq, (uint32_t)n, owner_dev); break;
  }
  CU(cudaGetLastError());
  return DINT_OK;
}

int dint_route_partition(dint_engine* e, const void* req_dev, const uint8_t* owner_dev, uint64_t n, uint32_t n_shards,
                         void* sorted_dev, uint32_t* perm_dev, uint32_t* counts_dev, void* cuda_stream) {
  if (!e || n_shards == 0 || n_shards > kMaxShards || n > 0xffffffffULL) return set_err(DINT_EINVAL, "bad argument");
  CU(cudaSetDevice(e->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const uint32_t tiles = (uint32_t)((n + kThreads - 1) / kThreads);
  if (tiles > e->route_tiles) {                          // scratch: per-tile per-shard counts + totals
    if (e->d_route) { CU(cudaFree(e->d_route)); e->d_route = nullptr; }
    e->route_tiles = tiles + tiles / 2 + 64;
    CU(cudaMalloc(&e->d_route, ((size_t)e->route_tiles * kMaxShards + 3 * kMaxShards) * sizeof(uint32_t)));
  }
  uint32_t* totals = e->d_route;                         // [0..8) records per shard
  uint32_t* tilecnt = e->d_route + 3 * kMaxShards;
  if (n == 0) { CU(cudaMemsetAsync(counts_dev, 0, n_shards * sizeof(uint32_t), s)); return DINT_OK; }
  e->stats.kernel_launches += 3;
  k_exact_count<<<tiles, kThreads, 0, s>>>(owner_dev, (uint32_t)n, n_shards, tilecnt);
  k_exact_scan<<<n_shards, kThreads, 0, s>>>(tilecnt, tiles, totals);
  const uint8_t* rq = (const uint8_t*)req_dev;
  uint8_t* out = (uint8_t*)sorted_dev;
  switch (e->msg) {
    case 6: route_scatter_t<6>(rq, owner_dev, (uint32_t)n, n_shards, tilecnt, totals, out, perm_dev, tiles, s); break;
    case 9: route_scatter_t<9>(rq, owner_dev, (uint32_t)n, n_shards, tilecnt, totals, out, perm_dev, tiles, s); break;
    case 23: route_scatter_t<23>(rq, owner_dev, (uint32_t)n, n_shards, tilecnt, totals, out, perm_dev, tiles, s); break;
    case 53: route_scatter_t<53>(rq, owner_dev, (uint32_t)n, n_shards, tilecnt, totals, out, perm_dev, tiles, s); break;
    default: route_scatter_t<55>(rq, owner_dev, (uint32_t)n, n_shards, tilecnt, totals, out, perm_dev, tiles, s); break;
  }
  CU(cudaMemcpyAsync(counts_dev, totals, n_shards * sizeof(uint32_t), cudaMemcpyDeviceToDevice, s));
  CU(cudaGetLastError());
  return DINT_OK;
}

uint32_t dint_route_tile_records(dint_engine* e) { return e ? route_tile_records(e) : 0; }

int dint_route_dispatch(dint_engine* e, const void* req_dev, const uint8_t* owner_in_dev, uint64_t n, uint32_t n_shards, uint32_t rank,
                        uint32_t cap, const dint_peer_ptrs* slab_ptrs, const dint_peer_ptrs* sig_ptrs, uint32_t epoch,
                        uint8_t* owner_dev, uint32_t* tilebase_dev, uint32_t* flags_dev, void* cuda_stream) {
  if (!e || !slab_ptrs || !flags_dev || n_shards == 0 || n_shards > kMaxShards || rank >= n_shards || cap == 0 || n >= (1ULL << 27) ||
      (n && (!req_dev || !owner_dev || !tilebase_dev)))
    return set_err(DINT_EINVAL, "bad argument");
  if ((uintptr_t)req_dev & 15) return set_err(DINT_EINVAL, "device buffers must be 16-byte aligned");
  if (!owner_in_dev && n_shards != e->ctx.n_shards) return set_err(DINT_EINVAL, "owner computation needs n_shards == cfg.n_shards");
  CU(cudaSetDevice(e->device));
  RouteArgs a{};
  a.req = (const uint8_t*)req_dev;
  a.owner_in = owner_in_dev;
  a.owner = owner_dev;
  a.tilebase = tilebase_dev;
  a.flags = flags_dev;
  a.n = (uint32_t)n;
  a.n_tiles = (uint32_t)((n + route_tile_records(e) - 1) / route_tile_records(e));
  a.world = n_shards;
  a.me = rank;
  a.cap = cap;
  a.epoch = epoch;
  for (uint32_t i = 0; i < kMaxShards; i++) { a.slab.p[i] = slab_ptrs->p[i]; a.sig.p[i] = sig_ptrs ? sig_ptrs->p[i] : 0; }
  cudaStream_t s = (cudaStream_t)cuda_stream;
  e->stats.kernel_launches += 1;
  switch (e->kind) {
    case DINT_LOCK2PL: return route_dispatch_t<K_LOCK2PL>(e, a, s);
    case DINT_FASST: return route_dispatch_t<K_FASST>(e, a, s);
    case DINT_LOG: return route_dispatch_t<K_LOG>(e, a, s);
    case DINT_STORE: return route_dispatch_t<K_STORE>(e, a, s);
    case DINT_TATP: return route_dispatch_t<K_TATP>(e, a, s);
    default: return route_dispatch_t<K_SMALLBANK>(e, a, s);
  }
}

int dint_route_combine(dint_engine* e, const dint_peer_ptrs* reply_slab_ptrs, const uint8_t* owner_dev, const uint32_t* tilebase_dev,
                       uint64_t n, uint32_t n_shards, uint32_t cap, void* out_dev, void* cuda_stream) {
  if (!e || !reply_slab_ptrs || n_shards == 0 || n_shards > kMaxShards || cap == 0 || n > 0xffffffffULL ||
      (n && (!owner_dev || !tilebase_dev || !out_dev)))
    return set_err(DINT_EINVAL, "bad argument");
  if ((uintptr_t)out_dev & 15) return set_err(DINT_EINVAL, "device buffers must be 16-byte aligned");
  if (n == 0) return DINT_OK;
  CU(cudaSetDevice(e->device));
  RouteArgs a{};
  a.owner = (uint8_t*)owner_dev;
  a.tilebase = (uint32_t*)tilebase_dev;
  a.out = (uint8_t*)out_dev;
  a.n = (uint32_t)n;
  a.n_tiles = (uint32_t)((n + route_tile_records(e) - 1) / route_tile_records(e));
  a.world = n_shards;
  a.cap = cap;
  for (uint32_t i = 0; i < kMaxShards; i++) a.slab.p[i] = reply_slab_ptrs->p[i];
  cudaStream_t s = (cudaStream_t)cuda_stream;
  e->stats.kernel_launches++;
  switch (e->msg) {
    case 6: return route_combine_t<6>(e, a, s);
    case 9: return route_combine_t<9>(e, a, s);
    case 23: return route_combine_t<23>(e, a, s);
    case 53: return route_combine_t<53>(e, a, s);
    default: return route_combine_t<55>(e, a, s);
  }
}

int dint_p2p_wait(dint_engine* e, const uint32_t* local_sig_dev, uint32_t n_shards, uint32_t epoch, uint32_t* flags_dev, void* cuda_stream) {
  if (!e || !local_sig_dev || n_shards == 0 || n_shards > kMaxShards) return set_err(DINT_EINVAL, "bad argument");
  CU(cudaSetDevice(e->device));
  e->stats.kernel_launches++;
  k_p2p_wait<<<1, 32, 0, (cudaStream_t)cuda_stream>>>(local_sig_dev, n_shards, epoch, flags_dev + 1, nullptr);
  CU(cudaGetLastError());
  return DINT_OK;
}

int dint_p2p_signal(dint_engine* e, const dint_peer_ptrs* sig_ptrs, uint32_t n_shards, uint32_t rank, uint32_t epoch, void* cuda_stream) {
  if (!e || !sig_ptrs || n_shards == 0 || n_shards > kMaxShards || rank >= n_shards) return set_err(DINT_EINVAL, "bad argument");
  CU(cudaSetDevice(e->device));
  PeerPtrs sg{};
  for (uint32_t i = 0; i < kMaxShards; i++) sg.p[i] = sig_ptrs->p[i];
  e->stats.kernel_launches++;
  k_p2p_signal<<<1, 32, 0, (cudaStream_t)cuda_stream>>>(sg, n_shards, rank, epoch);
  CU(cudaGetLastError());
  return DINT_OK;
}

int dint_route_unpermute(dint_engine* e, const void* sorted_dev, const uint32_t* perm_dev, uint64_t n, void* out_dev, void* cuda_stream) {
  if (!e || n > 0xffffffffULL) return set_err(DINT_EINVAL, "bad argument");
  if (n == 0) return DINT_OK;
  CU(cudaSetDevice(e->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  e->stats.kernel_launches++;
  const uint8_t* in = (const uint8_t*)sorted_dev;
  uint8_t* out = (uint8_t*)out_dev;
  switch (e->msg) {
    case 6: route_unpermute_t<6>(in, perm_dev, (uint32_t)n, out, s); break;
    case 9: route_unpermute_t<9>(in, perm_dev, (uint32_t)n, out, s); break;
    case 23: route_unpermute_t<23>(in, perm_dev, (uint32_t)n, out, s); break;
    case 53: route_unpermute_t<53>(in, perm_dev, (uint32_t)n, out, s); break;
    default: route_unpermute_t<55>(in, perm_dev, (uint32_t)n, out, s); break;
  }
  CU(cudaGetLastError());
  return DINT_OK;
}

int dint_sync(dint_engine* e) {
  if (!e) return DINT_EINVAL;
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  int rc = prof_flush(e);
  if (rc) return rc;
  unsigned long long before = e->stats.errors;
  if ((rc = pull_counters(e))) return rc;
  return e->stats.errors != before ? DINT_EPROTO : DINT_OK;
}

int dint_submit_device(dint_engine* e, const void* req_dev, uint64_t n, void* resp_dev, void* cuda_stream) {
  if (!e || (n && (!req_dev || !resp_dev))) return set_err(DINT_EINVAL, "null argument");
  if (((uintptr_t)req_dev | (uintptr_t)resp_dev) & 15) return set_err(DINT_EINVAL, "device buffers must be 16-byte aligned");
  CU(cudaSetDevice(e->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;        // NULL = the legacy default stream, as in every CUDA API
  return run_device(e, (const uint8_t*)req_dev, n, (uint8_t*)resp_dev, s);
}

int dint_submit(dint_engine* e, const void* req, uint64_t n, void* resp) {
  if (!e || (n && (!req || !resp))) return set_err(DINT_EINVAL, "null argument");
  CU(cudaSetDevice(e->device));
  // the host path moves data in slices of `hchunk` requests through a ring of kHostBufs device buffers:
  // small slices keep the PCIe fill/drain bubbles short, the ring keeps both copy engines and the SMs busy
  const uint32_t hchunk = e->host_chunk;
  if (!e->d_req[0]) {
    for (int i = 0; i < kHostBufs; i++) {
      int rc;
      if ((rc = dalloc(e, &e->d_req[i], (size_t)hchunk * e->msg + 16, false))) return rc;
      if ((rc = dalloc(e, &e->d_resp[i], (size_t)hchunk * e->msg + 16, false))) return rc;
    }
  }
  static const bool trace = getenv("DINT_HOST_TRACE") != nullptr;
  const auto t_begin = std::chrono::steady_clock::now();
  CU(cudaDeviceSynchronize());     // order after anything submitted on user streams
  { int rc = kv_maintain(e, e->stream); if (rc) return rc; }
  const uint8_t* rq = (const uint8_t*)req;
  uint8_t* rs = (uint8_t*)resp;
  unsigned long long err_before = e->stats.errors;
  // (Zero-copy replies -- K2 storing straight into pinned host memory instead of a D2H stage -- were measured in
  // round 2 and dropped: 1.42 vs 1.73 G req/s at 2^20 requests per call, profiles/r02_variants.md.)
  // three-stage pipeline: H2D (s_in) | kernels (stream) | D2H (s_out).  Slice k's replies are final only
  // after the launch that replays its listed requests -- K1 of slice k+1, or the flush after the last
  // slice -- so D2H(k) is ordered behind that.
  uint64_t k = 0;
  uint64_t prev_off = 0, prev_bytes = 0;
  auto copy_out_prev = [&](uint64_t kk) -> int {          // D2H of slice kk-1
    int pb = (int)((kk - 1) % kHostBufs);
    CU(cudaEventRecord(e->ev_comp[pb], e->stream));
    CU(cudaStreamWaitEvent(e->s_out, e->ev_comp[pb], 0));
    CU(cudaMemcpyAsync(rs + prev_off, e->d_resp[pb], prev_bytes, cudaMemcpyDeviceToHost, e->s_out));
    CU(cudaEventRecord(e->ev_out[pb], e->s_out));
    return DINT_OK;
  };
  // Slice schedule.  PCIe moves large copies better than small ones (B200 box, pinned, both directions busy:
  // 37 GB/s per direction at 2.4 MB, 46 at 9.4 MB, 50 at 38 MB: tools/pcie_probe.cu), but the first slice's
  // H2D and the last two slices' kernels + D2H overlap with nothing.  So a call is cut as a pyramid: slices
  // double from host_min_slice up to host_chunk, stay there, and halve back down at the end.  (Measured with
  // tools/e2e_probe.py: every schedule between 128K..1M slices lands within 5 % -- the copies, not the
  // kernels or the launches (11 us of CPU per slice), are the bound: 1M requests = 345 us vs 203 us for two
  // perfectly overlapped 9.4 MB copies.)
  HostSlices sched(n, e->host_min_slice, hchunk, e->host_ramp_up);
  uint64_t off = 0;
  for (uint64_t cn; (cn = sched.next()) != 0; k++) {
    int b = (int)(k % kHostBufs);
    size_t bytes = (size_t)cn * e->msg;
    if (k >= (uint64_t)kHostBufs) CU(cudaStreamWaitEvent(e->s_in, e->ev_comp[b], 0));   // slice k-kHostBufs no longer read
    CU(cudaMemcpyAsync(e->d_req[b], rq + off * e->msg, bytes, cudaMemcpyHostToDevice, e->s_in));
    CU(cudaEventRecord(e->ev_in[b], e->s_in));
    CU(cudaStreamWaitEvent(e->stream, e->ev_in[b], 0));
    if (k >= (uint64_t)kHostBufs) CU(cudaStreamWaitEvent(e->stream, e->ev_out[b], 0)); // its replies have left d_resp[b]
    int rc = submit_chunk(e, e->d_req[b], (uint32_t)cn, e->d_resp[b], e->stream);
    if (rc) return rc;
    if (k >= 1 && (rc = copy_out_prev(k))) return rc;                   // slice k-1 is final now
    prev_off = off * e->msg;
    prev_bytes = bytes;
    e->stats.h2d_bytes += bytes;
    e->stats.d2h_bytes += bytes;
    off += cn;
  }
  {
    int rc = flush_ordered(e, e->stream);
    if (rc) return rc;
    if (k >= 1 && (rc = copy_out_prev(k))) return rc;
  }
  if (!e->h_counters) CU(cudaHostAlloc((void**)&e->h_counters, 4 * sizeof(unsigned long long), cudaHostAllocDefault));
  CU(cudaMemcpyAsync(e->h_counters, e->ctx.counters, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
  { int rc2 = kv_publish_counts(e, e->stream); if (rc2) return rc2; }
  const auto t_enq = std::chrono::steady_clock::now();
  CU(cudaStreamSynchronize(e->s_out));
  CU(cudaStreamSynchronize(e->stream));
  int rc = prof_flush(e);
  if (rc) return rc;
  if (trace) {
    const auto t_end = std::chrono::steady_clock::now();
    fprintf(stderr, "[dint_submit] n=%llu slices=%llu enqueue=%.1f us total=%.1f us\n", (unsigned long long)n, (unsigned long long)k,
            std::chrono::duration<double, std::micro>(t_enq - t_begin).count(),
            std::chrono::duration<double, std::micro>(t_end - t_begin).count());
  }
  e->stats.errors = e->h_counters[0];
  e->stats.conflicted = e->h_counters[1];
  e->stats.max_run = e->h_counters[2];
  e->stats.fallback_chunks = e->h_counters[3];
  return e->stats.errors != err_before ? DINT_EPROTO : DINT_OK;
}

// ---- state snapshots (checkpoint / restore of one engine's whole server state, device to device) --------------
struct dint_snapshot {
  dint_engine* e = nullptr;
  std::vector<std::pair<void*, size_t>> live;   // the engine's state arrays
  std::vector<void*> copy;
  uint64_t kv_cap[kMaxTables]{};                 // table capacities at snapshot time (a rehash in between invalidates it)
};
static void snapshot_regions(dint_engine* e, std::vector<std::pair<void*, size_t>>& r) {
  const Ctx& c = e->ctx;
  const uint64_t g = e->total_groups;
  if (e->kind == DINT_LOCK2PL || e->kind == DINT_SMALLBANK) r.push_back({c.cnt2, g * sizeof(uint2)});
  if (e->kind == DINT_FASST) { r.push_back({c.ver, g * sizeof(uint32_t)}); r.push_back({c.lockbits, ((g + 31) / 32) * 4}); }
  if (e->kind == DINT_TATP) r.push_back({c.lockbits, ((g + 31) / 32) * 4});
  for (uint32_t t = 0; t < c.n_tables; t++) {
    r.push_back({c.tbl[t].entries, (size_t)(c.tbl[t].cap_mask + 1) << c.tbl[t].ent_shift});
    r.push_back({c.tbl[t].live, 16});
  }
  if (e->has_log) { r.push_back({c.ring, (size_t)c.ring_n * kLogEntry[e->kind]}); r.push_back({c.log_total, 2 * sizeof(unsigned long long)}); }
}
int dint_snapshot_create(dint_engine* e, dint_snapshot** out) {
  if (!e || !out) return set_err(DINT_EINVAL, "null argument");
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  dint_snapshot* s = new dint_snapshot();
  s->e = e;
  snapshot_regions(e, s->live);
  for (uint32_t t = 0; t < e->ctx.n_tables; t++) s->kv_cap[t] = e->ctx.tbl[t].cap_mask + 1;
  for (auto& r : s->live) {
    void* p = nullptr;
    cudaError_t ce = cudaMalloc(&p, r.second ? r.second : 1);
    if (ce != cudaSuccess) { for (void* q : s->copy) cudaFree(q); delete s; return set_err(DINT_ENOMEM, "snapshot", ce); }
    s->copy.push_back(p);
    CU(cudaMemcpyAsync(p, r.first, r.second, cudaMemcpyDeviceToDevice, e->stream));
  }
  CU(cudaStreamSynchronize(e->stream));
  *out = s;
  return DINT_OK;
}
int dint_snapshot_restore(dint_snapshot* s, void* cuda_stream) {
  if (!s) return set_err(DINT_EINVAL, "null argument");
  dint_engine* e = s->e;
  CU(cudaSetDevice(e->device));
  for (uint32_t t = 0; t < e->ctx.n_tables; t++)
    if (s->kv_cap[t] != e->ctx.tbl[t].cap_mask + 1) return set_err(DINT_EINVAL, "a KV table was rehashed since the snapshot");
  std::vector<std::pair<void*, size_t>> now;
  snapshot_regions(e, now);
  if (now.size() != s->live.size()) return set_err(DINT_EINVAL, "snapshot does not match the engine");
  for (size_t i = 0; i < now.size(); i++) {
    if (now[i].second != s->live[i].second) return set_err(DINT_EINVAL, "snapshot does not match the engine");
    CU(cudaMemcpyAsync(now[i].first, s->copy[i], now[i].second, cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream));
  }
  return DINT_OK;
}
void dint_snapshot_destroy(dint_snapshot* s) {
  if (!s) return;
  cudaSetDevice(s->e->device);
  for (void* p : s->copy) cudaFree(p);
  delete s;
}

int dint_lock_state(dint_engine* e, int table, uint32_t slot, uint32_t out[2]) {
  if (!e || !out) return DINT_EINVAL;
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  out[0] = out[1] = 0;
  const Ctx& c = e->ctx;
  uint32_t g = slot;
  if (e->kind == DINT_TATP || e->kind == DINT_SMALLBANK) {
    if (table < 0 || table >= (int)c.n_tables) return DINT_EINVAL;
    if (slot % c.n_shards != c.shard_id) return DINT_EINVAL;
    g = c.tbl[table].grp_base + slot / c.n_shards;
  } else if (e->kind == DINT_LOCK2PL || e->kind == DINT_FASST) {
    if (slot % c.n_shards != c.shard_id) return DINT_EINVAL;
    g = slot / c.n_shards;
  } else return DINT_EINVAL;
  if (g >= e->total_groups) return DINT_EINVAL;
  if (e->kind == DINT_LOCK2PL || e->kind == DINT_SMALLBANK) {
    uint2 v;
    CU(cudaMemcpy(&v, c.cnt2 + g, sizeof v, cudaMemcpyDeviceToHost));
    out[0] = v.x; out[1] = v.y;
  } else {
    uint32_t w;
    CU(cudaMemcpy(&w, c.lockbits + (g >> 5), 4, cudaMemcpyDeviceToHost));
    out[0] = (w >> (g & 31)) & 1u;
    if (e->kind == DINT_FASST) CU(cudaMemcpy(&out[1], c.ver + g, 4, cudaMemcpyDeviceToHost));
  }
  return DINT_OK;
}

uint32_t dint_lock_slot(dint_engine* e, int table, uint64_t k) {
  if (!e) return 0;
  const Ctx& c = e->ctx;
  if (e->kind == DINT_LOCK2PL || e->kind == DINT_FASST) return fast_mod(fasthash64_u32((uint32_t)k), c.slot_mod);
  if ((e->kind == DINT_TATP || e->kind == DINT_SMALLBANK) && table >= 0 && table < (int)c.n_tables)
    return fast_mod(fasthash64_u64(k), c.tbl[table].lock_mod);
  return 0;
}

int dint_dump_log(dint_engine* e, void* out, uint64_t* appended) {
  if (!e || !e->has_log) return DINT_EINVAL;
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  if (out) CU(cudaMemcpy(out, e->ctx.ring, (size_t)e->ctx.ring_n * kLogEntry[e->kind], cudaMemcpyDeviceToHost));
  if (appended) {
    unsigned long long t[2];
    CU(cudaMemcpy(t, e->ctx.log_total, sizeof t, cudaMemcpyDeviceToHost));
    *appended = t[0];
  }
  return DINT_OK;
}

int dint_get_stats(dint_engine* e, dint_stats* s) {
  if (!e || !s) return DINT_EINVAL;
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  int rc = pull_counters(e);
  if (rc) return rc;
  *s = e->stats;
  return DINT_OK;
}
void dint_reset_stats(dint_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  cudaMemset(e->ctx.counters, 0, 4 * sizeof(unsigned long long));
  e->stats = dint_stats{};
  for (int i = 0; i < KT_NUM; i++) { e->kt_ms[i] = 0; e->kt_n[i] = 0; }
}
int dint_profile(dint_engine* e, int enable) {
  if (!e) return DINT_EINVAL;
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  int rc = prof_flush(e);
  e->profiling = enable < 0 ? 0u : (uint32_t)enable == 1u ? 0xffffffffu : (uint32_t)enable;   // 1 = all kernels; else a bit mask
  return rc;
}
int dint_kernel_times(dint_engine* e, dint_kernel_time* out, int max_entries) {
  if (!e || !out) return DINT_EINVAL;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  prof_flush(e);
  int k = 0;
  for (int i = 0; i < KT_NUM && k < max_entries; i++) {
    if (!e->kt_n[i]) continue;
    memset(&out[k], 0, sizeof out[k]);
    snprintf(out[k].name, sizeof out[k].name, "%s", kKernelNames[i]);
    out[k].launches = e->kt_n[i];
    out[k].total_ms = e->kt_ms[i];
    k++;
  }
  return k;
}

// ---- KV entry points (store / tatp / smallbank) -------------------------------------------------------
int dint_load(dint_engine* e, int table, const uint64_t* keys, const void* vals, uint64_t n) {
  if (!e || table < 0 || table >= (int)e->ctx.n_tables || (n && (!keys || !vals))) return set_err(DINT_EINVAL, "bad table/arguments");
  CU(cudaSetDevice(e->device));
  const uint32_t vs = kValSize[e->kind];
  const uint64_t batch = 1u << 20;
  uint64_t* dk = nullptr;
  uint8_t* dv = nullptr;
  CU(cudaMalloc(&dk, batch * 8));
  cudaError_t ce = cudaMalloc(&dv, batch * vs);
  if (ce != cudaSuccess) { cudaFree(dk); return set_err(DINT_ENOMEM, "cudaMalloc", ce); }
  int rc = pull_counters(e);                      // failures are counted in counters[0]: compare against its value NOW, not against 0
  const unsigned long long err_before = e->stats.errors;
  for (uint64_t off = 0; off < n && rc == DINT_OK; off += batch) {
    uint64_t m = (n - off < batch) ? (n - off) : batch;
    if (cudaMemcpyAsync(dk, keys + off, m * 8, cudaMemcpyHostToDevice, e->stream) != cudaSuccess ||
        cudaMemcpyAsync(dv, (const uint8_t*)vals + off * vs, m * vs, cudaMemcpyHostToDevice, e->stream) != cudaSuccess) {
      rc = set_err(DINT_EIO, "load copy", cudaGetLastError());
      break;
    }
    {
      ProfScope ps(e, e->stream, KT_LOAD);
      kv_launch_load(e->kind, e->ctx, table, dk, dv, (uint32_t)m, e->stream);
    }
    if (cudaStreamSynchronize(e->stream) != cudaSuccess) rc = set_err(DINT_EIO, "k_kv_load", cudaGetLastError());
  }
  cudaFree(dk);
  cudaFree(dv);
  if (rc == DINT_OK) {
    kv_publish_counts(e, e->stream);
    cudaStreamSynchronize(e->stream);
    int r2 = pull_counters(e);
    if (r2) return r2;
    if (e->stats.errors != err_before) return set_err(DINT_ENOMEM, "KV table full during load");
  }
  return rc;
}

int dint_populate(dint_engine* e) {
  if (!e) return DINT_EINVAL;
  if (e->ctx.n_tables == 0) return DINT_OK;       // lock / log servers start from zeroed arrays
  return kv_populate(e->kind, e->cfg, [&](int table, const uint64_t* k, const void* v, uint64_t n) {
    return dint_load(e, table, k, v, n);
  });
}

int dint_kv_get(dint_engine* e, int table, uint64_t key, void* val, uint32_t* ver) {
  if (!e || table < 0 || table >= (int)e->ctx.n_tables) return DINT_EINVAL;
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  return kv_host_get(e->ctx, table, key, kValSize[e->kind], val, ver);
}

int64_t dint_kv_count(dint_engine* e, int table) {
  if (!e || table < 0 || table >= (int)e->ctx.n_tables) return DINT_EINVAL;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  unsigned long long v = 0;
  if (cudaMemcpy(&v, e->ctx.tbl[table].live, 8, cudaMemcpyDeviceToHost) != cudaSuccess) return DINT_EIO;
  return (int64_t)v;
}

}  // extern "C"

// ---- the whole sharded step over NVLink peer memory ---------------------------------------------------------
// A "rank" = one engine (one shard of the key space) with three streams: `side` partitions batch j+1 into the
// OWNERS' inboxes (dispatch), the caller's stream runs the engine on batch j -- K2 stores every reply tile
// straight into its SOURCE's return buffer (Ctx::seg_resp; posted stores over NVLink) -- and `ret` reassembles
// the replies of batch j-1 from the local return buffer (combine).  Cross-GPU synchronisation: two arrays of
// epoch words per rank (requests written / replies written; st.release.sys / ld.acquire.sys, bounded spin);
// buffer reuse needs no third flag: a source re-fills inbox set s only after its combine of the batch that used
// it, i.e. after every owner's "replies written", and an owner re-fills return-buffer set s only after the
// source's next dispatch into that set arrived, which the source ordered behind its combine.
// Ranks may live in different processes (one per GPU, buffers mapped through CUDA IPC / torch symmetric memory:
// dint_shard_*) or in ONE process (dint_cluster_*: cudaMalloc + peer access; several ranks may even share a
// device, then everything runs on one stream in dependency order).
constexpr int kMaxSets = 4;
struct dint_shard_ctx {
  dint_engine* e = nullptr;
  uint32_t W = 0, me = 0, cap = 0, S = 0;
  uint64_t inbox[kMaxSets][kMaxShards]{}, retbox[kMaxSets][kMaxShards]{};
  PeerPtrs sigreq{}, sigrsp{};
  uint32_t *my_req = nullptr, *my_rsp = nullptr;
  uint32_t epoch = 0;
  cudaStream_t side = nullptr, ret = nullptr, s_in = nullptr, s_out = nullptr;
  cudaEvent_t ev_disp[kMaxSets]{}, ev_comb[kMaxSets]{}, ev_fork = nullptr;
  cudaEvent_t ev_h2d[kMaxSets]{}, ev_d2h[kMaxSets]{};
  uint8_t* owner[kMaxSets]{};
  uint32_t* tilebase[kMaxSets]{};
  uint8_t *st_req[kMaxSets]{}, *st_dst[kMaxSets]{}, *st_out[kMaxSets]{};   // host-path staging (allocated on first use)
  uint32_t* flags = nullptr;
  uint64_t max_n = 0;
  bool one_stream = false;                 // ranks sharing a device: dispatch, engine and combine on ONE stream, in dependency order
  bool trace = false;                      // DINT_SHARD_TRACE: per-phase CUDA-event timing, printed at destroy
  std::vector<cudaEvent_t> tev;            // 6 events per batch
  double tsum[4]{};
  uint64_t tcount = 0;
};

static int shard_make(dint_engine* e, uint32_t n_shards, uint32_t rank, uint32_t cap, uint32_t n_sets, const dint_peer_ptrs* inbox_sets,
                      const dint_peer_ptrs* retbox_sets, const dint_peer_ptrs* sig_blocks, uint64_t max_n, bool one_stream,
                      dint_shard_ctx** out) {
  if (!e || !out || !inbox_sets || !retbox_sets || !sig_blocks || n_shards == 0 || n_shards > kMaxShards || rank >= n_shards || cap == 0 ||
      cap % kTile != 0 || n_sets < 2 || n_sets > (uint32_t)kMaxSets || max_n == 0 || max_n > 0xffffffffULL)
    return set_err(DINT_EINVAL, "bad argument (cap must be a multiple of 128, 2 <= n_sets <= 4)");
  CU(cudaSetDevice(e->device));
  dint_shard_ctx* c = new dint_shard_ctx();
  e->plain_launches = true;
  c->e = e; c->W = n_shards; c->me = rank; c->cap = cap; c->S = n_sets; c->max_n = max_n; c->one_stream = one_stream;
  for (uint32_t s = 0; s < n_sets; s++)
    for (uint32_t o = 0; o < n_shards; o++) {
      c->inbox[s][o] = inbox_sets[s].p[o];
      c->retbox[s][o] = retbox_sets[s].p[o];
    }
  for (uint32_t o = 0; o < n_shards; o++) {
    c->sigreq.p[o] = sig_blocks->p[o];
    c->sigrsp.p[o] = sig_blocks->p[o] + 128;          // signal block: request flags [n_sets][8] at +0, reply flags [8] at +128
  }
  c->my_req = (uint32_t*)sig_blocks->p[rank];
  c->my_rsp = (uint32_t*)(sig_blocks->p[rank] + 128);
  if (!c->one_stream) {
    CU(cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c->ret, cudaStreamNonBlocking));
  }
  CU(cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
  const uint32_t tr = route_tile_records(e);
  const size_t tiles = (size_t)((max_n + tr - 1) / tr);
  for (uint32_t s = 0; s < n_sets; s++) {
    CU(cudaEventCreateWithFlags(&c->ev_disp[s], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_comb[s], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_h2d[s], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_d2h[s], cudaEventDisableTiming));
    CU(cudaMalloc(&c->owner[s], max_n + 16));
    CU(cudaMalloc(&c->tilebase[s], tiles * kMaxShards * sizeof(uint32_t)));
  }
  CU(cudaMalloc(&c->flags, 4 * sizeof(uint32_t)));        // [0] records that did not fit, [1] timed-out waits, [2] first epoch left unserved
  CU(cudaMemset(c->flags, 0, 4 * sizeof(uint32_t)));
  c->trace = getenv("DINT_SHARD_TRACE") != nullptr;
  *out = c;
  return DINT_OK;
}

// ---- the three phases of one batch on one rank (all asynchronous) -------------------------------------------
static void shard_mark(dint_shard_ctx* c, uint32_t slot, int which, cudaStream_t st) {
  if (!c->trace) return;
  const size_t need = (size_t)6 * (slot + 1);
  while (c->tev.size() < need) { cudaEvent_t ev; cudaEventCreate(&ev); c->tev.push_back(ev); }
  cudaEventRecord(c->tev[(size_t)6 * slot + which], st);
}
// dispatch: partition n records of this rank into the owners' inbox set (epoch ep)
// (cap: the slab capacity THIS batch uses, <= the capacity the buffers were laid out for and the same on every rank: a
//  batch much smaller than max_n then does not make the owners wade through padding)
static int shard_dispatch(dint_shard_ctx* c, uint32_t slot, uint32_t ep, const void* req_dev, const uint8_t* dst_dev, uint64_t n, uint32_t cap, cudaStream_t st) {
  dint_engine* e = c->e;
  CU(cudaSetDevice(e->device));
  const uint32_t s = ep % c->S;
  const size_t slab = (size_t)cap * e->msg;
  if (ep > c->S && !c->one_stream) CU(cudaStreamWaitEvent(st, c->ev_comb[s], 0));   // my combine of batch ep - S: every owner is done with inbox set s
  shard_mark(c, slot, 0, st);
  dint_peer_ptrs in{}, sg{};
  // one request-flag word per (buffer set, source): the flag of epoch ep -- which may carry the overflow bit -- is not
  // overwritten before the owner has consumed it (the source reuses set s only after the owners' replies of ep)
  for (uint32_t o = 0; o < c->W; o++) { in.p[o] = c->inbox[s][o] + (uint64_t)c->me * slab; sg.p[o] = c->sigreq.p[o] + (uint64_t)s * 32; }
  int rc = dint_route_dispatch(e, req_dev, dst_dev, n, c->W, c->me, cap, &in, &sg, ep, c->owner[s], c->tilebase[s], c->flags, st);
  if (rc) return rc;
  shard_mark(c, slot, 1, st);
  if (!c->one_stream) CU(cudaEventRecord(c->ev_disp[s], st));
  return DINT_OK;
}
// engine: this rank's shard serves inbox set (epoch ep); every reply tile goes to its source's return buffer
static int shard_engine(dint_shard_ctx* c, uint32_t slot, uint32_t ep, uint32_t cap, cudaStream_t st) {
  dint_engine* e = c->e;
  CU(cudaSetDevice(e->device));
  const uint32_t s = ep % c->S;
  const size_t slab = (size_t)cap * e->msg;
  k_p2p_wait<<<1, 32, 0, st>>>(c->my_req + s * 8, c->W, ep, c->flags + 1, c->flags + 2);     // every source's slab has arrived (or one did not fit)
  shard_mark(c, slot, 2, st);
  e->seg_tiles = cap / kTile;
  e->pad_ok = true;
  e->skip = c->flags + 2;
  for (uint32_t r = 0; r < c->W; r++) e->seg_resp[r] = c->retbox[s][r] + (uint64_t)c->me * slab;   // my slab inside source r's return buffer
  int rc = run_device(e, (const uint8_t*)c->inbox[s][c->me], (uint64_t)c->W * cap, nullptr, st);
  e->seg_tiles = 0;
  e->pad_ok = false;
  e->skip = nullptr;
  if (rc) return rc;
  k_p2p_signal<<<1, 32, 0, st>>>(c->sigrsp, c->W, c->me, ep);
  shard_mark(c, slot, 3, st);
  e->stats.kernel_launches += 2;
  return DINT_OK;
}
// combine: the replies of batch ep are in my return-buffer set; put them back in request order
static int shard_combine(dint_shard_ctx* c, uint32_t slot, uint32_t ep, void* out_dev, uint64_t n, uint32_t cap, cudaStream_t st) {
  dint_engine* e = c->e;
  CU(cudaSetDevice(e->device));
  const uint32_t s = ep % c->S;
  const size_t slab = (size_t)cap * e->msg;
  if (!c->one_stream) CU(cudaStreamWaitEvent(st, c->ev_disp[s], 0));
  k_p2p_wait<<<1, 32, 0, st>>>(c->my_rsp, c->W, ep, c->flags + 1, nullptr);
  shard_mark(c, slot, 4, st);
  dint_peer_ptrs rb{};
  for (uint32_t o = 0; o < c->W; o++) rb.p[o] = c->retbox[s][c->me] + (uint64_t)o * slab;
  int rc = dint_route_combine(e, &rb, c->owner[s], c->tilebase[s], n, c->W, cap, out_dev, st);
  if (rc) return rc;
  shard_mark(c, slot, 5, st);
  if (!c->one_stream) CU(cudaEventRecord(c->ev_comb[s], st));
  e->stats.kernel_launches += 1;
  return DINT_OK;
}
static void shard_trace_collect(dint_shard_ctx* c, uint32_t k) {
  if (!c->trace) return;
  cudaSetDevice(c->e->device);
  cudaDeviceSynchronize();
  static const int pairs[4][2] = {{0, 1}, {2, 3}, {4, 5}, {0, 5}};
  for (uint32_t j = 0; j < k && (size_t)6 * (j + 1) <= c->tev.size(); j++)
    for (int q = 0; q < 4; q++) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, c->tev[(size_t)6 * j + pairs[q][0]], c->tev[(size_t)6 * j + pairs[q][1]]) == cudaSuccess) c->tsum[q] += ms;
    }
  c->tcount += k;
}

// One pipelined sequence of k batches over the ranks of THIS process (1 in the one-process-per-GPU deployment,
// G in a cluster).  Host enqueue order per batch: every rank's dispatch of j+1, every rank's engine of j, every
// rank's combine of j (of j-1 when the ranks share one stream) -- each phase only waits for phases enqueued
// before it, on this or another GPU, so one host thread can drive all ranks without blocking.
struct ShardBatch { const void* req; const uint8_t* dst; void* out; uint64_t n; uint32_t cap = 0; };   // cap: slab records of this batch (0 = the full capacity)
struct HostBatch { const uint8_t* req; const uint8_t* dst; uint8_t* out; uint64_t n; };
static int shard_staging(dint_shard_ctx* c) {
  if (c->st_req[0]) return DINT_OK;
  CU(cudaSetDevice(c->e->device));
  for (uint32_t s = 0; s < c->S; s++) {
    CU(cudaMalloc(&c->st_req[s], c->max_n * c->e->msg + 16));
    CU(cudaMalloc(&c->st_dst[s], c->max_n + 16));
    CU(cudaMalloc(&c->st_out[s], c->max_n * c->e->msg + 16));
  }
  return DINT_OK;
}
// `host` given: the batches come from / go to HOST memory through S staging sets -- H2D of batch j+1 (copy stream) and
// D2H of batch j-1 (another copy stream) run next to the exchange of batch j, the same slice ring as dint_submit.
static int shard_run(dint_shard_ctx* const* ranks, uint32_t R, uint32_t k, std::vector<std::vector<ShardBatch>>& b, cudaStream_t const* mains,
                     const std::vector<std::vector<HostBatch>>* host = nullptr) {
  if (k == 0) return DINT_OK;
  const bool one = ranks[0]->one_stream;
  const uint32_t lag = one ? 1u : 0u;
  int rc;
  for (uint32_t r = 0; r < R; r++) {
    dint_shard_ctx* c = ranks[r];
    if (host && (rc = shard_staging(c))) return rc;
    if (one) continue;
    CU(cudaSetDevice(c->e->device));
    CU(cudaEventRecord(c->ev_fork, mains[r]));
    CU(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
    CU(cudaStreamWaitEvent(c->ret, c->ev_fork, 0));
  }
  auto side = [&](uint32_t r) { return one ? mains[r] : ranks[r]->side; };
  auto retS = [&](uint32_t r) { return one ? mains[r] : ranks[r]->ret; };
  auto dispatch = [&](uint32_t r, uint32_t j) -> int {
    dint_shard_ctx* c = ranks[r];
    if (host) {                                          // stage batch j: H2D on the copy stream, the dispatch waits for it
      const HostBatch& h = (*host)[r][j];
      dint_engine* e = c->e;
      const uint32_t s = j % c->S;
      if (h.n > c->max_n) return set_err(DINT_EINVAL, "batch size");
      CU(cudaSetDevice(e->device));
      CU(cudaStreamWaitEvent(c->s_in, c->ev_d2h[s], 0)); // batch j - S has left this staging set (its dispatch is long done too)
      if (h.n) CU(cudaMemcpyAsync(c->st_req[s], h.req, h.n * e->msg, cudaMemcpyHostToDevice, c->s_in));
      if (h.dst && h.n) CU(cudaMemcpyAsync(c->st_dst[s], h.dst, h.n, cudaMemcpyHostToDevice, c->s_in));
      CU(cudaEventRecord(c->ev_h2d[s], c->s_in));
      CU(cudaStreamWaitEvent(side(r), c->ev_h2d[s], 0));
      e->stats.h2d_bytes += h.n * e->msg + (h.dst ? h.n : 0);
      b[r][j] = ShardBatch{c->st_req[s], h.dst ? c->st_dst[s] : nullptr, c->st_out[s], h.n, 0};
    }
    return shard_dispatch(c, j, c->epoch + 1 + j, b[r][j].req, b[r][j].dst, b[r][j].n, b[r][j].cap ? b[r][j].cap : c->cap, side(r));
  };
  auto combine = [&](uint32_t r, uint32_t j) -> int {
    dint_shard_ctx* c = ranks[r];
    int rc2 = shard_combine(c, j, c->epoch + 1 + j, b[r][j].out, b[r][j].n, b[r][j].cap ? b[r][j].cap : c->cap, retS(r));
    if (rc2 || !host) return rc2;
    const HostBatch& h = (*host)[r][j];
    const uint32_t s = j % c->S, es = (c->epoch + 1 + j) % c->S;
    if (one) CU(cudaEventRecord(c->ev_comb[es], retS(r)));
    CU(cudaStreamWaitEvent(c->s_out, c->ev_comb[es], 0));
    if (h.n) CU(cudaMemcpyAsync(h.out, c->st_out[s], h.n * c->e->msg, cudaMemcpyDeviceToHost, c->s_out));
    CU(cudaEventRecord(c->ev_d2h[s], c->s_out));
    c->e->stats.d2h_bytes += h.n * c->e->msg;
    return DINT_OK;
  };
  for (uint32_t r = 0; r < R; r++)
    if ((rc = dispatch(r, 0))) return rc;
  for (uint32_t j = 0; j < k; j++) {
    if (j + 1 < k)
      for (uint32_t r = 0; r < R; r++)
        if ((rc = dispatch(r, j + 1))) return rc;
    for (uint32_t r = 0; r < R; r++)
      if ((rc = shard_engine(ranks[r], j, ranks[r]->epoch + 1 + j, b[r][j].cap ? b[r][j].cap : ranks[r]->cap, mains[r]))) return rc;
    if (j >= lag)
      for (uint32_t r = 0; r < R; r++)
        if ((rc = combine(r, j - lag))) return rc;
  }
  for (uint32_t j = k - (lag < k ? lag : k); j < k; j++)
    for (uint32_t r = 0; r < R; r++)
      if ((rc = combine(r, j))) return rc;
  for (uint32_t r = 0; r < R; r++) {
    dint_shard_ctx* c = ranks[r];
    const uint32_t last = c->epoch + k;
    c->epoch = last;
    if (one) continue;
    CU(cudaSetDevice(c->e->device));
    for (uint32_t s = 0; s < c->S && s < k; s++) CU(cudaStreamWaitEvent(mains[r], c->ev_comb[(last - s) % c->S], 0));   // join
    CU(cudaStreamWaitEvent(mains[r], c->ev_disp[last % c->S], 0));
  }
  CU(cudaGetLastError());
  if (host)
    for (uint32_t r = 0; r < R; r++) {                   // returns when every reply is in host memory
      CU(cudaSetDevice(ranks[r]->e->device));
      CU(cudaStreamSynchronize(ranks[r]->s_out));
      CU(cudaStreamSynchronize(mains[r]));
    }
  for (uint32_t r = 0; r < R; r++) shard_trace_collect(ranks[r], k);
  return DINT_OK;
}

static int shard_run_host(dint_shard_ctx* const* ranks, uint32_t R, uint32_t k, const std::vector<std::vector<HostBatch>>& hb) {
  std::vector<cudaStream_t> mains(R);
  for (uint32_t r = 0; r < R; r++) mains[r] = ranks[0]->one_stream ? ranks[0]->e->stream : ranks[r]->e->stream;   // ranks sharing a device: one stream
  std::vector<std::vector<ShardBatch>> b(R, std::vector<ShardBatch>(k));
  return shard_run(ranks, R, k, b, mains.data(), &hb);
}

extern "C" {

int dint_shard_create(dint_engine* e, uint32_t n_shards, uint32_t rank, uint32_t cap, uint32_t n_sets, const dint_peer_ptrs* inbox_sets,
                      const dint_peer_ptrs* retbox_sets, const dint_peer_ptrs* sig_blocks, uint64_t max_n, dint_shard_ctx** out) {
  return shard_make(e, n_shards, rank, cap, n_sets, inbox_sets, retbox_sets, sig_blocks, max_n, false, out);
}

void dint_shard_destroy(dint_shard_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->e->device);
  cudaDeviceSynchronize();
  if (c->trace && c->tcount) {
    static const char* names[4] = {"dispatch", "engine", "combine", "dispatch start -> combine end"};
    fprintf(stderr, "[dint_shard rank %u] %llu batches, us per batch:", c->me, (unsigned long long)c->tcount);
    for (int q = 0; q < 4; q++) fprintf(stderr, " | %s %.1f", names[q], c->tsum[q] * 1e3 / (double)c->tcount);
    fprintf(stderr, "\n");
  }
  for (cudaEvent_t ev : c->tev) cudaEventDestroy(ev);
  for (uint32_t s = 0; s < c->S; s++) {
    if (c->ev_disp[s]) cudaEventDestroy(c->ev_disp[s]);
    if (c->ev_comb[s]) cudaEventDestroy(c->ev_comb[s]);
    if (c->ev_h2d[s]) cudaEventDestroy(c->ev_h2d[s]);
    if (c->ev_d2h[s]) cudaEventDestroy(c->ev_d2h[s]);
    if (c->owner[s]) cudaFree(c->owner[s]);
    if (c->tilebase[s]) cudaFree(c->tilebase[s]);
    if (c->st_req[s]) cudaFree(c->st_req[s]);
    if (c->st_dst[s]) cudaFree(c->st_dst[s]);
    if (c->st_out[s]) cudaFree(c->st_out[s]);
  }
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->flags) cudaFree(c->flags);
  if (c->side) cudaStreamDestroy(c->side);
  if (c->ret) cudaStreamDestroy(c->ret);
  if (c->s_in) cudaStreamDestroy(c->s_in);
  if (c->s_out) cudaStreamDestroy(c->s_out);
  c->e->plain_launches = false;
  delete c;
}

int dint_shard_flags(dint_shard_ctx* c, uint32_t out[2]) {
  if (!c || !out) return DINT_EINVAL;
  CU(cudaSetDevice(c->e->device));
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(out, c->flags, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  CU(cudaMemset(c->flags, 0, 2 * sizeof(uint32_t)));
  return DINT_OK;
}

// After a slab overflow: *first_unserved = index, inside the LAST submit call (of k batches), of the first batch that
// no shard served (it and every later batch left the state untouched; their replies are garbage), or 0xffffffff when
// nothing was skipped.  Clears the condition and the engine's inter-chunk bookkeeping; call it on every rank before the
// next submit, then serve the unserved batches again in pieces of at most `cap` records per rank (which cannot overflow).
int dint_shard_recover(dint_shard_ctx* c, uint32_t k_last, uint32_t* first_unserved) {
  if (!c || !first_unserved) return DINT_EINVAL;
  dint_engine* e = c->e;
  CU(cudaSetDevice(e->device));
  CU(cudaDeviceSynchronize());
  uint32_t bad = 0;
  CU(cudaMemcpy(&bad, c->flags + 2, sizeof bad, cudaMemcpyDeviceToHost));
  *first_unserved = 0xffffffffu;
  if (!bad) return DINT_OK;
  const uint32_t first_epoch = c->epoch - k_last + 1;
  *first_unserved = bad >= first_epoch ? bad - first_epoch : 0;
  CU(cudaMemset(c->flags, 0, 4 * sizeof(uint32_t)));
  // the skipped launches changed nothing on the device, but the host-side chunk bookkeeping advanced: start clean
  e->ord_pending = false;
  e->prev_n = 0;
  CU(cudaMemset(e->d_nc, 0, 8 * sizeof(uint32_t)));
  CU(cudaMemset(e->d_flags[0], 0, (size_t)((char*)e->d_flags[1] - (char*)e->d_flags[0]) * 2));
  CU(cudaDeviceSynchronize());
  return DINT_OK;
}

int dint_shard_submit_many(dint_shard_ctx* c, uint32_t k, const void* const* req_dev, const uint8_t* const* dst_dev, uint64_t n,
                           void* const* out_dev, void* cuda_stream) {
  if (!c || !req_dev || !out_dev || n == 0 || n > c->max_n) return set_err(DINT_EINVAL, "bad argument");
  if (k == 0) return DINT_OK;
  std::vector<std::vector<ShardBatch>> b(1, std::vector<ShardBatch>(k));
  for (uint32_t j = 0; j < k; j++) b[0][j] = ShardBatch{req_dev[j], dst_dev ? dst_dev[j] : nullptr, out_dev[j], n};
  cudaStream_t main = (cudaStream_t)cuda_stream;
  return shard_run(&c, 1, k, b, &main);
}

}  // extern "C"

extern "C" {

int dint_shard_submit_many_v(dint_shard_ctx* c, uint32_t k, const void* const* req_dev, const uint8_t* const* dst_dev, const uint64_t* n,
                             const uint32_t* cap, void* const* out_dev, void* cuda_stream) {
  if (!c || !req_dev || !out_dev || !n) return set_err(DINT_EINVAL, "bad argument");
  if (k == 0) return DINT_OK;
  std::vector<std::vector<ShardBatch>> b(1, std::vector<ShardBatch>(k));
  for (uint32_t j = 0; j < k; j++) {
    const uint32_t cj = cap ? cap[j] : 0;
    if (n[j] > c->max_n || cj > c->cap || cj % kTile != 0) return set_err(DINT_EINVAL, "batch size / slab capacity (a multiple of 128, <= the capacity of dint_shard_create)");
    b[0][j] = ShardBatch{req_dev[j], dst_dev ? dst_dev[j] : nullptr, out_dev[j], n[j], cj};
  }
  cudaStream_t main = (cudaStream_t)cuda_stream;
  return shard_run(&c, 1, k, b, &main);
}

int dint_shard_submit_host(dint_shard_ctx* c, uint32_t k, const void* const* req_host, const uint8_t* const* dst_host, uint64_t n,
                           void* const* out_host) {
  if (!c || !req_host || !out_host || n == 0 || n > c->max_n) return set_err(DINT_EINVAL, "bad argument");
  std::vector<std::vector<HostBatch>> hb(1, std::vector<HostBatch>(k));
  for (uint32_t j = 0; j < k; j++) hb[0][j] = HostBatch{(const uint8_t*)req_host[j], dst_host ? dst_host[j] : nullptr, (uint8_t*)out_host[j], n};
  return shard_run_host(&c, 1, k, hb);
}

// ---- dint_cluster_*: G shards driven by ONE process (SURVEY.md 8(b): dint_create(kind, cfg, n_gpus) / dint_submit(..., dst_shard, ...)) ----
struct dint_cluster {
  int kind = 0;
  uint32_t G = 0, cap = 0;
  uint64_t max_n = 0;
  bool by_dst = false, shared_device = false;
  std::vector<int> dev;
  std::vector<dint_engine*> eng;
  std::vector<dint_shard_ctx*> sh;
  std::vector<void*> bufs;                  // per rank: one allocation {inbox sets | return-buffer sets | signal block}
  uint64_t overflow_retries = 0;            // submit calls that met a slab overflow and served the rest in small rounds
};

void dint_cluster_destroy(dint_cluster* cl) {
  if (!cl) return;
  for (auto* c : cl->sh) dint_shard_destroy(c);
  for (size_t r = 0; r < cl->bufs.size(); r++) { cudaSetDevice(cl->dev[r]); cudaFree(cl->bufs[r]); }
  for (auto* e : cl->eng) dint_destroy(e);
  delete cl;
}

int dint_cluster_create(int kind, const dint_cfg* cfg, int n_gpus, const int* devices, uint64_t max_batch, dint_cluster** out) {
  if (!out || kind < 0 || kind >= DINT_NUM_KINDS || n_gpus < 1 || n_gpus > kMaxShards) return set_err(DINT_EINVAL, "bad kind / n_gpus");
  *out = nullptr;
  const bool by_dst = kind == DINT_TATP || kind == DINT_SMALLBANK;
  if (by_dst && n_gpus == 2) return set_err(DINT_EINVAL, "tatp / smallbank placement needs 1 or >= 3 shards (primary + 2 backups)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return set_err(DINT_ENODEV, "no CUDA device: dint_b200 has no CPU fallback"); }
  dint_cluster* cl = new dint_cluster();
  cl->kind = kind; cl->G = (uint32_t)n_gpus; cl->by_dst = by_dst;
  for (int r = 0; r < n_gpus; r++) {
    const int d = devices ? devices[r] : r % ndev;
    if (d < 0 || d >= ndev) { delete cl; return set_err(DINT_EINVAL, "bad device ordinal"); }
    cl->dev.push_back(d);
    for (int q = 0; q < r; q++) if (cl->dev[q] == d) cl->shared_device = true;
  }
  if (cl->shared_device)
    for (int r = 1; r < n_gpus; r++)
      if (cl->dev[r] != cl->dev[0]) { delete cl; return set_err(DINT_EINVAL, "devices must be all distinct or all the same"); }
  const uint32_t G = cl->G;
  const uint32_t msg = kMsgSize[kind];
  if (max_batch == 0) max_batch = 1u << 18;
  cl->max_n = max_batch;
  {
    // slab capacity per (source, owner): hashing spreads records evenly (mean + 25 % + 8 sigma); a client-chosen
    // placement is pre-counted on the host by dint_cluster_submit, which cuts a round where a slab would overflow
    const double mean = (double)max_batch / G;
    uint64_t cap = (uint64_t)(mean * (by_dst ? 2.0 : 1.25) + 8.0 * sqrt(mean) + 64);
    if (G == 1) cap = max_batch;
    cl->cap = (uint32_t)((cap + kTile - 1) / kTile * kTile);
  }
  int rc = DINT_OK;
  dint_cfg base;
  if (cfg) base = *cfg; else dint_default_cfg(kind, &base);
  const uint32_t chunk_need = (uint32_t)(((uint64_t)G * cl->cap + kTile - 1) / kTile * kTile);
  for (uint32_t r = 0; r < G && rc == DINT_OK; r++) {
    dint_cfg c = base;
    if (by_dst) { c.n_shards = 1; c.shard_id = 0; c.txn_shards = G; c.txn_shard_id = r; }
    else { c.n_shards = G; c.shard_id = r; }
    if (c.chunk == 0 || c.chunk < chunk_need) c.chunk = chunk_need;        // one batch of the exchange = one engine chunk
    dint_engine* e = nullptr;
    rc = dint_create(kind, &c, cl->dev[r], &e);
    if (rc == DINT_OK) cl->eng.push_back(e);
  }
  const uint32_t S = 3;
  const size_t region = ((size_t)G * cl->cap * msg + 255) / 256 * 256;
  std::vector<uint64_t> base_ptr(G);
  for (uint32_t r = 0; r < G && rc == DINT_OK; r++) {
    void* p = nullptr;
    if (cudaSetDevice(cl->dev[r]) != cudaSuccess || cudaMalloc(&p, 2 * S * region + 4096) != cudaSuccess) { rc = set_err(DINT_ENOMEM, "cluster buffers", cudaGetLastError()); break; }
    cudaMemset(p, 0, 2 * S * region + 4096);
    cl->bufs.push_back(p);
    base_ptr[r] = (uint64_t)p;
    if (!cl->shared_device)
      for (uint32_t q = 0; q < G; q++)
        if (q != r) {
          int can = 0;
          cudaDeviceCanAccessPeer(&can, cl->dev[r], cl->dev[q]);
          if (!can) { rc = set_err(DINT_ENODEV, "GPUs without peer access"); break; }
          cudaError_t ce = cudaDeviceEnablePeerAccess(cl->dev[q], 0);
          if (ce != cudaSuccess && ce != cudaErrorPeerAccessAlreadyEnabled) { rc = set_err(DINT_EIO, "cudaDeviceEnablePeerAccess", ce); break; }
          cudaGetLastError();
        }
  }
  for (uint32_t r = 0; r < G && rc == DINT_OK; r++) {
    cudaSetDevice(cl->dev[r]);
    cudaDeviceSynchronize();
  }
  for (uint32_t r = 0; r < G && rc == DINT_OK; r++) {
    dint_peer_ptrs in[kMaxSets]{}, rb[kMaxSets]{}, sig{};
    for (uint32_t s = 0; s < S; s++)
      for (uint32_t o = 0; o < G; o++) { in[s].p[o] = base_ptr[o] + (2 * s) * region; rb[s].p[o] = base_ptr[o] + (2 * s + 1) * region; }
    for (uint32_t o = 0; o < G; o++) sig.p[o] = base_ptr[o] + 2 * S * region;
    dint_shard_ctx* c = nullptr;
    rc = shard_make(cl->eng[r], G, r, cl->cap, S, in, rb, &sig, cl->max_n, cl->shared_device, &c);
    if (rc == DINT_OK) cl->sh.push_back(c);
  }
  if (rc != DINT_OK) { std::string keep = g_last_error; dint_cluster_destroy(cl); g_last_error = keep; return rc; }
  *out = cl;
  return DINT_OK;
}

int dint_cluster_populate(dint_cluster* cl) {
  if (!cl) return DINT_EINVAL;
  for (auto* e : cl->eng) { int rc = dint_populate(e); if (rc) return rc; }
  return DINT_OK;
}
dint_engine* dint_cluster_engine(dint_cluster* cl, int shard) { return (cl && shard >= 0 && shard < (int)cl->G) ? cl->eng[shard] : nullptr; }
uint32_t dint_cluster_size(dint_cluster* cl) { return cl ? cl->G : 0; }

// rounds over [from, to): a round hands rank r the r-th of G contiguous pieces of at most `lim` records (rank-major
// order = index order, SURVEY.md 8(e)); for a client-chosen placement the pieces are cut so that no slab can overflow.
// Returns the first record index that was NOT served (to = everything served), or a negative error.
static int64_t cluster_run(dint_cluster* cl, const uint8_t* rq, const uint8_t* dst_shard, uint8_t* rs, uint64_t from, uint64_t to, uint64_t lim) {
  const uint32_t G = cl->G, msg = kMsgSize[cl->kind];
  std::vector<std::vector<HostBatch>> hb(G);
  std::vector<uint64_t> round_off;
  uint64_t off = from;
  while (off < to) {
    uint64_t m = to - off < (uint64_t)G * lim ? to - off : (uint64_t)G * lim;
    for (;;) {
      const uint64_t q = (m + G - 1) / G;
      bool fits = true;
      if (dst_shard && G > 1) {
        for (uint32_t r = 0; r < G && fits; r++) {
          const uint64_t lo = off + (uint64_t)r * q, hi = lo + q < off + m ? lo + q : off + m;
          uint32_t cnt[kMaxShards] = {0};
          for (uint64_t i = lo; i < hi; i++) { const uint8_t o = dst_shard[i]; if (o < G) cnt[o]++; }
          for (uint32_t o = 0; o < G; o++) if (cnt[o] > cl->cap) fits = false;
        }
      }
      if (fits || m <= G) break;
      m = (m + 1) / 2;
    }
    const uint64_t q = (m + G - 1) / G;
    round_off.push_back(off);
    for (uint32_t r = 0; r < G; r++) {
      const uint64_t lo = off + (uint64_t)r * q;
      const uint64_t hi = lo + q < off + m ? lo + q : off + m;
      // (a rank without records in a tail round still takes part in the exchange: its slabs are all padding)
      hb[r].push_back(HostBatch{rq + lo * msg, dst_shard ? dst_shard + lo : nullptr, rs + lo * msg, lo < hi ? hi - lo : 0});
    }
    off += m;
  }
  const uint32_t k = (uint32_t)round_off.size();
  int rc = shard_run_host(cl->sh.data(), G, k, hb);
  if (rc) return rc;
  uint32_t first_unserved = 0xffffffffu;
  for (uint32_t r = 0; r < G; r++) {
    uint32_t fl[2] = {0, 0}, fu = 0xffffffffu;
    if ((rc = dint_shard_flags(cl->sh[r], fl))) return rc;
    if (fl[1]) return set_err(DINT_EIO, "exchange timed out");
    if ((rc = dint_shard_recover(cl->sh[r], k, &fu))) return rc;
    if (fu < first_unserved) first_unserved = fu;
  }
  return first_unserved == 0xffffffffu ? (int64_t)to : (int64_t)round_off[first_unserved];
}

int dint_cluster_submit(dint_cluster* cl, const void* req, uint64_t n, const uint8_t* dst_shard, void* resp) {
  if (!cl || (n && (!req || !resp))) return set_err(DINT_EINVAL, "null argument");
  if (cl->by_dst && cl->G > 1 && !dst_shard) return set_err(DINT_EINVAL, "tatp / smallbank: the client names the shard of every record (dst_shard)");
  if (n == 0) return DINT_OK;
  unsigned long long err_before = 0;
  for (auto* e : cl->eng) err_before += e->stats.errors;
  // Normal rounds; if a slab overflowed (keys skewed beyond the slack of the slabs) every shard stopped serving AT that
  // round, nothing behind it touched the state: serve the rest in rounds of at most `cap` records per rank, which fit
  // any slab whatever the keys are.
  int64_t done = cluster_run(cl, (const uint8_t*)req, dst_shard, (uint8_t*)resp, 0, n, cl->max_n);
  if (done < 0) return (int)done;
  if ((uint64_t)done < n) {
    cl->overflow_retries++;
    done = cluster_run(cl, (const uint8_t*)req, dst_shard, (uint8_t*)resp, (uint64_t)done, n, cl->cap < cl->max_n ? cl->cap : cl->max_n);
    if (done < 0) return (int)done;
    if ((uint64_t)done < n) return set_err(DINT_EIO, "internal: a round of at most cap records per rank overflowed");
  }
  unsigned long long err_after = 0;
  for (uint32_t r = 0; r < cl->G; r++) {
    dint_engine* e = cl->eng[r];
    int rc = pull_counters(e);
    if (rc) return rc;
    err_after += e->stats.errors;
  }
  return err_after != err_before ? DINT_EPROTO : DINT_OK;
}
uint64_t dint_cluster_overflow_retries(dint_cluster* cl) { return cl ? cl->overflow_retries : 0; }

}  // extern "C"

extern "C" {
// ---- lock_fasst closed-loop clients on the GPU (clients.cuh) ------------------------------------------------
struct dint_clients {
  dint_engine* e = nullptr;
  ClientCtx cc{};
  uint8_t *req = nullptr, *resp = nullptr;
  double* cdf = nullptr;
  uint64_t seed = 0;
  bool started = false;
};

void dint_clients_destroy(dint_clients* c) {
  if (!c) return;
  cudaSetDevice(c->e->device);
  cudaDeviceSynchronize();
  cudaFree(c->req); cudaFree(c->resp); cudaFree(c->cdf);
  cudaFree(c->cc.hdr); cudaFree(c->cc.rng); cudaFree(c->cc.rk); cudaFree(c->cc.rv); cudaFree(c->cc.stats);
  delete c;
}

int dint_clients_create(dint_engine* e, uint32_t n_clients, uint64_t seed, uint32_t n_keys, double zipf_theta, uint32_t read_pct,
                        dint_clients** out) {
  if (!e || !out || e->kind != DINT_FASST || n_clients == 0 || n_keys == 0) return set_err(DINT_EINVAL, "lock_fasst engine, n_clients > 0, n_keys > 0");
  CU(cudaSetDevice(e->device));
  dint_clients* c = new dint_clients();
  c->e = e;
  c->seed = seed;
  ClientCtx& cc = c->cc;
  cc.n_clients = n_clients; cc.n_keys = n_keys; cc.read_pct = read_pct;
  const size_t n = n_clients;
  if (cudaMalloc(&c->req, n * 9 + 16) != cudaSuccess || cudaMalloc(&c->resp, n * 9 + 16) != cudaSuccess ||
      cudaMalloc(&cc.hdr, n * 8) != cudaSuccess || cudaMalloc(&cc.rng, n * 8) != cudaSuccess || cudaMalloc(&cc.rk, n * 40) != cudaSuccess ||
      cudaMalloc(&cc.rv, n * 40) != cudaSuccess || cudaMalloc(&cc.stats, 8 * sizeof(unsigned long long)) != cudaSuccess) {
    cudaError_t ce = cudaGetLastError();
    dint_clients_destroy(c);
    return set_err(DINT_ENOMEM, "client state", ce);
  }
  CU(cudaMemset(cc.stats, 0, 8 * sizeof(unsigned long long)));
  CU(cudaMemset(cc.rv, 0, n * 40));
  if (zipf_theta > 0) {                                  // workloads.cc Zipf::init
    std::vector<double> cdf(n_keys);
    double acc = 0;
    for (uint32_t k = 0; k < n_keys; k++) { acc += 1.0 / std::pow((double)(k + 1), zipf_theta); cdf[k] = acc; }
    for (auto& v : cdf) v /= acc;
    CU(cudaMalloc(&c->cdf, (size_t)n_keys * sizeof(double)));
    CU(cudaMemcpy(c->cdf, cdf.data(), (size_t)n_keys * sizeof(double), cudaMemcpyHostToDevice));
    cc.cdf = c->cdf;
    cc.zipf_n = n_keys;
  }
  *out = c;
  return DINT_OK;
}

// `rounds` closed-loop rounds, asynchronous on cuda_stream: every round = the engine on the clients' request buffer
// (dint_submit_device) + ONE kernel that absorbs the replies and emits the next round's requests
int dint_clients_run(dint_clients* c, uint32_t rounds, void* cuda_stream) {
  if (!c) return set_err(DINT_EINVAL, "null argument");
  dint_engine* e = c->e;
  CU(cudaSetDevice(e->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const uint32_t blocks = (c->cc.n_clients + 255) / 256;
  if (!c->started) {
    k_clients_init<<<blocks, 256, 0, s>>>(c->cc, c->seed, c->req);
    c->started = true;
    e->stats.kernel_launches++;
  }
  for (uint32_t r = 0; r < rounds; r++) {
    int rc = run_device(e, c->req, c->cc.n_clients, c->resp, s);
    if (rc) return rc;
    k_clients_step<<<blocks, 256, 0, s>>>(c->cc, c->resp, c->req);
    e->stats.kernel_launches++;
  }
  CU(cudaGetLastError());
  return DINT_OK;
}

// out: requests served, committed transactions, validation aborts, lock rejects, rounds (synchronises)
int dint_clients_stats(dint_clients* c, uint64_t out[5]) {
  if (!c || !out) return set_err(DINT_EINVAL, "null argument");
  CU(cudaSetDevice(c->e->device));
  CU(cudaDeviceSynchronize());
  unsigned long long h[5];
  CU(cudaMemcpy(h, c->cc.stats, sizeof h, cudaMemcpyDeviceToHost));
  for (int i = 0; i < 5; i++) out[i] = h[i];
  return DINT_OK;
}

// test hook: the requests the clients will send next and the replies they absorbed last (host buffers of n_clients * 9 bytes)
int dint_clients_peek(dint_clients* c, void* next_req_host, void* last_resp_host) {
  if (!c) return set_err(DINT_EINVAL, "null argument");
  CU(cudaSetDevice(c->e->device));
  CU(cudaDeviceSynchronize());
  if (!c->started) {
    k_clients_init<<<(c->cc.n_clients + 255) / 256, 256>>>(c->cc, c->seed, c->req);
    c->started = true;
    CU(cudaDeviceSynchronize());
  }
  if (next_req_host) CU(cudaMemcpy(next_req_host, c->req, (size_t)c->cc.n_clients * 9, cudaMemcpyDeviceToHost));
  if (last_resp_host) CU(cudaMemcpy(last_resp_host, c->resp, (size_t)c->cc.n_clients * 9, cudaMemcpyDeviceToHost));
  return DINT_OK;
}

}  // extern "C"

extern "C" {
// ---- TATP / SmallBank closed-loop clients on the GPU (txn_clients.cuh) -------------------------------------------------
struct dint_txn_clients {
  std::vector<dint_engine*> eng;
  int kind = 0, device = 0;
  uint32_t G = 0, msz = 0;
  TxnDevCtx x{};
  int p = 0;                          // parity of the round whose requests are pending
  uint32_t* h_tot = nullptr;          // pinned copy of x.tot
  uint32_t tot[8] = {0}, tot_prev[8] = {0};
  bool served = false;                // a round has been served: last replies exist
  uint64_t st_requests = 0, st_rounds = 0;
  cudaEvent_t ev = nullptr;
  std::vector<void*> allocs;
};

void dint_txn_clients_destroy(dint_txn_clients* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (void* q : c->allocs) cudaFree(q);
  if (c->h_tot) cudaFreeHost(c->h_tot);
  if (c->ev) cudaEventDestroy(c->ev);
  delete c;
}

// k_txn_step (absorb or begin, then count) + k_txn_scan + k_txn_emit for parity p, then the per-shard totals to the host
static int txn_clients_round(dint_txn_clients* c, int init, cudaStream_t s) {
  const TxnDevCtx& x = c->x;
  if (c->kind == DINT_TATP) k_txn_step<DINT_TATP><<<x.nb, kTxnThreads, 0, s>>>(x, init, c->p);
  else k_txn_step<DINT_SMALLBANK><<<x.nb, kTxnThreads, 0, s>>>(x, init, c->p);
  k_txn_scan<<<c->G, kTxnScanThreads, 0, s>>>(x, c->p);
  if (c->kind == DINT_TATP) k_txn_emit<DINT_TATP><<<x.nb, kTxnThreads, 0, s>>>(x, c->p);
  else k_txn_emit<DINT_SMALLBANK><<<x.nb, kTxnThreads, 0, s>>>(x, c->p);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(c->h_tot, x.tot, 9 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  CU(cudaEventRecord(c->ev, s));
  CU(cudaEventSynchronize(c->ev));
  if (c->h_tot[8]) return set_err(DINT_EIO, "a client sent one shard more records in one round than the buffers are sized for");
  memcpy(c->tot_prev, c->tot, sizeof c->tot);
  for (uint32_t s_ = 0; s_ < c->G; s_++) c->tot[s_] = c->h_tot[s_];
  return DINT_OK;
}

int dint_txn_clients_create(dint_engine* const* shards, uint32_t n_shards, uint32_t n_clients, uint32_t gid0, uint32_t subscribers,
                            dint_txn_clients** out) {
  if (!shards || !out) return set_err(DINT_EINVAL, "null argument");
  *out = nullptr;
  if (n_shards == 0 || n_shards == 2 || n_shards > 8) return set_err(DINT_EINVAL, "n_shards must be 1 or 3..8 (primary + 2 distinct backups)");
  if (n_clients == 0 || n_clients > (1u << 26)) return set_err(DINT_EINVAL, "n_clients must be 1..2^26");
  if (subscribers < 3) return set_err(DINT_EINVAL, "subscribers / accounts must be >= 3");
  for (uint32_t i = 0; i < n_shards; i++) {
    const dint_engine* e = shards[i];
    if (!e) return set_err(DINT_EINVAL, "null engine");
    if ((e->kind != DINT_TATP && e->kind != DINT_SMALLBANK) || e->kind != shards[0]->kind)
      return set_err(DINT_EINVAL, "the engines must all be tatp or all smallbank");
    if (e->device != shards[0]->device) return set_err(DINT_EINVAL, "the engines must all be on one device");
    if (n_shards > 3 && (e->cfg.txn_shards != n_shards || e->cfg.txn_shard_id != i))
      return set_err(DINT_EINVAL, "with more than 3 shards, engine i must be configured as shard i of n_shards (txn_shards / txn_shard_id)");
  }
  dint_txn_clients* c = new dint_txn_clients();
  c->eng.assign(shards, shards + n_shards);
  c->kind = shards[0]->kind; c->device = shards[0]->device; c->G = n_shards; c->msz = kMsgSize[c->kind];
  TxnDevCtx& x = c->x;
  x.P.G = n_shards; x.P.subscribers = subscribers; x.P.accounts = subscribers; x.P.hot = txn::sb_hot_accounts(subscribers);
  x.n_clients = n_clients; x.nb = (n_clients + kTxnThreads - 1) / kTxnThreads; x.gid0 = gid0;
  x.bound = txn::max_per_shard(c->kind, n_shards);
  const size_t n = n_clients, G = n_shards;
  int rc = DINT_OK;
  auto alloc = [&](void** q, size_t bytes) {
    if (rc) return;
    cudaError_t ce = cudaMalloc(q, bytes);           // 256-byte aligned: the engines need 16
    if (ce != cudaSuccess) { *q = nullptr; rc = set_err(DINT_ENOMEM, "client state", ce); return; }
    c->allocs.push_back(*q);
  };
  if (cudaSetDevice(c->device) != cudaSuccess) { delete c; return set_err(DINT_EIO, "cudaSetDevice", cudaGetLastError()); }
  alloc(&x.cl, n * (c->kind == DINT_TATP ? sizeof(txn::TatpClient) : sizeof(txn::SbClient)));
  for (uint32_t s = 0; s < n_shards; s++) {
    alloc((void**)&x.req[s], n * x.bound * c->msz + 16);
    alloc((void**)&x.resp[s], n * x.bound * c->msz + 16);
  }
  for (int q = 0; q < 2; q++) {
    alloc((void**)&x.loff[q], G * n * 4);
    alloc((void**)&x.base[q], G * x.nb * 4);
    alloc((void**)&x.route[q], n * 4);
  }
  alloc((void**)&x.ctatot, G * x.nb * 4);
  alloc((void**)&x.tot, 16 * 4);
  alloc((void**)&x.stats, 18 * sizeof(unsigned long long));
  if (!rc && cudaMallocHost((void**)&c->h_tot, 16 * 4) != cudaSuccess) rc = set_err(DINT_ENOMEM, "pinned totals", cudaGetLastError());
  if (!rc && cudaEventCreateWithFlags(&c->ev, cudaEventDisableTiming) != cudaSuccess) rc = set_err(DINT_EIO, "event", cudaGetLastError());
  if (!rc && (cudaMemset(x.tot, 0, 16 * 4) != cudaSuccess || cudaMemset(x.stats, 0, 18 * sizeof(unsigned long long)) != cudaSuccess))
    rc = set_err(DINT_EIO, "cudaMemset", cudaGetLastError());
  // every client begins its first transaction; the first round's records go to the shard buffers
  if (!rc) rc = txn_clients_round(c, 1, nullptr);
  if (rc) { dint_txn_clients_destroy(c); return rc; }
  *out = c;
  return DINT_OK;
}

// `rounds` rounds on cuda_stream: serve the pending records with the shard engines, then absorb + count, scan, emit.
// Returns after the last round's totals reached the host (each round synchronises once on them).
int dint_txn_clients_run(dint_txn_clients* c, uint32_t rounds, void* cuda_stream) {
  if (!c) return set_err(DINT_EINVAL, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  for (uint32_t r = 0; r < rounds; r++) {
    for (uint32_t i = 0; i < c->G; i++) {
      if (!c->tot[i]) continue;                            // as Cluster.submit: an empty shard is not called
      int rc = run_device(c->eng[i], c->x.req[i], c->tot[i], c->x.resp[i], s);
      if (rc) return rc;
      c->st_requests += c->tot[i];
    }
    c->st_rounds++;
    c->served = true;
    c->p ^= 1;
    int rc = txn_clients_round(c, 0, s);
    if (rc) return rc;
  }
  return DINT_OK;
}

// out: requests served, transactions begun, committed, rounds, begun by type[7], committed by type[7] (synchronises)
int dint_txn_clients_stats(dint_txn_clients* c, uint64_t out[18]) {
  if (!c || !out) return set_err(DINT_EINVAL, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaDeviceSynchronize());
  unsigned long long h[18];
  CU(cudaMemcpy(h, c->x.stats, sizeof h, cudaMemcpyDeviceToHost));
  for (int i = 0; i < 18; i++) out[i] = h[i];
  out[0] = c->st_requests;
  out[3] = c->st_rounds;
  return DINT_OK;
}

// rebuild one round in client order (each client's records contiguous, in push order) from the shard buffers
static int txn_clients_gather(dint_txn_clients* c, int p, uint8_t* const* bufs, const uint32_t* tot, uint8_t* out, uint8_t* dst) {
  const size_t n = c->x.n_clients, G = c->G, nb = c->x.nb, msz = c->msz;
  std::vector<uint32_t> route(n), loff(G * n), base(G * nb);
  std::vector<std::vector<uint8_t>> recs(G);
  CU(cudaMemcpy(route.data(), c->x.route[p], n * 4, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(loff.data(), c->x.loff[p], G * n * 4, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(base.data(), c->x.base[p], G * nb * 4, cudaMemcpyDeviceToHost));
  for (size_t s = 0; s < G; s++) {
    recs[s].resize((size_t)tot[s] * msz);
    if (tot[s]) CU(cudaMemcpy(recs[s].data(), bufs[s], (size_t)tot[s] * msz, cudaMemcpyDeviceToHost));
  }
  size_t j = 0;
  for (size_t cl = 0; cl < n; cl++) {
    const uint32_t r = route[cl];
    uint32_t k[8] = {0};
    for (uint32_t i = 0; i < (r & 15u); i++, j++) {
      const uint32_t s = (r >> (4 + 3 * i)) & 7u;
      const size_t slot = (size_t)base[s * nb + cl / kTxnThreads] + loff[s * n + cl] + k[s]++;
      if (slot >= tot[s]) return set_err(DINT_EIO, "peek: inconsistent offsets");
      if (out) memcpy(out + j * msz, recs[s].data() + slot * msz, msz);
      if (dst) dst[j] = (uint8_t)s;
    }
  }
  return DINT_OK;
}

// test hook: the pending round's requests + destination shards and the last round's replies, in client order, as
// dint_txn_next / dint_txn_feed lay them out.  n_out = {records pending, replies of the last round}; pass NULL buffers to
// learn the sizes first.
int dint_txn_clients_peek(dint_txn_clients* c, void* next_req_host, uint8_t* next_dst_host, void* last_resp_host, uint64_t n_out[2]) {
  if (!c) return set_err(DINT_EINVAL, "null argument");
  CU(cudaSetDevice(c->device));
  CU(cudaDeviceSynchronize());
  uint64_t a = 0, b = 0;
  for (uint32_t s = 0; s < c->G; s++) { a += c->tot[s]; b += c->served ? c->tot_prev[s] : 0; }
  if (n_out) { n_out[0] = a; n_out[1] = b; }
  if (next_req_host || next_dst_host) {
    int rc = txn_clients_gather(c, c->p, c->x.req, c->tot, (uint8_t*)next_req_host, next_dst_host);
    if (rc) return rc;
  }
  if (last_resp_host && c->served) {
    int rc = txn_clients_gather(c, c->p ^ 1, c->x.resp, c->tot_prev, (uint8_t*)last_resp_host, nullptr);
    if (rc) return rc;
  }
  return DINT_OK;
}

}  // extern "C"
