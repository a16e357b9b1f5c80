// txn_clients.cuh -- the TATP and SmallBank closed-loop clients ON the GPU (SURVEY.md section 8(f) rank 2): the device
// driver around the state machines of txn_clients.h (the host driver is txn_workloads.cc).  One thread per client; the
// client structs live in device memory.  One round, on one stream:
//   k_txn_step   find the client's replies of the last round (tatp_emit / sb_emit run again with a LOCATE sink over
//                the offsets saved then), absorb them -- which may finish the transaction and begin the next, with the
//                client's own fastrand stream -- then COUNT the next step's records per shard and scan the counts
//                inside the CTA.  Stats: warp-aggregated atomics.
//   k_txn_scan   one CTA per shard scans the CTA totals: CTA bases and the shard's total.
//   k_txn_emit   emit once more with a WRITE sink: every record goes to req[s] + off[s][c] + (its index among the
//                client's records for s), ord set as the host sets it.  Shard s therefore receives exactly the host
//                round's partition_by_shard: client order, then push order within a client.
// The host then reads the G totals (one sync per round: the engines' chunk loops are sized on the host) and serves
// shard s's totals[s] records with its engine.
//
// Offsets are kept for two rounds (parity `cur`): the LOCATE pass of round r+1 reads round r's, and the test hook
// dint_txn_clients_peek rebuilds the last round's replies in client order from them.  route[p][c] records, for the
// round of parity p, the client's record count (bits 0-3) and the shard of its i-th record (bits 4+3i..6+3i).
#pragma once
#include "common.cuh"
#include "txn_clients.h"

namespace dint {

constexpr uint32_t kTxnThreads = 256;
constexpr uint32_t kTxnScanThreads = 1024;

struct TxnDevCtx {
  txn::Params P;
  uint32_t n_clients, nb, bound;     // nb = CTAs of k_txn_step; bound = txn::max_per_shard
  void* cl;                          // TatpClient[n_clients] or SbClient[n_clients]
  uint64_t gid0;
  uint8_t* req[8];                   // per shard: this round's requests
  uint8_t* resp[8];                  // per shard: the replies to them
  uint32_t* loff[2];                 // [parity][G][n_clients]  exclusive offset of a client's records inside its CTA
  uint32_t* base[2];                 // [parity][G][nb]         exclusive offset of a CTA inside the shard
  uint32_t* ctatot;                  // [G][nb]                 records of a CTA
  uint32_t* route[2];                // [parity][n_clients]
  uint32_t* tot;                     // [0..G) records per shard this round; [8] = a client exceeded `bound`
  unsigned long long* stats;         // dint_txn_stats layout: [1] txns [2] committed [4+t] begun [11+t] committed by type
};

#ifdef __CUDACC__
template <int KIND> struct TxnKind;
template <> struct TxnKind<4> {
  using Client = txn::TatpClient;
  static constexpr int MSZ = txn::TM;
  DINT_D static void begin(const txn::Params& P, Client& c) { txn::tatp_begin(P, c); }
  template <class S> DINT_D static uint32_t emit(const txn::Params& P, const Client& c, S& s) { return txn::tatp_emit(P, c, s); }
  template <class R> DINT_D static int absorb(const txn::Params& P, Client& c, const R& r) { return txn::tatp_absorb(P, c, r); }
};
template <> struct TxnKind<5> {
  using Client = txn::SbClient;
  static constexpr int MSZ = txn::SMSZ;
  DINT_D static void begin(const txn::Params& P, Client& c) { txn::sb_begin(P, c); }
  template <class S> DINT_D static uint32_t emit(const txn::Params& P, const Client& c, S& s) { return txn::sb_emit(P, c, s); }
  template <class R> DINT_D static int absorb(const txn::Params& P, Client& c, const R& r) { return txn::sb_absorb(P, c, r); }
};

// record index of client c's k-th record for shard s, for the round of parity p
DINT_D uint32_t txn_slot(const TxnDevCtx& x, int p, uint32_t s, uint32_t c, uint32_t k) {
  return x.base[p][(size_t)s * x.nb + c / kTxnThreads] + x.loff[p][(size_t)s * x.n_clients + c] + k;
}

// counts per shard, 8 bits each (a client sends a shard at most 9 records a round), and the route word
struct TxnCountSink {
  unsigned long long cnt = 0;
  uint32_t route = 0, n = 0;
  DINT_D void push(const uint8_t*, uint32_t shard, int) {
    cnt += 1ull << (8 * shard);
    route |= shard << (4 + 3 * n);
    n++;
  }
};
// where the replies to a client's records are
template <int MSZ>
struct TxnLocateSink {
  const TxnDevCtx& x;
  int p;
  uint32_t c;
  unsigned long long k = 0;
  uint32_t n = 0;
  const uint8_t* at[9];
  DINT_D TxnLocateSink(const TxnDevCtx& x_, int p_, uint32_t c_) : x(x_), p(p_), c(c_) {}
  DINT_D void push(const uint8_t*, uint32_t shard, int) {
    const uint32_t ks = (uint32_t)(k >> (8 * shard)) & 255u;
    k += 1ull << (8 * shard);
    at[n < 9 ? n : 8] = x.resp[shard] + (size_t)txn_slot(x, p, shard, c, ks) * MSZ;
    n++;
  }
  DINT_D const uint8_t* rec(int i) const { return at[i]; }
};
// the records themselves, at their slots in the shard buffers
template <int MSZ>
struct TxnWriteSink {
  const TxnDevCtx& x;
  int p;
  uint32_t c;
  unsigned long long k = 0;
  DINT_D TxnWriteSink(const TxnDevCtx& x_, int p_, uint32_t c_) : x(x_), p(p_), c(c_) {}
  DINT_D void push(const uint8_t* rec, uint32_t shard, int ord) {
    const uint32_t ks = (uint32_t)(k >> (8 * shard)) & 255u;
    k += 1ull << (8 * shard);
    if (ks >= x.bound) return;                       // k_txn_step has flagged the round; never write past the slot
    uint8_t* d = x.req[shard] + (size_t)txn_slot(x, p, shard, c, ks) * MSZ;
#pragma unroll
    for (int i = 0; i < MSZ; i++) d[i] = rec[i];
    if (ord >= 0) d[0] = (uint8_t)ord;
  }
};

// block-wide exclusive scan of one value per thread; returns the thread's offset, *total = the block's sum
DINT_D uint32_t txn_block_scan(uint32_t v, uint32_t* s_warp, uint32_t* total) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= (uint32_t)d) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  uint32_t before = 0, all = 0;
  for (uint32_t w = 0; w < blockDim.x / 32; w++) {
    const uint32_t t = s_warp[w];
    before += w < warp ? t : 0u;
    all += t;
  }
  __syncthreads();                                   // s_warp is reused by the next call
  *total = all;
  return before + inc - v;
}

// init = 1: every client begins its first transaction (counted in txns, as dint_txn_create counts it);
// otherwise absorb the replies of round parity p_prev.  Then count the next round's records into parity p.
// (__maxnreg__: left to itself ptxas gives the TATP instance 64 registers and spills 20 bytes)
template <int KIND>
__global__ void __maxnreg__(96) k_txn_step(const TxnDevCtx x, int init, int p) {
  using K = TxnKind<KIND>;
  __shared__ uint32_t s_warp[kTxnThreads / 32];
  const uint32_t c = blockIdx.x * kTxnThreads + threadIdx.x;
  int began = -1, committed = -1;
  unsigned long long cnt = 0;
  uint32_t route = 0;
  if (c < x.n_clients) {
    typename K::Client& cl = ((typename K::Client*)x.cl)[c];
    if (init) {
      cl = typename K::Client{};
      cl.seed = 0xdeadbeefULL + x.gid0 + c;                  // client_udp_shard.cc:1121
      K::begin(x.P, cl);
      began = cl.txn;
    } else {
      TxnLocateSink<K::MSZ> loc(x, p ^ 1, c);
      K::emit(x.P, cl, loc);
      const int ev = K::absorb(x.P, cl, loc);
      if (ev >= 0) {
        began = cl.txn;
        if (ev & 1) committed = ev >> 1;
      }
    }
    TxnCountSink cs;
    K::emit(x.P, cl, cs);
    cnt = cs.cnt;
    route = cs.route | cs.n;
    x.route[p][c] = route;
  }
  bool over = false;
  for (uint32_t s = 0; s < x.P.G; s++) {
    uint32_t v = (uint32_t)(cnt >> (8 * s)) & 255u;
    if (v > x.bound) { over = true; v = x.bound; }
    uint32_t total;
    const uint32_t off = txn_block_scan(v, s_warp, &total);
    if (c < x.n_clients) x.loff[p][(size_t)s * x.n_clients + c] = off;
    if (threadIdx.x == 0) x.ctatot[(size_t)s * x.nb + blockIdx.x] = total;
  }
  if (over) atomicOr(&x.tot[8], 1u);
  // stats: one atomic per warp and counter
  const uint32_t all = 0xffffffffu;
  const uint32_t nb = __popc(__ballot_sync(all, began >= 0)), nc = __popc(__ballot_sync(all, committed >= 0));
  const bool lead = (threadIdx.x & 31) == 0;
  if (lead && nb) atomicAdd(&x.stats[1], (unsigned long long)nb);
  if (lead && nc) atomicAdd(&x.stats[2], (unsigned long long)nc);
  for (int t = 0; t < 7; t++) {
    const uint32_t b = __popc(__ballot_sync(all, began == t)), m = __popc(__ballot_sync(all, committed == t));
    if (lead && b) atomicAdd(&x.stats[4 + t], (unsigned long long)b);
    if (lead && m) atomicAdd(&x.stats[11 + t], (unsigned long long)m);
  }
}

// one CTA per shard: exclusive scan of the CTA totals -> base[p][s][*], tot[s]
__global__ void __launch_bounds__(kTxnScanThreads) k_txn_scan(const TxnDevCtx x, int p) {
  __shared__ uint32_t s_warp[kTxnScanThreads / 32];
  const uint32_t s = blockIdx.x;
  uint32_t carry = 0;
  for (uint32_t i0 = 0; i0 < x.nb; i0 += kTxnScanThreads) {
    const uint32_t i = i0 + threadIdx.x;
    const uint32_t v = i < x.nb ? x.ctatot[(size_t)s * x.nb + i] : 0u;
    uint32_t total;
    const uint32_t off = txn_block_scan(v, s_warp, &total);
    if (i < x.nb) x.base[p][(size_t)s * x.nb + i] = carry + off;
    carry += total;
  }
  if (threadIdx.x == 0) x.tot[s] = carry;
}

template <int KIND>
__global__ void __launch_bounds__(kTxnThreads) k_txn_emit(const TxnDevCtx x, int p) {
  using K = TxnKind<KIND>;
  const uint32_t c = blockIdx.x * kTxnThreads + threadIdx.x;
  if (c >= x.n_clients) return;
  const typename K::Client& cl = ((const typename K::Client*)x.cl)[c];
  TxnWriteSink<K::MSZ> w(x, p, c);
  K::emit(x.P, cl, w);
}
#endif  // __CUDACC__

}  // namespace dint
