// txn_workloads.cc -- (part of libdint_wl.so) the HOST driver of the reference's TATP and SmallBank closed-loop clients
// as round-based generators.  The state machines themselves are txn_clients.h, shared with the device driver
// (txn_clients.cuh); see there for the transaction types, mixes and the reference code they restate.
//
// A ROUND = every logical client has the requests of its current protocol step outstanding (1-9 wire
// records).  dint_txn_next() emits the round -- each client's records contiguous, in the order the reference
// pushes them per shard -- plus the destination shard of every record; dint_txn_feed() hands the replies back
// in the same layout and advances every client's state machine.
#include <cstdint>
#include <cstring>
#include <vector>

#include "txn_clients.h"

using namespace dint::txn;

namespace {

// the host sink: records appended to the round in push order, plus their destination shard
struct Out {
  uint8_t* req; uint8_t* dst; uint32_t n = 0; uint32_t msz = TM;
  void push(const uint8_t* rec, uint32_t shard, int ord) {
    memcpy(req + (size_t)n * msz, rec, msz);
    if (ord >= 0) req[(size_t)n * msz] = (uint8_t)ord;       // msg->ord = j: index inside the shard's list
    dst[n++] = (uint8_t)shard;
  }
};
// the replies of one client: contiguous, in push order
struct Contig {
  const uint8_t* r; uint32_t msz;
  const uint8_t* rec(int i) const { return r + (size_t)i * msz; }
};

}  // namespace

struct dint_txn {
  int kind;                 // 4 = tatp, 5 = smallbank
  uint32_t n_clients;
  Params P;
  std::vector<TatpClient> tc;
  std::vector<SbClient> sc;
  uint64_t st_requests = 0, st_txns = 0, st_committed = 0, st_rounds = 0;
  uint64_t st_by_type[8] = {0}, st_commit_by_type[8] = {0};

  void began(uint8_t txn) { st_txns++; st_by_type[txn]++; }
  // ev: what absorb returned; new_txn: the client's transaction after it
  void count(int ev, uint8_t new_txn) {
    if (ev < 0) return;
    if (ev & 1) { st_committed++; st_commit_by_type[ev >> 1]++; }
    began(new_txn);
  }
};

extern "C" {

// kind 4 (tatp): n_clients logical clients with gids [gid0, gid0 + n_clients); G shards; `subscribers`
// = kSubscriberNum of the key generator (reference 7,000,000; must equal the servers' population).
// kind 5 (smallbank): `subscribers` = kAccountNum (reference 24,000,000), hot set = 4 % of it (960,000).
dint_txn* dint_txn_create(int kind, uint32_t n_clients, uint32_t gid0, uint32_t n_shards, uint32_t subscribers) {
  // primary + 2 distinct backups need >= 3 shards; 1 = everything on one server (three copies of each write)
  if ((kind != 4 && kind != 5) || n_clients == 0 || n_shards == 0 || n_shards == 2 || n_shards > 8 || subscribers < 3) return nullptr;
  dint_txn* w = new dint_txn();
  w->kind = kind; w->n_clients = n_clients;
  w->P.G = n_shards; w->P.subscribers = subscribers; w->P.accounts = subscribers; w->P.hot = sb_hot_accounts(subscribers);
  if (kind == 4) {
    w->tc.assign(n_clients, TatpClient{});
    for (uint32_t i = 0; i < n_clients; i++) {
      w->tc[i].seed = 0xdeadbeefULL + gid0 + i;              // client_udp_shard.cc:1121
      tatp_begin(w->P, w->tc[i]);
      w->began(w->tc[i].txn);
    }
  } else {
    w->sc.assign(n_clients, SbClient{});
    for (uint32_t i = 0; i < n_clients; i++) {
      w->sc[i].seed = 0xdeadbeefULL + gid0 + i;
      sb_begin(w->P, w->sc[i]);
      w->began(w->sc[i].txn);
    }
  }
  return w;
}
void dint_txn_destroy(dint_txn* w) { delete w; }
uint32_t dint_txn_max_round(const dint_txn* w) { return w->n_clients * 9; }

// emits one round; returns the number of wire records.  req: capacity dint_txn_max_round() records;
// dst[i] = destination shard of record i.
uint64_t dint_txn_next(dint_txn* w, void* req, uint8_t* dst) {
  Out o;
  o.req = (uint8_t*)req; o.dst = dst;
  if (w->kind == 5) { o.msz = SMSZ; for (auto& c : w->sc) c.n_out = (uint8_t)sb_emit(w->P, c, o); }
  else for (auto& c : w->tc) c.n_out = (uint8_t)tatp_emit(w->P, c, o);
  w->st_requests += o.n;
  w->st_rounds++;
  return o.n;
}
void dint_txn_feed(dint_txn* w, const void* resp) {
  const uint8_t* r = (const uint8_t*)resp;
  if (w->kind == 5) {
    for (auto& c : w->sc) {
      const uint32_t n = c.n_out;        // read before absorb: it may start a new transaction
      const int ev = sb_absorb(w->P, c, Contig{r, SMSZ});
      w->count(ev, c.txn);                 // c.txn is read after absorb: the transaction it began
      r += (size_t)n * SMSZ;
    }
    return;
  }
  for (auto& c : w->tc) {
    const uint32_t n = c.n_out;
    const int ev = tatp_absorb(w->P, c, Contig{r, TM});
    w->count(ev, c.txn);
    r += (size_t)n * TM;
  }
}
// out: requests, transactions started, committed, rounds, then started-by-type[7], committed-by-type[7]
void dint_txn_stats(const dint_txn* w, uint64_t out[18]) {
  out[0] = w->st_requests; out[1] = w->st_txns; out[2] = w->st_committed; out[3] = w->st_rounds;
  for (int i = 0; i < 7; i++) { out[4 + i] = w->st_by_type[i]; out[11 + i] = w->st_commit_by_type[i]; }
}

}  // extern "C"
