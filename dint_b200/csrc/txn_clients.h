// txn_clients.h -- the reference's TATP and SmallBank closed-loop client state machines, ONE statement compiled twice:
// by g++ into libdint_wl.so (txn_workloads.cc, the host driver) and by nvcc into libdint_b200.so (txn_clients.cuh, the
// device driver: one thread per client).
//
// tatp/caladan/client_udp_shard.cc:177-1184 (seven transaction types, mix 35/35/10/2/14/2/2, tatp/udp/tatp.h:57-63) and
// smallbank/caladan/client_udp_shard.cc:169-1300 (six types, mix 15/15/15/25/15/15, hot-account skew
// smallbank/udp/smallbank.h:16-18,24-46).  Like the reference, each client draws from the LCG fastrand(seed = 0xdeadbeef +
// client gid) (tatp/udp/tatp.h:32-42), so a client's transaction stream is the reference's for that gid.
//
// A ROUND = every client has the requests of its current protocol step outstanding (1-9 wire records: the reference
// fans a step out to the shards in parallel and joins).  Per client and round the driver calls
//   *_emit(P, c, sink)     the step's records, in the order the reference pushes them, as sink.push(rec, shard, ord)
//                          (ord >= 0: the record's ord byte is set to it; -1: left as built).  Emit is const and draws
//                          nothing from the RNG, so a driver may run it several times on the same state: to count
//                          records per shard, to write them, and to find where their replies are.
//   *_absorb(P, c, rp)     the replies (rp.rec(i) = reply to the i-th pushed record); may finish the transaction and
//                          begin the next.  Returns -1, or (finished type << 1 | committed): a new transaction of type
//                          c.txn has then begun.  The counters live in the drivers.
// Sharding generalised from 3 to G shards (SURVEY.md section 8(e)): primary p = key % G, backups (p+1) % G and
// (p+2) % G, log records to those same three; G = 3 is exactly the reference.
//
// Device code rules kept here: plain structs (no std::), no function-local static tables (the mixes are thresholds),
// and SmallBank's balance arithmetic is float adds / subtracts / compares only, so there is no a*b+c for nvcc to
// contract into an FMA: host and device produce the same IEEE results.
#pragma once
#include <cstdint>
#include <cstring>
#include "common.cuh"

namespace dint {
namespace txn {

DINT_HD uint32_t fastrand(uint64_t* seed) {
  *seed = *seed * 1103515245ULL + 12345ULL;
  return (uint32_t)(*seed >> 32);
}
DINT_HD void put64(uint8_t* p, uint64_t v) { memcpy(p, &v, 8); }
DINT_HD uint64_t get64(const uint8_t* p) { uint64_t v; memcpy(&v, p, 8); return v; }
DINT_HD uint32_t get32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }
DINT_HD void put32(uint8_t* p, uint32_t v) { memcpy(p, &v, 4); }

// Most records one client sends ONE shard in one round (sizes the device driver's shard buffers).  TATP: a step
// pushes at most 4 records (update_subscriber_data's reads + locks), except the log fan-out of two records (2 x 3
// replicas = 6) -- which at G >= 3 sends each shard at most one copy of each record.  SmallBank: at most 3 rows; the log
// fan-out of 3 written rows is 9 records at G = 1 and at most 3 per shard at G >= 3.
DINT_HD uint32_t max_per_shard(int kind, uint32_t G) { return kind == 4 ? (G == 1 ? 6u : 4u) : (G == 1 ? 9u : 3u); }

struct Params {
  uint32_t G;                    // shards: 1 or 3..8
  uint32_t subscribers;          // tatp: kSubscriberNum of the key generator
  uint32_t accounts, hot;        // smallbank: kAccountNum, kHotAccountNum
};

// ================================================ TATP ==============================================
// wire: {ord@0, type@1, table@2, key@3, val@11[40], ver@51}  (tatp/udp/net.h:57-65)
constexpr int TM = 55;
enum { T_READ = 0, T_LOCK = 1, T_ABORT = 2, T_GRANT_READ = 4, T_NOT_EXIST = 6, T_GRANT_LOCK = 7, T_REJECT_LOCK = 8,
       T_COMMIT_PRIM = 12, T_COMMIT_BCK = 13, T_COMMIT_LOG = 14, T_INSERT_PRIM = 18, T_INSERT_BCK = 19,
       T_DELETE_PRIM = 22, T_DELETE_BCK = 23, T_DELETE_LOG = 24 };
enum { TB_SUB = 0, TB_SEC = 1, TB_ACC = 2, TB_SF = 3, TB_CF = 4 };
enum { X_GET_SUB = 0, X_GET_ACC, X_GET_DEST, X_UPD_SUB, X_UPD_LOC, X_INS_CF, X_DEL_CF };

struct TMsg { uint8_t b[TM]; };

struct TatpClient {
  uint64_t seed;
  uint8_t txn, phase, n_out;     // n_out: records of the step in flight (host driver bookkeeping)
  uint32_t s_id, vlr;
  uint8_t sf_type, start_time, end_time, cf_to_fetch;
  TMsg a, b, c, d;               // saved replies; roles depend on the transaction (see tatp_absorb)
  bool lock_a, lock_b;
};

DINT_HD uint64_t sub_nbr_of(uint32_t s_id) {            // tatp/udp/tatp.h:17-25,132-144
  uint64_t r = 0;
  for (int g = 0; g < 3; g++) {
    uint32_t i = s_id % 1000;
    s_id /= 1000;
    r |= ((uint64_t)(((i / 100) % 10) << 8 | ((i / 10) % 10) << 4 | (i % 10))) << (12 * g);
  }
  return r;
}
DINT_HD uint32_t nurand(const Params& P, uint64_t* seed) {            // tatp/udp/tatp.h:40-43
  const uint32_t x = fastrand(seed) % P.subscribers;
  return (x | (fastrand(seed) & 1048575u)) % P.subscribers;
}
DINT_HD void mk(TMsg& m, uint8_t type, uint8_t table, uint64_t key) {
  memset(m.b, 0, TM);
  m.b[1] = type; m.b[2] = table; put64(m.b + 3, key);
}
// key % G with 32-bit divides only (G < 2^16): a u64 remainder is a subroutine call on the SM
DINT_HD uint32_t mod_shards(uint64_t key, uint32_t G) {
  const uint32_t hi = (uint32_t)(key >> 32) % G, lo = (uint32_t)key % G, two32 = (0xffffffffu % G + 1u) % G;
  return (hi * two32 + lo) % G;
}
DINT_HD uint32_t prim(const Params& P, uint64_t key) { return mod_shards(key, P.G); }

// Push-order bookkeeping of one client's step: ord = index of the record inside its shard's list (msg->ord = j)
template <class Sink>
struct Pusher {
  Sink& s;
  uint32_t n;
  uint8_t per_shard[8];
  DINT_HD explicit Pusher(Sink& s_) : s(s_), n(0), per_shard{0, 0, 0, 0, 0, 0, 0, 0} {}
  DINT_HD void push(const TMsg& m, uint32_t shard, bool set_ord) {
    s.push(m.b, shard, set_ord ? (int)per_shard[shard % 8] : -1);
    per_shard[shard % 8]++;
    n++;
  }
};

// tatp/caladan/client_udp_shard.cc:1144 (mix) and the transaction parameters, in the reference's draw order
DINT_HD void tatp_begin(const Params& P, TatpClient& c) {
  const uint32_t x = fastrand(&c.seed) % 100;
  c.txn = (uint8_t)(x < 35 ? X_GET_SUB : x < 70 ? X_GET_ACC : x < 80 ? X_GET_DEST : x < 82 ? X_UPD_SUB
                    : x < 96 ? X_UPD_LOC : x < 98 ? X_INS_CF : X_DEL_CF);
  c.phase = 0;
  c.lock_a = c.lock_b = false;
  switch (c.txn) {
    case X_GET_SUB: c.s_id = nurand(P, &c.seed); break;
    case X_GET_ACC: c.s_id = nurand(P, &c.seed); c.sf_type = (uint8_t)((fastrand(&c.seed) & 3) + 1); break;
    case X_GET_DEST:
    case X_INS_CF:
      c.s_id = nurand(P, &c.seed);
      c.sf_type = (uint8_t)((fastrand(&c.seed) % 4) + 1);
      c.start_time = (uint8_t)((fastrand(&c.seed) % 3) * 8);
      c.end_time = (uint8_t)(fastrand(&c.seed) % 24);
      c.cf_to_fetch = (uint8_t)(c.start_time / 8 + 1);
      break;
    case X_UPD_SUB: c.s_id = nurand(P, &c.seed); c.sf_type = (uint8_t)((fastrand(&c.seed) % 4) + 1); break;
    case X_UPD_LOC: c.s_id = nurand(P, &c.seed); c.vlr = fastrand(&c.seed); break;
    default:  // X_DEL_CF
      c.s_id = nurand(P, &c.seed);
      c.sf_type = (uint8_t)((fastrand(&c.seed) % 4) + 1);
      c.start_time = (uint8_t)((fastrand(&c.seed) % 3) * 8);
      break;
  }
}
DINT_HD int tatp_finish(const Params& P, TatpClient& c, bool committed) {
  const int ev = (int)c.txn << 1 | (committed ? 1 : 0);
  tatp_begin(P, c);
  return ev;
}

DINT_HD uint64_t k_sub(const TatpClient& c) { return c.s_id; }
DINT_HD uint64_t k_sf(const TatpClient& c) { return (uint64_t)c.s_id | ((uint64_t)c.sf_type << 32); }
DINT_HD uint64_t k_cf(const TatpClient& c, uint32_t st) { return k_sf(c) | ((uint64_t)st << 40); }

// Replication fan-out of up to three records.  Per-shard arrival order follows the reference's push order:
// log: for shard { rec0, rec1 } (:490-499); backups: rec0,rec1 -> +1 then rec0,rec1 -> +2 (:523-531).
template <class O>
DINT_HD void emit_log(const Params& P, O& o, const TMsg* recs, int n, uint8_t type) {
  for (uint32_t s = 0; s < P.G; s++)
    for (int k = 0; k < n; k++) {
      const uint32_t p = prim(P, get64(recs[k].b + 3));
      for (uint32_t off = 0; off < 3; off++)
        if ((p + off) % P.G == s) { TMsg t = recs[k]; t.b[1] = type; o.push(t, s, false); }
    }
}
template <class O>
DINT_HD void emit_bck(const Params& P, O& o, const TMsg* recs, int n, uint8_t type) {
  for (uint32_t s = 0; s < P.G; s++)
    for (uint32_t off = 1; off <= 2; off++)
      for (int k = 0; k < n; k++)
        if ((prim(P, get64(recs[k].b + 3)) + off) % P.G == s) { TMsg t = recs[k]; t.b[1] = type; o.push(t, s, false); }
}
template <class O>
DINT_HD void emit_prim(const Params& P, O& o, const TMsg* recs, int n, uint8_t type) {
  for (uint32_t s = 0; s < P.G; s++)
    for (int k = 0; k < n; k++)
      if (prim(P, get64(recs[k].b + 3)) == s) { TMsg t = recs[k]; t.b[1] = type; o.push(t, s, false); }
}

// one protocol step of one client; returns the number of records pushed
template <class Sink>
DINT_HD uint32_t tatp_emit(const Params& P, const TatpClient& c, Sink& sink) {
  Pusher<Sink> o(sink);
  TMsg m;
  switch (c.txn) {
    case X_GET_SUB: mk(m, T_READ, TB_SUB, k_sub(c)); o.push(m, prim(P, k_sub(c)), false); break;                 // :177-199
    case X_GET_ACC: mk(m, T_READ, TB_ACC, k_sf(c)); o.push(m, prim(P, k_sf(c)), false); break;                   // :305-331 (ai_type in sf_type)
    case X_GET_DEST:                                                                                               // :202-302
      if (c.phase == 0) { mk(m, T_READ, TB_SF, k_sf(c)); o.push(m, prim(P, k_sf(c)), false); }
      else for (uint32_t i = 0; i < c.cf_to_fetch; i++) { mk(m, T_READ, TB_CF, k_cf(c, i * 8)); o.push(m, prim(P, k_cf(c, i * 8)), true); }
      break;
    case X_UPD_SUB:                                                                                                // :334-571
      switch (c.phase) {
        case 0:   // a = sub read, b = sub lock, c = specfac read, d = specfac lock
          mk(m, T_READ, TB_SUB, k_sub(c)); o.push(m, prim(P, k_sub(c)), true);
          mk(m, T_LOCK, TB_SUB, k_sub(c)); o.push(m, prim(P, k_sub(c)), true);
          mk(m, T_READ, TB_SF, k_sf(c)); o.push(m, prim(P, k_sf(c)), true);
          mk(m, T_LOCK, TB_SF, k_sf(c)); o.push(m, prim(P, k_sf(c)), true);
          break;
        case 1: { TMsg t = c.b; t.b[1] = T_ABORT; o.push(t, prim(P, k_sub(c)), false); break; }                   // release sub lock
        case 2: { TMsg t = c.d; t.b[1] = T_ABORT; o.push(t, prim(P, k_sf(c)), false); break; }                    // release specfac lock
        case 3:   // verify
          mk(m, T_READ, TB_SUB, k_sub(c)); o.push(m, prim(P, k_sub(c)), true);
          mk(m, T_READ, TB_SF, k_sf(c)); o.push(m, prim(P, k_sf(c)), true);
          break;
        case 4: { TMsg rr[2] = {c.a, c.c}; emit_log(P, o, rr, 2, T_COMMIT_LOG); break; }      // :487-518
        case 5: { TMsg rr[2] = {c.a, c.c}; emit_bck(P, o, rr, 2, T_COMMIT_BCK); break; }      // :520-548
        default: { TMsg rr[2] = {c.a, c.c}; emit_prim(P, o, rr, 2, T_COMMIT_PRIM); break; }   // :550-568
      }
      break;
    case X_UPD_LOC:                                                                                                // :574-728
      switch (c.phase) {
        case 0: mk(m, T_READ, TB_SEC, sub_nbr_of(c.s_id)); o.push(m, prim(P, sub_nbr_of(c.s_id)), false); break;
        case 1:   // a = sub read, b = sub lock
          mk(m, T_READ, TB_SUB, k_sub(c)); o.push(m, prim(P, k_sub(c)), true);
          mk(m, T_LOCK, TB_SUB, k_sub(c)); o.push(m, prim(P, k_sub(c)), true);
          break;
        case 2: mk(m, T_READ, TB_SUB, k_sub(c)); o.push(m, prim(P, k_sub(c)), false); break;                      // verify
        case 3: { TMsg t = c.b; t.b[1] = T_ABORT; o.push(t, prim(P, k_sub(c)), false); break; }
        case 4: emit_log(P, o, &c.a, 1, T_COMMIT_LOG); break;
        case 5: emit_bck(P, o, &c.a, 1, T_COMMIT_BCK); break;
        default: emit_prim(P, o, &c.a, 1, T_COMMIT_PRIM); break;
      }
      break;
    case X_INS_CF:                                                                                                 // :731-951
      switch (c.phase) {
        case 0: mk(m, T_READ, TB_SEC, sub_nbr_of(c.s_id)); o.push(m, prim(P, sub_nbr_of(c.s_id)), false); break;
        case 1: mk(m, T_READ, TB_SF, k_sf(c)); o.push(m, prim(P, k_sf(c)), false); break;                         // c = specfac read
        case 2:   // a = callfwd read, b = callfwd lock
          mk(m, T_READ, TB_CF, k_cf(c, c.start_time)); o.push(m, prim(P, k_cf(c, c.start_time)), true);
          mk(m, T_LOCK, TB_CF, k_cf(c, c.start_time)); o.push(m, prim(P, k_cf(c, c.start_time)), true);
          break;
        case 3: { TMsg t = c.b; t.b[1] = T_ABORT; o.push(t, prim(P, k_cf(c, c.start_time)), false); break; }
        case 4:   // verify specfac version + callfwd still absent
          mk(m, T_READ, TB_SF, k_sf(c)); o.push(m, prim(P, k_sf(c)), true);
          mk(m, T_READ, TB_CF, k_cf(c, c.start_time)); o.push(m, prim(P, k_cf(c, c.start_time)), true);
          break;
        case 5: emit_log(P, o, &c.a, 1, T_COMMIT_LOG); break;
        case 6: emit_bck(P, o, &c.a, 1, T_INSERT_BCK); break;
        default: emit_prim(P, o, &c.a, 1, T_INSERT_PRIM); break;
      }
      break;
    default:  // X_DEL_CF                                                                                          // :954-1117
      switch (c.phase) {
        case 0: mk(m, T_READ, TB_SEC, sub_nbr_of(c.s_id)); o.push(m, prim(P, sub_nbr_of(c.s_id)), false); break;
        case 1:   // a = callfwd read, b = callfwd lock
          mk(m, T_READ, TB_CF, k_cf(c, c.start_time)); o.push(m, prim(P, k_cf(c, c.start_time)), true);
          mk(m, T_LOCK, TB_CF, k_cf(c, c.start_time)); o.push(m, prim(P, k_cf(c, c.start_time)), true);
          break;
        case 2: { TMsg t = c.b; t.b[1] = T_ABORT; o.push(t, prim(P, k_cf(c, c.start_time)), false); break; }
        case 3: mk(m, T_READ, TB_CF, k_cf(c, c.start_time)); o.push(m, prim(P, k_cf(c, c.start_time)), false); break;   // verify
        case 4: emit_log(P, o, &c.a, 1, T_DELETE_LOG); break;
        case 5: emit_bck(P, o, &c.a, 1, T_DELETE_BCK); break;
        default: emit_prim(P, o, &c.a, 1, T_DELETE_PRIM); break;
      }
      break;
  }
  return o.n;
}

// rp.rec(i): the reply to the i-th record tatp_emit pushed for this client's step
template <class Replies>
DINT_HD int tatp_absorb(const Params& P, TatpClient& c, const Replies& rp) {
  auto R = [&](int i) { TMsg m; memcpy(m.b, rp.rec(i), TM); return m; };
  auto type = [&](int i) { return rp.rec(i)[1]; };
  auto ver = [&](const TMsg& m) { return get32(m.b + 51); };
  switch (c.txn) {
    case X_GET_SUB: return tatp_finish(P, c, true);
    case X_GET_ACC: return tatp_finish(P, c, type(0) == T_GRANT_READ);
    case X_GET_DEST:
      if (c.phase == 0) {
        if (type(0) == T_NOT_EXIST || rp.rec(0)[11] == 0) return tatp_finish(P, c, false);   // record absent or is_active == 0 (:231-237)
        c.phase = 1;
      } else {
        bool ok = false;
        for (uint32_t i = 0; i < c.cf_to_fetch; i++)
          if (type(i) == T_GRANT_READ && i * 8 <= c.start_time && c.end_time < rp.rec(i)[11]) ok = true;   // :287-297
        return tatp_finish(P, c, ok);
      }
      break;
    case X_UPD_SUB:
      switch (c.phase) {
        case 0:
          c.a = R(0); c.b = R(1); c.c = R(2); c.d = R(3);
          c.lock_a = type(1) == T_GRANT_LOCK; c.lock_b = type(3) == T_GRANT_LOCK;
          if (type(2) == T_NOT_EXIST || !c.lock_a || !c.lock_b) {         // :400-420
            if (c.lock_a) c.phase = 1; else if (c.lock_b) c.phase = 2; else return tatp_finish(P, c, false);
          } else {
            uint16_t bits = (uint16_t)fastrand(&c.seed);                  // sub_val->bits (:425)
            memcpy(c.a.b + 11 + 30, &bits, 2);
            c.c.b[11 + 2] = (uint8_t)fastrand(&c.seed);                   // specfac_val->data_a (:429)
            c.phase = 3;
          }
          break;
        case 1: if (c.lock_b) c.phase = 2; else return tatp_finish(P, c, false); break;
        case 2: return tatp_finish(P, c, false);
        case 3:
          if (ver(c.a) != get32(rp.rec(0) + 51) || ver(c.c) != get32(rp.rec(1) + 51)) { c.phase = 1; }   // abort both (:470-484)
          else {
            put32(c.a.b + 51, ver(c.a) + 1); put32(c.c.b + 51, ver(c.c) + 1);                        // :487-488
            c.phase = 4;
          }
          break;
        case 4: c.phase = 5; break;
        case 5: c.phase = 6; break;
        default: return tatp_finish(P, c, true);
      }
      break;
    case X_UPD_LOC:
      switch (c.phase) {
        case 0: c.phase = 1; break;
        case 1:
          c.a = R(0); c.b = R(1);
          if (type(1) == T_REJECT_LOCK) return tatp_finish(P, c, false);   // :642
          memcpy(c.a.b + 11 + 36, &c.vlr, 4); c.phase = 2;                   // sub_val->vlr_location (:646)
          break;
        case 2:
          if (get32(rp.rec(0) + 51) != ver(c.a)) c.phase = 3;                // :661-667
          else { put32(c.a.b + 51, ver(c.a) + 1); c.phase = 4; }
          break;
        case 3: return tatp_finish(P, c, false);
        case 4: c.phase = 5; break;
        case 5: c.phase = 6; break;
        default: return tatp_finish(P, c, true);
      }
      break;
    case X_INS_CF:
      switch (c.phase) {
        case 0: c.phase = 1; break;
        case 1: c.c = R(0); if (type(0) == T_NOT_EXIST) return tatp_finish(P, c, false); c.phase = 2; break;   // :781
        case 2:
          c.a = R(0); c.b = R(1);
          if (type(0) == T_GRANT_READ || type(1) == T_REJECT_LOCK) {       // :831-841: row exists or lock refused
            if (type(1) == T_GRANT_LOCK) c.phase = 3; else return tatp_finish(P, c, false);
          } else {
            c.a.b[11 + 1] = 101;                                           // numberx[0] = magic (:846)
            c.a.b[11 + 0] = c.end_time;                                    // end_time (:847)
            c.phase = 4;
          }
          break;
        case 3: return tatp_finish(P, c, false);
        case 4:
          if (ver(c.c) != get32(rp.rec(0) + 51) || type(1) == T_GRANT_READ) c.phase = 3;   // :884-891
          else { put32(c.a.b + 51, 0); c.phase = 5; }                        // :894 ver = 0
          break;
        case 5: c.phase = 6; break;
        case 6: c.phase = 7; break;
        default: return tatp_finish(P, c, true);
      }
      break;
    default:  // X_DEL_CF
      switch (c.phase) {
        case 0: c.phase = 1; break;
        case 1:
          c.a = R(0); c.b = R(1);
          if (type(0) == T_NOT_EXIST || type(1) == T_REJECT_LOCK) {        // :1024-1033
            if (type(1) == T_GRANT_LOCK) c.phase = 2; else return tatp_finish(P, c, false);
          } else c.phase = 3;
          break;
        case 2: return tatp_finish(P, c, false);
        case 3:
          if (type(0) == T_NOT_EXIST || get32(rp.rec(0) + 51) != ver(c.a)) c.phase = 2;   // :1053-1060
          else c.phase = 4;
          break;
        case 4: c.phase = 5; break;
        case 5: c.phase = 6; break;
        default: return tatp_finish(P, c, true);
      }
      break;
  }
  return -1;
}

// ================================================ SmallBank =========================================
// wire: {ord@0, type@1, table@2, key@3, val@11[8] = {u32 magic; float bal}, ver@19}  (smallbank/udp/net.h:43-52)
constexpr int SMSZ = 23;
enum { S_ACQ_S = 0, S_ACQ_X = 1, S_REL_S = 2, S_REL_X = 3, S_COMMIT_PRIM = 4, S_COMMIT_BCK = 5, S_COMMIT_LOG = 6,
       S_GRANT_S = 7, S_REJECT_S = 8, S_GRANT_X = 9, S_REJECT_X = 10 };
enum { B_AMALGAMATE = 0, B_BALANCE, B_DEPOSIT, B_SEND, B_TRANSACT, B_WRITECHECK };
enum { SP_ACQ = 0, SP_REL_ABORT, SP_LOG, SP_BCK, SP_PRIM, SP_RELEASE };
struct SbRow { uint8_t table, excl, write, granted; uint64_t acct; TMsg m; };
struct SbClient {
  uint64_t seed;
  uint8_t txn, phase, n_rows, n_out, rel_idx;    // n_out: records of the step in flight (host driver bookkeeping)
  SbRow r[3];
};
DINT_HD float get_bal(const TMsg& m) { float f; memcpy(&f, m.b + 11 + 4, 4); return f; }
DINT_HD void set_bal(TMsg& m, float f) { memcpy(m.b + 11 + 4, &f, 4); }

DINT_HD void sb_get_account(const Params& P, uint64_t* seed, uint64_t* a) {            // smallbank/udp/smallbank.h:24-30
  if (fastrand(seed) % 100 < 90) *a = fastrand(seed) % P.hot; else *a = fastrand(seed) % P.accounts;
}
DINT_HD void sb_get_two_accounts(const Params& P, uint64_t* seed, uint64_t* a0, uint64_t* a1) {   // smallbank.h:32-46
  const uint32_t n = (fastrand(seed) % 100 < 90) ? P.hot : P.accounts;
  *a0 = fastrand(seed) % n;
  *a1 = fastrand(seed) % n;
  while (*a1 == *a0) *a1 = fastrand(seed) % n;
}
DINT_HD void sb_row(SbRow& r, uint8_t table, bool excl, bool write, uint64_t acct) {
  r.table = table; r.excl = excl; r.write = write; r.granted = 0; r.acct = acct;
}
DINT_HD void sb_begin(const Params& P, SbClient& c) {
  const uint32_t x = fastrand(&c.seed) % 100;
  c.txn = (uint8_t)(x < 15 ? B_AMALGAMATE : x < 30 ? B_BALANCE : x < 45 ? B_DEPOSIT : x < 70 ? B_SEND
                    : x < 85 ? B_TRANSACT : B_WRITECHECK);
  c.phase = SP_ACQ;
  uint64_t a0, a1;
  switch (c.txn) {
    case B_AMALGAMATE:       // client_udp_shard.cc:169-438: sav(a0) X, chk(a0) X, chk(a1) X, all written
      sb_get_two_accounts(P, &c.seed, &a0, &a1);
      c.n_rows = 3; sb_row(c.r[0], 0, true, true, a0); sb_row(c.r[1], 1, true, true, a0); sb_row(c.r[2], 1, true, true, a1);
      break;
    case B_BALANCE:          // :441-578: sav(a) S, chk(a) S, read only
      sb_get_account(P, &c.seed, &a0);
      c.n_rows = 2; sb_row(c.r[0], 0, false, false, a0); sb_row(c.r[1], 1, false, false, a0);
      break;
    case B_DEPOSIT:          // :581-684: chk(a) X += 1.3
      sb_get_account(P, &c.seed, &a0);
      c.n_rows = 1; sb_row(c.r[0], 1, true, true, a0);
      break;
    case B_SEND:             // :687-932: chk(a0) X, chk(a1) X, move 5.0
      sb_get_two_accounts(P, &c.seed, &a0, &a1);
      c.n_rows = 2; sb_row(c.r[0], 1, true, true, a0); sb_row(c.r[1], 1, true, true, a1);
      break;
    case B_TRANSACT:         // :935-1038: sav(a) X += 20.20
      sb_get_account(P, &c.seed, &a0);
      c.n_rows = 1; sb_row(c.r[0], 0, true, true, a0);
      break;
    default:                 // B_WRITECHECK :1041-1239: sav(a) S, chk(a) X -= 5 (+1 penalty)
      sb_get_account(P, &c.seed, &a0);
      c.n_rows = 2; sb_row(c.r[0], 0, false, false, a0); sb_row(c.r[1], 1, true, true, a0);
      break;
  }
}
DINT_HD int sb_finish(const Params& P, SbClient& c, bool ok) {
  const int ev = (int)c.txn << 1 | (ok ? 1 : 0);
  sb_begin(P, c);
  return ev;
}
template <class Sink>
DINT_HD uint32_t sb_emit(const Params& P, const SbClient& c, Sink& sink) {
  Pusher<Sink> o(sink);
  TMsg rr[3];
  int nw = 0;
  for (int i = 0; i < c.n_rows; i++) if (c.r[i].write) rr[nw++] = c.r[i].m;
  switch (c.phase) {
    case SP_ACQ:
      for (int i = 0; i < c.n_rows; i++) {
        TMsg m; memset(m.b, 0, sizeof m.b);
        m.b[1] = c.r[i].excl ? S_ACQ_X : S_ACQ_S; m.b[2] = c.r[i].table; put64(m.b + 3, c.r[i].acct);
        o.push(m, mod_shards(c.r[i].acct, P.G), c.n_rows > 1);
      }
      break;
    case SP_REL_ABORT: {
      TMsg m = c.r[c.rel_idx].m; m.b[1] = c.r[c.rel_idx].excl ? S_REL_X : S_REL_S;
      o.push(m, mod_shards(c.r[c.rel_idx].acct, P.G), false);
      break;
    }
    case SP_LOG: emit_log(P, o, rr, nw, S_COMMIT_LOG); break;
    case SP_BCK: emit_bck(P, o, rr, nw, S_COMMIT_BCK); break;
    case SP_PRIM: emit_prim(P, o, rr, nw, S_COMMIT_PRIM); break;
    default:
      for (int i = 0; i < c.n_rows; i++) {
        TMsg m = c.r[i].m; m.b[1] = c.r[i].excl ? S_REL_X : S_REL_S;
        o.push(m, mod_shards(c.r[i].acct, P.G), c.n_rows > 1);
      }
      break;
  }
  return o.n;
}
DINT_HD int sb_next_granted(const SbClient& c, int from) {
  for (int i = from; i < c.n_rows; i++) if (c.r[i].granted) return i;
  return -1;
}
template <class Replies>
DINT_HD int sb_absorb(const Params& P, SbClient& c, const Replies& rp) {
  switch (c.phase) {
    case SP_ACQ: {
      bool all = true;
      for (int i = 0; i < c.n_rows; i++) {
        memcpy(c.r[i].m.b, rp.rec(i), SMSZ);
        const uint8_t t = c.r[i].m.b[1];
        c.r[i].granted = (t == S_GRANT_S || t == S_GRANT_X);
        all &= (bool)c.r[i].granted;
      }
      bool logic_abort = false;
      if (all) {
        TMsg& m0 = c.r[0].m;
        switch (c.txn) {
          case B_AMALGAMATE:
            set_bal(c.r[2].m, get_bal(c.r[2].m) + (get_bal(c.r[0].m) + get_bal(c.r[1].m)));
            set_bal(c.r[0].m, 0.f); set_bal(c.r[1].m, 0.f);
            break;
          case B_DEPOSIT: set_bal(m0, get_bal(m0) + 1.3f); break;
          case B_SEND:
            if (get_bal(c.r[0].m) < 5.0f) logic_abort = true;
            else { set_bal(c.r[0].m, get_bal(c.r[0].m) - 5.0f); set_bal(c.r[1].m, get_bal(c.r[1].m) + 5.0f); }
            break;
          case B_TRANSACT: set_bal(m0, get_bal(m0) + 20.20f); break;
          case B_WRITECHECK:
            if (get_bal(c.r[0].m) + get_bal(c.r[1].m) < 5.0f) set_bal(c.r[1].m, get_bal(c.r[1].m) - 6.0f);
            else set_bal(c.r[1].m, get_bal(c.r[1].m) - 5.0f);
            break;
          default: break;
        }
      }
      if (!all || logic_abort) {
        const int g = sb_next_granted(c, 0);
        if (g < 0) return sb_finish(P, c, false);
        c.rel_idx = (uint8_t)g; c.phase = SP_REL_ABORT;
      } else if (c.txn == B_BALANCE) {
        c.phase = SP_RELEASE;
      } else {
        for (int i = 0; i < c.n_rows; i++) if (c.r[i].write) put32(c.r[i].m.b + 19, get32(c.r[i].m.b + 19) + 1);   // ver++
        c.phase = SP_LOG;
      }
      break;
    }
    case SP_REL_ABORT: {
      const int g = sb_next_granted(c, c.rel_idx + 1);
      if (g < 0) return sb_finish(P, c, false);
      c.rel_idx = (uint8_t)g;
      break;
    }
    case SP_LOG: c.phase = SP_BCK; break;
    case SP_BCK: c.phase = SP_PRIM; break;
    case SP_PRIM: c.phase = SP_RELEASE; break;
    default: return sb_finish(P, c, true);
  }
  return -1;
}

// smallbank's hot set: kHotAccountNum / kAccountNum of the reference (960,000 of 24,000,000), at least 2
DINT_HD uint32_t sb_hot_accounts(uint32_t accounts) {
  const uint32_t h = (uint32_t)((uint64_t)accounts * 960000 / 24000000);
  return h < 2 ? 2u : h;
}

}  // namespace txn
}  // namespace dint
