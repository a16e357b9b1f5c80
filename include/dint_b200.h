/*
 * dint_b200.h -- C ABI of libdint_b200.so, the B200-resident replacement for the per-request
 * server hot path of DINT (NSDI'24).
 *
 * The reference has no plugin/FFI API: the public interface of its hot path is the WIRE PROTOCOL
 * (one packed struct per UDP datagram; the reply is the same buffer with type/val/ver rewritten and
 * echoed to the sender) plus the server command line.  This ABI is what a transport front-end (UDP
 * recvmmsg/sendmmsg batcher, Caladan, DPDK burst loop) binds instead of calling the reference's
 * handler body one datagram at a time.  Each entry point cites the reference code it replaces
 * (paths relative to the DINT repository root).
 *
 * Semantics contract of dint_submit*: the n requests are processed AS IF one reference server
 * thread had received them one by one in index order (request i sees the effects of every j < i);
 * resp[i] is byte-for-byte the datagram that thread would have sent for req[i].  kRetry-class
 * replies, which exist only for thread-vs-thread spin contention in the reference
 * (lock_2pl/udp/server.cc:75-80, smallbank/udp/server_shard.cc:111-119), are never produced.
 *
 * There is no CPU fallback: every compute entry point fails with DINT_ENODEV when no CUDA device
 * is usable.
 */
#ifndef DINT_B200_H
#define DINT_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* Which reference server the engine stands in for. */
enum dint_kind {
  DINT_LOCK2PL = 0,   /* lock_2pl/udp/server.cc:55-123       wire: lock_2pl/udp/net.h:25-31   (6 B)  */
  DINT_FASST = 1,     /* lock_fasst/udp/server.cc:49-120     wire: lock_fasst/udp/net.h:25-31 (9 B)  */
  DINT_LOG = 2,       /* log_server/udp/server.cc:48-89      wire: log_server/udp/net.h:23-30 (53 B) */
  DINT_STORE = 3,     /* store/udp/server.cc:50-98           wire: store/udp/net.h:34-41      (53 B) */
  DINT_TATP = 4,      /* tatp/udp/server_shard.cc:88-211     wire: tatp/udp/net.h:57-65       (55 B) */
  DINT_SMALLBANK = 5, /* smallbank/udp/server_shard.cc:82-190 wire: smallbank/udp/net.h:43-52 (23 B) */
  DINT_NUM_KINDS = 6
};

/* Error codes (negative return values). */
enum {
  DINT_OK = 0,
  DINT_EINVAL = -22,  /* bad argument */
  DINT_ENOMEM = -12,  /* device/host allocation failed */
  DINT_ENODEV = -19,  /* no usable CUDA device (there is no CPU fallback) */
  DINT_EIO = -5,      /* a CUDA call failed; see dint_last_error() */
  DINT_EPROTO = -71   /* the batch held a request the reference would panic() on; the offending
                         replies carry type 0xFF, the rest of the batch was processed normally */
};

/*
 * Sizes the reference bakes in as constexpr (SURVEY.md section 5 "config / flags").  Defaults =
 * the reference constants; dint_default_cfg() fills them in.
 */
typedef struct dint_cfg {
  uint32_t lock_slots;     /* kLockHashSize 36,000,000: lock_2pl/udp/utils.h:16, lock_fasst/udp/utils.h:16 */
  uint32_t log_ring;       /* kMaxLogEntryNum 1,000,000: log_server/udp/utils.h:16, tatp/udp/kvs.h:19 */
  uint32_t subs_sizing;    /* kSubscriberNum that SIZES hash tables and lock-hash moduli:
                              store 2,000,000 (store/udp/tatp.h:10, server.cc:113),
                              tatp 7,000,000 (tatp/udp/tatp.h:28, server_shard.cc:75-79, tatp.h:12-14) */
  uint32_t subs_populate;  /* subscribers dint_populate() inserts (<= subs_sizing; a prefix of the
                              reference population, whose LCG streams are sequential in s_id) */
  uint32_t accts_sizing;   /* smallbank kAccountNum 24,000,000 (smallbank/udp/smallbank.h:17,
                              server_shard.cc:72-73, smallbank.h:10-14) */
  uint32_t accts_populate; /* accounts dint_populate() inserts */
  uint32_t n_shards;       /* key-space shards (GPUs); this engine owns lock slots / buckets with
                              slot % n_shards == shard_id.  1 = whole key space. */
  uint32_t shard_id;
  uint32_t chunk;          /* requests per internal launch group (0 = default 1<<20) */
  uint32_t kv_capacity_log2[5]; /* per-table open-addressing capacity (0 = auto: >= 2x expected keys) */
  uint32_t flags;          /* reserved, must be 0 */
  uint32_t txn_shards;     /* tatp / smallbank replica placement (tatp/caladan/client_udp_shard.cc:187,490-531 generalised
                              from 3 to G shards): 0 or 1 = this server holds every key (the reference: all three
                              shards populate everything); G > 3: dint_populate() keeps only keys whose primary
                              (key % G) is txn_shard_id, txn_shard_id-1 or txn_shard_id-2 (mod G) */
  uint32_t txn_shard_id;
  uint32_t reserved[2];
} dint_cfg;

typedef struct dint_engine dint_engine;

/* Counters since create (or the last dint_reset_stats). */
typedef struct dint_stats {
  uint64_t requests;        /* requests processed */
  uint64_t chunks;          /* internal launch groups */
  uint64_t kernel_launches; /* kernels launched by this engine */
  uint64_t conflicted;      /* requests that took the ordered (intra-batch conflict) path */
  uint64_t max_run;         /* longest same-slot run seen on the ordered path */
  uint64_t errors;          /* requests answered with type 0xFF */
  uint64_t h2d_bytes, d2h_bytes;
  uint64_t kv_rebuilds;     /* KV tables rehashed to reclaim tombstones (the reference frees entries on delete:
                               store/udp/kvs.h:124-133) */
  uint64_t fallback_chunks; /* chunks whose listed requests overflowed a replay bucket and were replayed by the
                               radix-sort fallback instead */
  uint64_t reserved[2];
} dint_stats;

/* Per-kernel device time, accumulated with CUDA events while profiling is on. */
typedef struct dint_kernel_time {
  char name[32];
  uint64_t launches;
  double total_ms;
} dint_kernel_time;

uint32_t dint_msg_size(int kind);                       /* sizeof(struct message) of that server */
void dint_default_cfg(int kind, dint_cfg *cfg);

/* Replaces server start-up: main() + net_init() + kvs_init()/array definitions
 * (lock_fasst/udp/server.cc:124-149, store/udp/server.cc:101-132, tatp/udp/server_shard.cc:71-85,278-320).
 * Allocates all state in HBM of CUDA device `device`; tables start EMPTY (see dint_populate). */
int dint_create(int kind, const dint_cfg *cfg, int device, dint_engine **out);
void dint_destroy(dint_engine *e);

/* Replaces populate_table / populate_*_table / populate_saving_and_checking_tables
 * (store/udp/tatp.h:45-66, tatp/udp/tatp.h:285-412, smallbank/udp/smallbank.h:105-127):
 * the same deterministic population, bytes the reference leaves uninitialised are zero. */
int dint_populate(dint_engine *e);

/* Bulk kvs_insert (store/udp/kvs.h:77-104) of n (key, value) pairs from HOST arrays into `table`;
 * vals is n * val_size bytes (40; smallbank 8).  Also the path that loads an image dumped from
 * another server.  Keys must not already exist (the reference's insert never checks either). */
int dint_load(dint_engine *e, int table, const uint64_t *keys, const void *vals, uint64_t n);

/* Replaces the `while (1) { net_recv; handler body; net_send; }` loop for a batch
 * (lock_2pl/udp/server.cc:70-122, lock_fasst/udp/server.cc:78-119, log_server/udp/server.cc:73-88,
 * store/udp/server.cc:75-97, tatp/udp/server_shard.cc:113-210, smallbank/udp/server_shard.cc:107-189).
 * req/resp: HOST arrays of n packed wire structs (resp may alias req).  Copies in, computes on the
 * GPU, copies out, returns when resp is complete.  Returns 0, DINT_EPROTO, or another error. */
int dint_submit(dint_engine *e, const void *req, uint64_t n, void *resp);

/* Same, with DEVICE arrays (16-byte aligned), asynchronous on `cuda_stream` (a cudaStream_t; NULL = the
 * legacy default stream, as everywhere in CUDA).  Successive calls must be issued on streams that
 * order them (the engine's state is one sequential history).  Request errors surface at the next
 * dint_sync()/dint_get_stats(). */
int dint_submit_device(dint_engine *e, const void *req_dev, uint64_t n, void *resp_dev, void *cuda_stream);
/* Multi-GPU routing helper (SURVEY.md section 8(e)): owner[i] = shard that owns request i's group
 * (lock slot / bucket: fasthash64 % size % n_shards -- the same modulus the single server would use, so
 * collision behaviour is unchanged by sharding); 0xFF for records no shard owns (invalid / log-only
 * requests are served by whoever receives them: owner = shard_id).  Device pointers, async on stream. */
int dint_route_owner(dint_engine *e, const void *req_dev, uint64_t n, uint8_t *owner_dev, void *cuda_stream);
/* Dispatch / combine for the multi-GPU exchange.  dint_route_partition: stable partition of n wire records by
 * owner_dev[i] (< n_shards; from dint_route_owner, or chosen by the client as in tatp / smallbank) into
 * sorted_dev (grouped by shard, each group in original order); perm_dev[pos] = original index;
 * counts_dev[0..n_shards) = records per shard.  dint_route_unpermute: out_dev[perm[pos]] = sorted_dev[pos].
 * All pointers are device pointers; asynchronous on cuda_stream. */
int dint_route_partition(dint_engine *e, const void *req_dev, const uint8_t *owner_dev, uint64_t n, uint32_t n_shards,
                         void *sorted_dev, uint32_t *perm_dev, uint32_t *counts_dev, void *cuda_stream);
/* Fixed-capacity dispatch / combine (no host round trip for the split sizes), local or over NVLink peer memory.
 * Every source rank sends every shard o one SLAB of `cap` records: its records for o first, in request order,
 * then padding records (every byte 0xFE: a padding record is answered unchanged and touches nothing).
 *   dint_route_dispatch: ONE kernel, one pass over the batch (single-pass prefix sums by decoupled look-back; n < 2^27).
 *     owner_in_dev = client-chosen shard per record (tatp / smallbank
 *     placement) or NULL = computed as dint_route_owner would (needs n_shards == cfg.n_shards).  slab_ptrs->p[o] =
 *     device address of THIS source's slab for shard o: inside a local send buffer (then exchange the slabs with
 *     an all-to-all) or inside rank o's receive buffer mapped over NVLink (then no collective is needed: with
 *     sig_ptrs != NULL the kernel's last CTA release-stores `epoch` to word `rank` of sig_ptrs->p[o] for every o).
 *     Outputs for the combine: owner_dev[n] (one byte per record, 0xFF = undeliverable) and tilebase_dev
 *     [ceil(n / dint_route_tile_records())][8].  flags_dev[0] += records that did not fit their slab.
 *   dint_route_combine: reply_slab_ptrs->p[o] = where shard o's replies to THIS source's slab are (local receive
 *     buffer or rank o's reply buffer over NVLink); out_dev[i] = reply to request i (0xFF bytes if undelivered).
 * The reference does this routing in its clients (e.g. `key % kNumServers` before sendto,
 * tatp/caladan/client_ebpf_shard.cc); with this call any rank may receive any request. */
typedef struct dint_peer_ptrs { uint64_t p[8]; } dint_peer_ptrs;
uint32_t dint_route_tile_records(dint_engine *e);
int dint_route_dispatch(dint_engine *e, const void *req_dev, const uint8_t *owner_in_dev, uint64_t n, uint32_t n_shards,
                        uint32_t rank, uint32_t cap, const dint_peer_ptrs *slab_ptrs, const dint_peer_ptrs *sig_ptrs,
                        uint32_t epoch, uint8_t *owner_dev, uint32_t *tilebase_dev, uint32_t *flags_dev, void *cuda_stream);
int dint_route_combine(dint_engine *e, const dint_peer_ptrs *reply_slab_ptrs, const uint8_t *owner_dev,
                       const uint32_t *tilebase_dev, uint64_t n, uint32_t n_shards, uint32_t cap, void *out_dev,
                       void *cuda_stream);
/* Epoch flags for the exchange over peer memory (one process per GPU; the buffers are each rank's
 * symmetric-memory regions mapped into this process; sig_ptrs->p[o] = rank o's signal words [n_shards] u32):
 *   dint_p2p_wait:    blocks the stream until local_sig[0..n_shards) have all reached epoch (acquire).
 *   dint_p2p_signal:  release-signals epoch to every peer's sig[rank] (e.g. replies ready in my reply buffer).
 * flags_dev[1] = 1 if a wait timed out. */
int dint_p2p_wait(dint_engine *e, const uint32_t *local_sig_dev, uint32_t n_shards, uint32_t epoch, uint32_t *flags_dev,
                  void *cuda_stream);
int dint_p2p_signal(dint_engine *e, const dint_peer_ptrs *sig_ptrs, uint32_t n_shards, uint32_t rank, uint32_t epoch,
                    void *cuda_stream);
/* The whole sharded step over NVLink peer memory, driven from ONE host call per sequence of batches (what
 * dint_b200/shard.py uses at N > 1, one process per GPU).  Every rank owns n_sets (2..4) buffer sets {inbox, return
 * buffer}, each n_shards * cap records (cap a multiple of 128), plus one 256-byte signal block (epoch words: requests
 * written [n_sets][8] at +0, replies written [8] at +128), all in memory its peers map (CUDA IPC / torch symmetric memory), zeroed once.
 *   inbox_sets[s].p[o], retbox_sets[s].p[o]: device address of rank o's set s; sig_blocks->p[o]: rank o's block.
 * dint_shard_submit_many: k batches of n (<= max_n) records each, the same k on every rank; batch j+1 is partitioned
 * into the OWNERS' inboxes (dint_route_dispatch) while batch j runs through the local engine on cuda_stream -- its
 * apply kernel stores every reply tile straight into the SOURCE's return buffer (posted stores) -- and the replies of
 * batch j-1 are put back in request order from the local return buffer (dint_route_combine); out_dev[j] is complete
 * when cuda_stream reaches the end of the call.  The engine sees the batches in order, so the result equals k
 * sequential collective steps.  dst_dev: NULL, or per batch the client-chosen shard of every record.
 * dint_shard_submit_host: the same with HOST buffers (pinned recommended): H2D | dispatch | engine | combine | D2H
 * pipelined n_sets deep; returns when every out_host[j] is complete.
 * dint_shard_flags (synchronises): [0] records that overflowed a slab, [1] timed-out waits, since the last call;
 * both must be 0 for the replies to stand. */
typedef struct dint_shard_ctx dint_shard_ctx;
int dint_shard_create(dint_engine *e, uint32_t n_shards, uint32_t rank, uint32_t cap, uint32_t n_sets,
                      const dint_peer_ptrs *inbox_sets, const dint_peer_ptrs *retbox_sets,
                      const dint_peer_ptrs *sig_blocks, uint64_t max_n, dint_shard_ctx **out);
void dint_shard_destroy(dint_shard_ctx *c);
int dint_shard_submit_many(dint_shard_ctx *c, uint32_t k, const void *const *req_dev, const uint8_t *const *dst_dev, uint64_t n,
                           void *const *out_dev, void *cuda_stream);
/* Batches of different sizes in one pipelined sequence (tatp / smallbank rounds): n[j] records in batch j (may differ
 * between ranks) and cap[j] = the slab capacity batch j uses (a multiple of 128, <= the cap of dint_shard_create, THE SAME
 * ON EVERY RANK; NULL or 0 = the full capacity): sized to the batch, the owners do not wade through padding. */
int dint_shard_submit_many_v(dint_shard_ctx *c, uint32_t k, const void *const *req_dev, const uint8_t *const *dst_dev,
                             const uint64_t *n, const uint32_t *cap, void *const *out_dev, void *cuda_stream);
int dint_shard_submit_host(dint_shard_ctx *c, uint32_t k, const void *const *req_host, const uint8_t *const *dst_host, uint64_t n,
                           void *const *out_host);
int dint_shard_flags(dint_shard_ctx *c, uint32_t out[2]);
/* Slab overflow (more records of one source for one owner than `cap`): the source flags it to EVERY owner with the
 * batch, and from that batch on no shard serves anything -- the state stays exactly what it was after the last complete
 * batch.  dint_shard_recover (call on every rank, synchronises): *first_unserved = index, inside the last submit call of
 * k_last batches, of the first batch left unserved (0xffffffff: none); clears the condition.  Serve the unserved
 * batches again in pieces of at most `cap` records per rank -- those cannot overflow.  (dint_cluster_submit does this.) */
int dint_shard_recover(dint_shard_ctx *c, uint32_t k_last, uint32_t *first_unserved);

/*
 * Multi-GPU server in ONE process: SURVEY.md section 8(b)'s `dint_create(kind, cfg, n_gpus)` / `dint_submit(e, req, n,
 * dst_shard, resp)`.  This is what a C/C++ transport front-end binds to serve one key space from all GPUs of a box
 * (the reference runs one `server_shard <id>` process per machine and lets the CLIENT pick the shard:
 * tatp/udp/server_shard.cc:278-320, tatp/caladan/client_udp_shard.cc:187,490-531).
 *   dint_cluster_create: n_gpus shard engines; devices[i] = CUDA ordinal of shard i (NULL: 0..n_gpus-1).  All
 *     ordinals distinct (peer access over NVLink is enabled between them), or all the same (several shards resident
 *     on one GPU: same results, used by the 1-GPU tests).  max_batch = records per shard and round (0 = 262144).
 *     lock_2pl / lock_fasst / store: shard i owns the lock slots / buckets with slot % n_gpus == i -- the slot ONE
 *     reference server would compute, so the cluster answers exactly like ONE server.  tatp / smallbank: shard i
 *     is `server_shard i+1` of an n_gpus-machine deployment (primary key % n_gpus, backups +1 and +2; n_gpus = 1 or
 *     >= 3) and holds only the keys it is a replica of.
 *   dint_cluster_submit: req/resp are HOST arrays of n wire structs; dst_shard[i] (tatp / smallbank: required, the
 *     shard the client would have sent record i to; other kinds: NULL) -- resp[i] answers req[i]; semantics: every
 *     shard sees its records in index order.  Keys skewed beyond the slack of the exchange slabs (all records of
 *     a round hashing to one shard) are handled: the round that does not fit is served again in smaller pieces.
 *     Returns 0, DINT_EPROTO, or an error; never blocks on the network.
 */
typedef struct dint_cluster dint_cluster;
int dint_cluster_create(int kind, const dint_cfg *cfg, int n_gpus, const int *devices, uint64_t max_batch, dint_cluster **out);
int dint_cluster_populate(dint_cluster *c);
int dint_cluster_submit(dint_cluster *c, const void *req, uint64_t n, const uint8_t *dst_shard, void *resp);
dint_engine *dint_cluster_engine(dint_cluster *c, int shard);   /* state inspection of one shard */
uint32_t dint_cluster_size(dint_cluster *c);
uint64_t dint_cluster_overflow_retries(dint_cluster *c);   /* submit calls that met a slab overflow (recovered, see dint_shard_recover) */
void dint_cluster_destroy(dint_cluster *c);
int dint_route_unpermute(dint_engine *e, const void *sorted_dev, const uint32_t *perm_dev, uint64_t n, void *out_dev,
                         void *cuda_stream);
int dint_sync(dint_engine *e);   /* waits for everything submitted on this engine's device */

/* ---- state inspection: parity of the final server state, not only of the wire ------------------ */
/* kvs_get on the device table (store/udp/kvs.h:37-55): 0 = found, 1 = not found. */
int dint_kv_get(dint_engine *e, int table, uint64_t key, void *val, uint32_t *ver);
int64_t dint_kv_count(dint_engine *e, int table);
/* lock_2pl: out = {num_ex, num_sh}; lock_fasst: {lock, ver}; tatp: {lock, 0}; smallbank: {num_ex, num_sh} */
int dint_lock_state(dint_engine *e, int table, uint32_t slot, uint32_t out[2]);
/* slot the reference would compute for a lock id / key (fasthash64 % size) -- for tests */
uint32_t dint_lock_slot(dint_engine *e, int table, uint64_t key_or_lid);
/* copies ring 0 of the commit log (log_ring entries of dint_log_entry_size bytes, laid out as the
 * reference's struct log_entry) and the number of appends so far */
int dint_dump_log(dint_engine *e, void *out, uint64_t *appended);
uint32_t dint_log_entry_size(int kind);

/* Checkpoint / restore of the whole server state of one engine (lock words, versions, counters, KV tables, log ring),
 * device to device.  The reference has no such facility (its state dies with the process); a batched server can take
 * one between two calls at HBM copy speed.  dint_snapshot_restore is asynchronous on cuda_stream and must be ordered
 * between submit calls; it fails if a KV table was rehashed since the snapshot. */
typedef struct dint_snapshot dint_snapshot;
int dint_snapshot_create(dint_engine *e, dint_snapshot **out);
int dint_snapshot_restore(dint_snapshot *s, void *cuda_stream);
void dint_snapshot_destroy(dint_snapshot *s);

/*
 * lock_fasst closed-loop clients ON the GPU (SURVEY.md section 8(f) rank 2).  The reference's clients are Caladan
 * uthreads on other machines (lock_fasst/caladan/client.cc:183-280, trace shape lock_fasst/caladan/trace_init.sh:9-27);
 * here n_clients of those state machines live next to the engine, one request outstanding each per round, so committed
 * txn/s and the abort rate are produced live instead of replayed.  n_keys / zipf_theta / read_pct: the workload family
 * (reference: 24,000,000 ids, uniform (theta 0), read_pct 80).  Same decisions, draw for draw, as the host-side
 * clients of dint_b200/csrc/workloads.cc (seed, client id).
 *   dint_clients_run: `rounds` rounds, asynchronous on cuda_stream.
 *   dint_clients_stats (synchronises): requests served, committed transactions, validation aborts, lock rejects, rounds.
 *   dint_clients_peek (test hook, synchronises): the next round's requests / the last round's replies, n_clients * 9 bytes.
 */
typedef struct dint_clients dint_clients;
int dint_clients_create(dint_engine *e, uint32_t n_clients, uint64_t seed, uint32_t n_keys, double zipf_theta, uint32_t read_pct,
                        dint_clients **out);
int dint_clients_run(dint_clients *c, uint32_t rounds, void *cuda_stream);
int dint_clients_stats(dint_clients *c, uint64_t out[5]);
int dint_clients_peek(dint_clients *c, void *next_req_host, void *last_resp_host);
void dint_clients_destroy(dint_clients *c);

/*
 * TATP and SmallBank closed-loop clients ON the GPU (SURVEY.md section 8(f) rank 2).  The reference's clients are Caladan
 * uthreads on other machines (tatp/caladan/client_udp_shard.cc:177-1184, smallbank/caladan/client_udp_shard.cc:169-1300):
 * each runs one transaction at a time, fanning every protocol step out to the shard servers -- primary key % G, backups
 * +1 and +2, the commit log on all three -- and joining on the replies.  Here n_clients of those state machines live on
 * the device of the shard engines, one thread each, and drive them round after round, so committed txn/s and the abort
 * rate per transaction type come from a live closed loop.  The state machines are the host clients' own
 * (dint_b200/csrc/txn_clients.h, shared with dint_txn_* of libdint_wl.so): same gids (gid0 + i), same fastrand streams,
 * the same requests in the same order, shard by shard.
 *   dint_txn_clients_create: shards[i] = engine of shard i, all tatp or all smallbank, all on one device; n_shards = 1 or
 *     3..8 (primary + 2 distinct backups); with n_shards > 3, engine i must be configured with txn_shards = n_shards and
 *     txn_shard_id = i.  subscribers: kSubscriberNum (tatp, reference 7,000,000) or kAccountNum (smallbank, 24,000,000)
 *     of the key generators -- what the engines populated.  n_clients <= 2^26.  Every client begins its first
 *     transaction and emits its first round (synchronises).
 *   dint_txn_clients_run: `rounds` rounds on cuda_stream.  A round = each shard engine serves the records pending for it
 *     (dint_submit_device; empty shards are skipped), then three client kernels absorb the replies and write the next
 *     round's records into the per-shard buffers.  The host reads the per-shard record counts once per round (the
 *     engines size their launches on the host), so the call returns when the last round's records are written.
 *   dint_txn_clients_stats (synchronises): the dint_txn_stats layout -- requests served, transactions begun, committed,
 *     rounds served, begun by type[7], committed by type[7].
 *   dint_txn_clients_peek (test hook, synchronises): the pending round's requests and destination shards, and the last
 *     round's replies, in client order (each client's records contiguous, in push order), as dint_txn_next / dint_txn_feed
 *     lay them out.  n_out = {pending records, replies of the last round}; NULL buffers: sizes only.
 */
typedef struct dint_txn_clients dint_txn_clients;
int dint_txn_clients_create(dint_engine *const *shards, uint32_t n_shards, uint32_t n_clients, uint32_t gid0,
                            uint32_t subscribers, dint_txn_clients **out);
int dint_txn_clients_run(dint_txn_clients *c, uint32_t rounds, void *cuda_stream);
int dint_txn_clients_stats(dint_txn_clients *c, uint64_t out[18]);
int dint_txn_clients_peek(dint_txn_clients *c, void *next_req_host, uint8_t *next_dst_host, void *last_resp_host,
                          uint64_t n_out[2]);
void dint_txn_clients_destroy(dint_txn_clients *c);

int dint_get_stats(dint_engine *e, dint_stats *s);
void dint_reset_stats(dint_engine *e);
/* per-kernel CUDA-event timing: 0 = off, 1 = every kernel, otherwise a bit mask over
 * {1<<0 k_classify, 1<<1 k_log_scan, 1<<2 k_apply, 1<<3 k_ordered, 1<<4 k_kv_load} */
int dint_profile(dint_engine *e, int enable);
int dint_kernel_times(dint_engine *e, dint_kernel_time *out, int max_entries);  /* returns #entries */
const char *dint_last_error(void);

/* pinned host memory for req/resp buffers */
void *dint_host_alloc(size_t bytes);
void dint_host_free(void *p);

/* hooks for unit tests of the host/device-shared arithmetic (no GPU needed) */
uint64_t dint_test_fasthash64(uint64_t x, int len);      /* len 4 or 8, seed 0xdeadbeef */
uint32_t dint_test_fastmod(uint64_t n, uint32_t d);
/* test hook: the slice sizes dint_submit cuts a call of n requests into (host logic, no GPU needed);
 * returns the number of slices, writes the first `cap` of them */
uint32_t dint_test_host_slices(uint64_t n, uint32_t min_slice, uint32_t max_slice, int ramp_up, uint32_t *out, uint32_t cap);

#ifdef __cplusplus
}
#endif
#endif
