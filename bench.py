#!/usr/bin/env python
"""bench.py -- the driver-facing benchmark (DESIGN.md section 6 "Measurement").

  python bench.py --gpus N --steps K --warmup W            # this repo's GPU engine
  python bench.py ... --dump-outputs DIR                    # also write the replies of the last timed step to DIR
  python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU server (oracle/_ref)

Metric (BASELINE.json): committed txns/sec on lock_fasst.  Workload at N = 1: the reference's own lock_fasst trace
shape (lock_fasst/caladan/trace_init.sh: 24,000,000 lock ids, uniform, 5-10 ids per transaction, write probability
0.2) driven closed-loop by 1,048,576 logical clients through the FaSST protocol of lock_fasst/caladan/client.cc
against a 36,000,000-slot lock table ("REF" in SURVEY.md 8(d)).  One STEP = one batch of 4 client rounds =
4,194,304 wire requests.  W + K steps of the closed loop are recorded (every reply of the recording is compared with
the UNMODIFIED reference server binary fed the same stream); the timed region replays the K recorded steps once,
device resident, from the server state the W warm-up steps left, so that it reproduces the recording bit for bit.
Every step reads a different 37.7 MB trace segment (K segments >> L2).  At N > 1 every rank drives its own 1,048,576
clients and the key space grows with N (36 M slots and 24 M ids PER GPU: constant contention), requests travel to
the owning GPU through the dispatch / engine / combine step over NVLink; the reference's fixed 36 M / 24 M constants
at N > 1, TATP and SmallBank on the reference's shard placement, HOT, store GET, lock_2pl, log_server and the UDP
front-end are reported under "extra".
"""
import argparse
import json
import os

import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the benchmark leaves the tree it runs from as it found it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

CLIENTS = 1 << 20
ROUNDS_PER_STEP = 4
STEP_REQS = CLIENTS * ROUNDS_PER_STEP
TIMED_SECONDS = float(os.environ.get("DINT_BENCH_SECONDS", "1.0"))      # minimum length of the extras' timed regions
# algorithmic bytes per request (SURVEY.md 8(d)): wire in + wire out + state at the reference's field granularity
FASST_BYTES = {4: 22, 5: 26, 6: 22, 7: 22, 8: 30}          # by reply type
STORE_GET_BYTES = 186
WORKLOAD = ("lock_fasst REF: 24,000,000 uniform lock ids, 5-10 ids/txn, p(write)=0.2, closed-loop FaSST clients "
            "(read/acquire/validate/commit), 36,000,000-slot table; 1048576 logical clients, 4 rounds = 4194304 requests per step")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region (NVML, ~2 ms period)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.max_mhz = None

    def run(self):
        try:
            import pynvml as N
            N.nvmlInit()
            h = N.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            while not self.stop_flag:
                try:
                    reasons = N.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    reasons = N.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM), reasons))
                time.sleep(0.002)
        except Exception as ex:       # no NVML: report that rather than inventing numbers
            self.samples.append((None, repr(ex)))

    def stop(self):
        self.stop_flag = True
        self.join(timeout=2)
        sm = sorted(s[0] for s in self.samples if isinstance(s[0], int))
        bits = 0
        for s in self.samples:
            if isinstance(s[1], int):
                bits |= s[1]
        # NVML reason bits: 0x8 hw_slowdown, 0x40 hw_thermal_slowdown, 0x20 sw_thermal_slowdown, 0x4 sw_power_cap
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": [n for b, n in names.items() if bits & b], "samples": len(sm)}


class Background(threading.Thread):
    """fn() on a host thread while the GPU work goes on; .result after join (or an {"unavailable": ...} dict)."""

    def __init__(self, fn):
        super().__init__(daemon=True)
        self.fn, self.result = fn, {"unavailable": "did not finish"}
        self.start()

    def run(self):
        try:
            self.result = self.fn()
        except Exception as ex:
            self.result = {"unavailable": repr(ex)[:300]}

    def get(self, timeout):
        self.join(timeout=timeout)
        return self.result


def masked_equal(kind, got, want):
    """Replies equal up to the value bytes the reference's populate_* leaves indeterminate (tests/golden_util.py)."""
    import golden_util as G
    from dint_b200 import wire
    if kind not in (wire.STORE, wire.TATP):
        return bool(np.array_equal(got, want))
    return G.mismatch(kind, np.asarray(got).reshape(-1), np.asarray(want).reshape(-1)) is None


def reference_check(kind, req, resp, txn_per_req, what, threads=1, timeout=600):
    """The UNMODIFIED reference server (oracle/_ref, replay shim, `server 1`) over the very request stream the GPU
    served: are the GPU's replies the reference's?  The same run is the 1-core handler-only CPU baseline."""
    import oracle_lib as O
    n = req.size // O.MSG_SIZE[kind]
    if O.ref_available(kind):
        t0 = time.time()
        out, st = O.run_ref(kind, req, threads=threads, repeat=1, want_out=True, timeout=timeout)
        eq = masked_equal(kind, resp, out)
        return {"value": st["req_per_s"] * txn_per_req, "unit": "txn/s", "cores": threads, "kind": "reference", "req_per_s": st["req_per_s"],
                "sample": f"{what}: {n} requests once through the oracle/_ref server binary under the replay shim "
                          f"({st['seconds']:.2f} s handler time, {time.time() - t0:.0f} s wall incl. start-up / population)",
                "gpu_replies_equal_reference": eq, "compared_requests": n}
    ora = O.Oracle(kind)
    t0 = time.perf_counter()
    out = ora.process(req)
    dt = time.perf_counter() - t0
    return {"value": n / dt * txn_per_req, "unit": "txn/s", "cores": 1, "kind": "port", "req_per_s": n / dt,
            "sample": f"{what}: {n} requests once through oracle/libdint_oracle.so (the C restatement; oracle/_ref not built)",
            "gpu_replies_equal_reference": bool(np.array_equal(out, resp)), "compared_requests": n}


def udp_as_shipped(O, kind, sample_req, txn_per_req, seconds=4.0):
    """SURVEY 8(d) B1: the unmodified reference server with REAL sockets on loopback (`server 8`, the reference's
    thread count, exp/run_lock_fasst.sh), two syscalls per request as deployed; informational, never the value."""
    try:
        cores = os.cpu_count() or 8
        ct = max(8, min(32, cores // 4))
        r = O.run_ref_udp(kind, sample_req, server_threads=8, client_threads=ct, window=32, seconds=seconds)
        return {"req_per_s": r["req_per_s"], "txn_per_s": r["req_per_s"] * txn_per_req, "server_threads": 8,
                "client_threads": ct, "lost_datagrams": r["lost"], "seconds": r["seconds"],
                "note": "oracle/_ref server, bind address rewritten to 127.0.0.1, replies counted not compared"}
    except Exception as ex:
        return {"unavailable": repr(ex)[:200]}


# ----------------------------------------------------------------------------------------------------
def record_closed_loop(submit, wl, n_steps, msg):
    """Drive the client state machines against `submit(req) -> resp`; per-step request / reply arrays and
    per-step committed-transaction counts."""
    reqs = np.empty((n_steps, STEP_REQS * msg), dtype=np.uint8)
    resps = np.empty_like(reqs)
    committed = []
    rb = CLIENTS * msg
    for s in range(n_steps):
        before = wl.stats()["committed"]
        for r in range(ROUNDS_PER_STEP):
            q = wl.next(reqs[s, r * rb:(r + 1) * rb])
            a = submit(q)
            wl.feed(a)
            resps[s, r * rb:(r + 1) * rb] = a
        committed.append(wl.stats()["committed"] - before)
    return reqs, resps, committed


def fasst_alg_bytes(resps, msg=9):
    cnt = np.bincount(resps.reshape(-1, msg)[:, 0], minlength=9)
    return int(sum(FASST_BYTES[t] * int(cnt[t]) for t in FASST_BYTES)), {str(t): int(cnt[t]) for t in FASST_BYTES}


def dump_replies(out_dir, raw, n_sample=1 << 21):
    """--dump-outputs: lock_fasst reply records `raw` (wire bytes) as one float64 .npy per wire field (exact for every
    u32), 48 MB in all.  Of a longer stream a fixed sample of n_sample records is written, the same in every run, so
    that the outputs of two builds can be compared reply for reply."""
    from dint_b200 import wire
    rec = wire.as_records(wire.FASST, raw)
    if len(rec) > n_sample:
        rec = rec[np.sort(np.random.default_rng(0).choice(len(rec), n_sample, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for f in rec.dtype.names:
        np.save(os.path.join(out_dir, f"lock_fasst_reply_{f}.npy"), rec[f].astype(np.float64))


def run_fasst(args, torch, fam_name, fam, steps, warmup, do_e2e=True, do_ref=True, dump_dir=None):
    """N = 1.  Returns the result dict main() turns into the JSON line."""
    from dint_b200 import Engine, PinnedBuffer, wire
    from dint_b200.workloads import Workload
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    n_steps, msg = steps + warmup, 9
    rq_pin, rs_pin = PinnedBuffer(CLIENTS * msg), PinnedBuffer(CLIENTS * msg)
    # ---- record the closed loop against the GPU engine (host path: one dint_submit per client round) ----
    with Engine(wire.FASST, device=dev.index, chunk=args.chunk) as eng:
        wl = Workload(wire.FASST, n_clients=CLIENTS, seed=20230, **fam)

        def submit(q):
            rq_pin.array[:] = q
            return eng.submit(rq_pin.array, out=rs_pin.array)
        reqs, resps, committed = record_closed_loop(submit, wl, n_steps, msg)
        wl_stats = wl.stats()
    txn_per_req = wl_stats["committed"] / wl_stats["requests"]
    out = {"wl_stats": wl_stats}
    ref_bg = None
    if do_ref:                                   # every recorded reply vs the unmodified reference binary, in the background
        ref_bg = Background(lambda: reference_check(wire.FASST, reqs.reshape(-1), resps.reshape(-1), txn_per_req,
                                                    f"the whole recorded closed loop ({n_steps} steps)"))
    # ---- device-resident replay from a fresh state: the timed region ----
    with Engine(wire.FASST, device=dev.index, chunk=args.chunk) as eng:
        d_req = torch.from_numpy(reqs).to(dev)
        d_out = [torch.empty((STEP_REQS * msg,), dtype=torch.uint8, device=dev) for _ in range(steps)]
        stream = torch.cuda.current_stream(dev)
        for s in range(warmup):
            eng.submit_tensor(d_req[s], d_out[0])
        torch.cuda.synchronize(dev)
        ok = bool((d_out[0].cpu().numpy() == resps[warmup - 1]).all()) if warmup else True
        snap = eng.snapshot()                    # the state the timed steps start from
        eng.reset_stats()
        eng.profile(Engine.PROF_APPLY)           # events around the dominant kernel only (all-kernel profiling costs ~20 %)
        sampler = ClockSampler(dev.index)
        sampler.start()
        time.sleep(0.01)
        torch.cuda.synchronize(dev)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record(stream)
        for s in range(steps):
            eng.submit_tensor(d_req[warmup + s], d_out[s])
        ev[1].record(stream)
        torch.cuda.synchronize(dev)
        ms = ev[0].elapsed_time(ev[1])
        clocks = sampler.stop()
        eng.profile(False)
        if dump_dir is not None:
            dump_replies(dump_dir, d_out[steps - 1].cpu().numpy())
        kt, st = eng.kernel_times(), eng.stats()
        n_bad = sum(0 if bool((d_out[s].cpu().numpy() == resps[warmup + s]).all()) else 1 for s in range(steps))
        out.update(ms=ms, kernel_times=kt, stats=st, clocks=clocks, parity_replay=(ok and n_bad == 0))
        # a fully profiled cycle (not the timed one) for the per-kernel breakdown
        eng.reset_stats()
        eng.profile(True)
        eng.restore(snap, stream.cuda_stream)
        for s in range(steps):
            eng.submit_tensor(d_req[warmup + s], d_out[s])
        torch.cuda.synchronize(dev)
        eng.profile(False)
        out["all_kernel_times"] = eng.kernel_times()
        eng.free_snapshot(snap)
        del d_req, d_out
    out.update(committed=sum(committed[warmup:]), requests=steps * STEP_REQS, steps_timed=steps)
    alg, mix = fasst_alg_bytes(resps[warmup:])
    out.update(alg_bytes=alg, reply_mix=mix)
    # ---- end to end through the host-facing C ABI call (pinned host buffers, H2D + D2H inside) ----
    if do_e2e:
        with Engine(wire.FASST, device=dev.index, chunk=args.chunk) as eng:
            host_in = [PinnedBuffer(STEP_REQS * msg) for _ in range(steps)]
            host_out = PinnedBuffer(STEP_REQS * msg)
            for s in range(warmup):
                host_in[0].array[:] = reqs[s]
                eng.submit(host_in[0].array, out=host_out.array)
            for s in range(steps):
                host_in[s].array[:] = reqs[warmup + s]              # staging into pinned memory: not timed
            torch.cuda.synchronize(dev)
            t_e2e = 0.0
            for s in range(steps):
                t0 = time.perf_counter()
                eng.submit(host_in[s].array, out=host_out.array)   # timed: H2D + kernels + D2H, returns when resp is complete
                t_e2e += time.perf_counter() - t0
            out.update(e2e_s=t_e2e, e2e_steps=steps, e2e_parity=bool((host_out.array == resps[n_steps - 1]).all()),
                       e2e_committed=sum(committed[warmup:]), e2e_requests=STEP_REQS * steps)
    if ref_bg is not None:
        out["cpu_baseline"] = ref_bg.get(timeout=600)
    out["first_step"] = (reqs[0], resps[0], txn_per_req)
    return out


# ---------------------------------------------------------------------------------------------------- N > 1
def gather_prefix(torch, dist, rank, world, arr):
    """uint8 numpy array of equal size on every rank -> list of all ranks' arrays on rank 0 (NCCL gather)."""
    t = torch.from_numpy(np.ascontiguousarray(arr)).cuda()
    parts = [torch.empty_like(t) for _ in range(world)] if rank == 0 else None
    dist.gather(t, parts, dst=0)
    return [p.cpu().numpy() for p in parts] if rank == 0 else None


def run_fasst_sharded(args, torch, dist, rank, world, scaled, steps, warmup, do_e2e=True, dump_dir=None):
    """Every rank drives its own 1,048,576 clients; requests are routed to the owning shard through the library's
    dispatch / engine / combine step over NVLink peer memory (dint_shard_submit_many).  scaled=True: the key space
    grows with the GPU count (36 M slots and 24 M ids per GPU: the per-GPU state and the contention stay what they are
    at N = 1); scaled=False: the reference's constants (every added GPU adds clients to the SAME 24 M ids)."""
    import oracle_lib as O
    from dint_b200 import wire
    from dint_b200.shard import ShardedEngine
    from dint_b200.workloads import Workload
    dev = torch.device("cuda", torch.cuda.current_device())
    n_steps, msg = steps + warmup, 9
    big = args.chunk + args.chunk // 2                   # one round + slab padding fits one engine chunk
    slots = 36_000_000 * (world if scaled else 1)
    ids = 24_000_000 * (world if scaled else 1)
    mk = lambda: ShardedEngine(wire.FASST, chunk=big, strict=False, use_p2p=True, p2p_max_n=CLIENTS, lock_slots=slots)
    se = mk()
    wl = Workload(wire.FASST, n_clients=CLIENTS, seed=20230 + rank, n_keys=ids, zipf_theta=0.0)
    reqs, resps, committed = record_closed_loop(se.submit, wl, n_steps, msg)
    wl_stats = wl.stats()
    flags_rec = se.check_p2p()
    se.close()
    # ---- oracle parity of the sharded run: ONE sequential server fed the rank-major concatenation, round by round ----
    P = min(n_steps, warmup + 1)                         # a prefix (it must start from the initial state)
    g_req = gather_prefix(torch, dist, rank, world, reqs[:P])
    g_resp = gather_prefix(torch, dist, rank, world, resps[:P])
    par_bg = None
    if rank == 0:
        def check():
            rb = CLIENTS * msg
            seq_req = np.concatenate([g_req[r][s, k * rb:(k + 1) * rb] for s in range(P) for k in range(ROUNDS_PER_STEP) for r in range(world)])
            seq_got = np.concatenate([g_resp[r][s, k * rb:(k + 1) * rb] for s in range(P) for k in range(ROUNDS_PER_STEP) for r in range(world)])
            n = seq_req.size // msg
            if not scaled and O.ref_available(wire.FASST):
                want, st = O.run_ref(wire.FASST, seq_req, threads=1, repeat=1, want_out=True, timeout=900)
                how = "the unmodified reference server binary (oracle/_ref, `server 1`)"
            else:
                t0 = time.perf_counter()
                want = O.Oracle(wire.FASST, lock_slots=slots).process(seq_req)
                how = (f"the oracle restatement with kLockHashSize = {slots} (the reference binary's table size is a constexpr 36,000,000)"
                       if scaled else "the oracle restatement")
            return {"gpu_replies_equal_reference": bool(np.array_equal(want, seq_got)), "compared_requests": int(n), "checker": how,
                    "order": "rank-major concatenation of every client round (SURVEY.md 8(e)): the first %d steps of all %d ranks" % (P, world)}
        par_bg = Background(check)
    # ---- timed replay from fresh shards ----
    se = mk()
    d_req = torch.from_numpy(reqs).to(dev)
    rb = CLIENTS * msg
    stream = torch.cuda.current_stream(dev)
    last = [None] * steps

    def step(s_, slot):
        last[slot] = se.submit_many([d_req[s_][r * rb:(r + 1) * rb] for r in range(ROUNDS_PER_STEP)])

    for s in range(warmup):
        step(s, 0)
    torch.cuda.synchronize(dev)
    se.engine.reset_stats()
    se.engine.profile(se.engine.PROF_APPLY)
    sampler = ClockSampler(dev.index)
    sampler.start()
    dist.barrier()
    torch.cuda.synchronize(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record(stream)
    for s in range(steps):
        step(warmup + s, s)
    ev[1].record(stream)
    torch.cuda.synchronize(dev)
    dist.barrier()
    ms = ev[0].elapsed_time(ev[1])
    clocks = sampler.stop()
    se.engine.profile(False)
    if dump_dir is not None and rank == 0:
        dump_replies(dump_dir, torch.cat(last[steps - 1]).cpu().numpy())
    n_bad = 0
    for s in range(steps):
        got = torch.cat(last[s]).cpu().numpy()
        n_bad += 0 if bool((got == resps[warmup + s]).all()) else 1
    ok = n_bad == 0 and se.check_p2p() == (0, 0) and flags_rec == (0, 0)
    out = dict(ms=ms, kernel_times=se.engine.kernel_times(), stats=se.engine.stats(), clocks=clocks, parity_replay=ok,
               committed=sum(committed[warmup:]), requests=steps * STEP_REQS, steps_timed=steps, wl_stats=wl_stats)
    alg, mix = fasst_alg_bytes(resps[warmup:])
    out.update(alg_bytes=alg, reply_mix=mix)
    se.close()
    del d_req
    # ---- end to end: pinned host -> H2D | dispatch | engine | combine | D2H (dint_shard_submit_host), per step ----
    if do_e2e:
        se = mk()
        pin_in = [torch.from_numpy(reqs[warmup + s].copy()).pin_memory() for s in range(steps)]
        pin_w = [torch.from_numpy(reqs[s].copy()).pin_memory() for s in range(warmup)]
        pin_out = torch.empty(STEP_REQS * msg, dtype=torch.uint8).pin_memory()
        rounds = lambda p: [p[r * rb:(r + 1) * rb] for r in range(ROUNDS_PER_STEP)]
        for s in range(warmup):
            se.submit_many_host(rounds(pin_w[s]), rounds(pin_out))
        t_e2e = 0.0
        for s in range(steps):
            dist.barrier()
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            se.submit_many_host(rounds(pin_in[s]), rounds(pin_out))
            t_e2e += time.perf_counter() - t0
        ok2 = bool((pin_out.numpy() == resps[n_steps - 1]).all()) and se.check_p2p() == (0, 0)
        out.update(e2e_s=t_e2e, e2e_steps=steps, e2e_parity=ok2, e2e_committed=sum(committed[warmup:]), e2e_requests=STEP_REQS * steps)
        se.close()
    if par_bg is not None:
        out["oracle_parity"] = par_bg.get(timeout=900)
    out["first_step"] = (reqs[0], resps[0], wl_stats["committed"] / wl_stats["requests"])
    return out


def run_txn_sharded(args, torch, dist, rank, world, kind_name, rounds_timed=12, rounds_warm=8, clients=1 << 19):
    """BASELINE.json configs[3] / [4]: the TATP mix and SmallBank with hot accounts on N >= 3 GPUs, the reference's
    placement generalised from 3 to N shard servers (primary key % N, backups +1 / +2, log on the three replica
    holders: tatp/caladan/client_udp_shard.cc:187,490-531, smallbank/caladan/client_udp_shard.cc:441-577).  Every rank
    IS one shard server (it holds only the keys it is a replica of) and also receives the requests of its own
    `clients` closed-loop clients, which name the destination shard of every record; the exchange step delivers them."""
    from dint_b200 import wire
    from dint_b200.shard import ShardedEngine
    from dint_b200.txn_workloads import TxnWorkload
    dev = torch.device("cuda", torch.cuda.current_device())
    kind = wire.TATP if kind_name == "tatp" else wire.SMALLBANK
    subscribers = 7_000_000 if kind == wire.TATP else 24_000_000
    msg = wire.MSG_SIZE[kind]
    wl = TxnWorkload(kind, n_clients=clients, n_shards=world, subscribers=subscribers, gid0=rank * clients)
    max_n = int(wl._dst.size)
    big = 1 << 22
    t0 = time.time()
    mk = lambda: ShardedEngine(kind, by_dst=True, chunk=big, strict=False, use_p2p=True, p2p_max_n=max_n, slab_slack=2.0)
    se = mk()
    se.populate()
    t_pop = time.time() - t0
    rec, committed = [], []
    mine_req, mine_resp = [], []                          # what rank 0's shard is sent by this rank, per round
    for r in range(rounds_warm + rounds_timed):
        before = wl.stats()["committed"]
        rq, dst = wl.next()
        rs = se.submit(rq, dst)
        wl.feed(rs)
        rec.append((rq.copy(), dst.copy(), np.array(rs, copy=True)))
        committed.append(wl.stats()["committed"] - before)
        sel = dst == 0
        mine_req.append(np.ascontiguousarray(rq.reshape(-1, msg)[sel]).reshape(-1))
        mine_resp.append(np.ascontiguousarray(np.asarray(rs).reshape(-1, msg)[sel]).reshape(-1))
    st = wl.stats()
    flags_rec = se.check_p2p()
    se.close()
    # shard 0's whole input stream (round by round, source-rank-major) and what it answered, to rank 0
    payload = [None] * world if rank == 0 else None
    dist.gather_object((mine_req, mine_resp), payload, dst=0)
    bg = None
    if rank == 0:
        n_rounds = rounds_warm + rounds_timed
        s_req = np.concatenate([payload[r][0][k] for k in range(n_rounds) for r in range(world)])
        s_resp = np.concatenate([payload[r][1][k] for k in range(n_rounds) for r in range(world)])
        bg = Background(lambda: reference_check(kind, s_req, s_resp, st["committed"] / max(1, st["requests"]),
                                                f"shard server 0's whole input stream of the recorded closed loop ({n_rounds} rounds, all {world} ranks' clients)", timeout=900))
    # timed: device-resident replay from freshly populated shards; the state is restored per cycle OUTSIDE the timed region
    se = mk()
    se.populate()
    d = [(torch.from_numpy(q).to(dev), torch.from_numpy(dd).to(dev)) for q, dd, _ in rec]
    stream = torch.cuda.current_stream(dev)
    for r in range(rounds_warm):
        se.submit_many([d[r][0]], dsts=[d[r][1]])
    torch.cuda.synchronize(dev)
    snap = se.engine.snapshot()
    total_ms, cycles, outs = 0.0, 0, None
    go = torch.ones(1, device=dev)
    while True:
        se.engine.restore(snap, stream.cuda_stream)
        torch.cuda.synchronize(dev)
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        outs = [se.submit_many([d[r][0]], dsts=[d[r][1]])[0] for r in range(rounds_warm, rounds_warm + rounds_timed)]
        e1.record(stream)
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms += float(t[0])
        cycles += 1
        if total_ms >= TIMED_SECONDS * 1e3 or cycles >= 400:
            break
    ok = all(bool((outs[i].cpu().numpy() == rec[rounds_warm + i][2]).all()) for i in range(rounds_timed))
    ok = ok and se.check_p2p() == (0, 0) and flags_rec == (0, 0)
    est = se.engine.stats()
    se.engine.free_snapshot(snap)
    se.close()
    w = torch.tensor([sum(committed[rounds_warm:]), sum(x[1].size for x in rec[rounds_warm:]), st["committed"], st["txns"], st["requests"],
                      est["kernel_launches"], est["conflicted"], 1.0 if ok else 0.0, est["requests"]], device=dev, dtype=torch.float64)
    dist.all_reduce(w, op=dist.ReduceOp.SUM)
    if rank != 0:
        return None
    tc, tr = float(w[0]) * cycles, float(w[1]) * cycles
    res = {"workload": f"{kind_name} mix, {clients} closed-loop clients per GPU, {world} shard servers (one per GPU, reference placement generalised to "
                       f"{world} shards), {subscribers} {'subscribers' if kind == wire.TATP else 'accounts'}; {rounds_timed} protocol rounds per cycle, "
                       f"{cycles} cycles timed (device-resident replay of the recorded closed loop, state restored between cycles)",
           "txn_per_s": tc / (total_ms * 1e-3), "requests_per_s": tr / (total_ms * 1e-3), "abort_rate": 1.0 - float(w[2]) / max(1.0, float(w[3])),
           "requests_per_txn": float(w[4]) / max(1.0, float(w[3])), "timed_region_s": total_ms * 1e-3,
           "replies_bit_exact_vs_closed_loop_recording": float(w[7]) == world, "gpu_launches": int(w[5]),
           "conflicted_fraction_of_records_served_incl_padding": float(w[6]) / max(1.0, float(w[8])), "populate_s": round(t_pop, 1)}
    res["cpu_baseline"] = bg.get(timeout=900)
    return res


# ---------------------------------------------------------------------------------------------------- extras (N = 1)
def run_closed_loop_extra(args, torch, rank, kind_name, rounds=16, warm=24):
    """lock_2pl / log_server side measurement: the reference's closed-loop clients (workloads.cc) recorded against
    the GPU engine through the host path, then replayed device-resident and timed; replies must be bit-exact."""
    from dint_b200 import Engine, wire
    from dint_b200.workloads import Workload, REF
    kind = {"lock_2pl": wire.LOCK2PL, "log_server": wire.LOG}[kind_name]
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    fam = REF if kind == wire.LOCK2PL else {}
    wl = Workload(kind, n_clients=CLIENTS, seed=20230 + rank, **fam)
    if kind == wire.LOG:
        warm = 3                                          # no protocol state to warm up
    reqs, resps, committed = [], [], []
    with Engine(kind, device=dev.index, chunk=args.chunk) as eng:
        for _ in range(warm + rounds):
            before = wl.stats()["committed"]
            q = wl.next()
            a = eng.submit(q)
            wl.feed(a)
            reqs.append(q.copy()); resps.append(a.copy())
            committed.append(wl.stats()["committed"] - before)   # transactions whose last reply arrived this round
    st = wl.stats()
    n_chk = min(len(reqs), 8 if kind == wire.LOG else warm + rounds)
    bg = Background(lambda: reference_check(kind, np.concatenate(reqs[:n_chk]), np.concatenate(resps[:n_chk]), st["committed"] / max(1, st["requests"]),
                                            f"the first {n_chk} rounds of the recorded closed loop"))
    with Engine(kind, device=dev.index, chunk=args.chunk) as eng:
        d_req = [torch.from_numpy(r).to(dev) for r in reqs]
        d_out = [torch.empty_like(d_req[0]) for _ in range(rounds)]
        for r in range(warm):
            eng.submit_tensor(d_req[r], d_out[0])
        torch.cuda.synchronize(dev)
        snap = eng.snapshot()
        stream = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for r in range(rounds):
            eng.submit_tensor(d_req[warm + r], d_out[r])
        e1.record()
        torch.cuda.synchronize(dev)
        cycles = max(1, int(np.ceil(min(TIMED_SECONDS, 0.5) * 1e3 / max(e0.elapsed_time(e1), 1e-3))))
        eng.reset_stats()
        e0.record()
        for _ in range(cycles):
            eng.restore(snap, stream.cuda_stream)
            for r in range(rounds):
                eng.submit_tensor(d_req[warm + r], d_out[r])
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        ok = all(bool((d_out[r].cpu().numpy() == resps[warm + r]).all()) for r in range(rounds))
        est = eng.stats()
        eng.free_snapshot(snap)
    n_req = rounds * CLIENTS * cycles
    res = {"workload": ("lock_2pl REF: 24,000,000 uniform lock ids, 5-10 ids/txn, p(exclusive)=0.2, closed-loop 2PL clients "
                        "(acquire in id order, release in reverse, retry after a reject)" if kind == wire.LOCK2PL else
                        "log_server: key uniform [0, 7,009,999], ver [0,127], 40 random bytes per append") +
                       f"; {CLIENTS} logical clients, {rounds} rounds x {cycles} cycles timed (device-resident replay of the recorded closed loop)",
           "requests_per_s": n_req / (ms * 1e-3), "timed_region_s": ms * 1e-3, "replies_bit_exact_vs_closed_loop_recording": ok,
           "gpu_launches": est["kernel_launches"], "conflicted_fraction": est["conflicted"] / max(1, est["requests"])}
    if kind == wire.LOCK2PL:
        res["txn_per_s"] = sum(committed[warm:]) * cycles / (ms * 1e-3)
        res["requests_per_txn"] = rounds * CLIENTS / max(1, sum(committed[warm:]))
        res["lock_rejects"] = st["lock_rejects"]
    res["cpu_baseline"] = bg.get(timeout=300)
    return res


def run_gpu_clients(args, torch, fam, warm_rounds=48):
    """SURVEY 8(f) rank 2: the closed-loop clients themselves on the GPU (dint_clients_*): no trace, no host in the
    loop -- committed txn/s and abort rates are produced live for as long as the timed region lasts.  The client
    kernel shares the GPU with the server, so this is lower than the replay of a recorded trace (which times the
    server alone, as the reference's server throughput is measured with clients on other machines)."""
    from dint_b200 import Engine, GpuClients, wire
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    with Engine(wire.FASST, device=dev.index, chunk=args.chunk) as eng:
        gc = GpuClients(eng, CLIENTS, seed=20230, **fam)
        stream = torch.cuda.current_stream(dev)
        gc.run(warm_rounds, stream.cuda_stream)
        torch.cuda.synchronize(dev)
        s0 = gc.stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        gc.run(64, stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        rounds = max(64, int(np.ceil(min(TIMED_SECONDS, 0.5) * 1e3 / (e0.elapsed_time(e1) / 64))))
        s0 = gc.stats()
        e0.record(stream)
        gc.run(rounds, stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        s1 = gc.stats()
        gc.close()
    d = {k: s1[k] - s0[k] for k in s1}
    return {"workload": f"{CLIENTS} lock_fasst closed-loop clients RESIDENT ON THE GPU (one kernel per round absorbs the replies and emits the next "
                        f"requests; same state machine and draws as the host clients: tests/test_gpu_clients.py), {rounds} rounds timed",
            "txn_per_s": d["committed"] / (ms * 1e-3), "requests_per_s": d["requests"] / (ms * 1e-3), "timed_region_s": ms * 1e-3,
            "committed_per_request": d["committed"] / max(1, d["requests"]),
            "abort_stats": {k: d[k] for k in ("committed", "validation_aborts", "lock_rejects")}, "us_per_round": ms * 1e3 / rounds}


def udp_verify(port, req, window=64):
    """One client socket, windows of `window` datagrams (loopback keeps their order) against a FRESH lock_fasst server: the
    replies must be ONE sequential reference server's (the oracle restatement).  Returns True / False / a reason."""
    import socket
    import oracle_lib as O
    try:
        rec = np.ascontiguousarray(req).view(np.uint8).reshape(-1, 9)
        want = O.Oracle(1).process(req).reshape(-1, 9)
        got = np.empty_like(rec)
        with socket.socket(socket.AF_INET, socket.SOCK_DGRAM) as c:
            c.settimeout(5.0)
            c.connect(("127.0.0.1", port))
            for lo in range(0, len(rec), window):
                hi = min(lo + window, len(rec))
                for i in range(lo, hi):
                    c.send(rec[i].tobytes())
                for i in range(lo, hi):
                    got[i] = np.frombuffer(c.recv(64), dtype=np.uint8)
        return bool(np.array_equal(got, want))
    except Exception as ex:
        return "not checked: " + repr(ex)[:120]


def run_udp_front_end(seconds=4.0):
    """dint_udp_server (the reference's UDP server shape over the C ABI, dint_b200/csrc/udp_server.cc) with the GPU
    engine behind it, driven over loopback by the same multi-socket replayer that times the unmodified reference
    server for cpu_baseline.udp_as_shipped.  Runs in child processes with deadlines."""
    import signal
    import socket
    import tempfile
    from dint_b200 import _build, wire
    blast = os.path.join(ROOT, "oracle", "_ref", "udp_blast")
    if not (os.path.exists(_build.UDP_SERVER) and os.path.exists(blast)):
        return {"unavailable": "dint_udp_server or oracle/_ref/udp_blast not built"}
    n = 1 << 20
    rng = np.random.default_rng(20230)
    rec = np.zeros(n, dtype=wire.MSG_DTYPE[wire.FASST])
    rec["type"] = rng.choice(4, size=n, p=(0.6, 0.15, 0.05, 0.2))          # read / acquire / abort / commit mix of the REF trace
    rec["lid"] = rng.integers(0, 24_000_000, size=n)
    with socket.socket(socket.AF_INET, socket.SOCK_DGRAM) as s0:
        s0.bind(("127.0.0.1", 0))
        port = s0.getsockname()[1]
    cores = os.cpu_count() or 8
    n_sock = 8                                    # the reference's own thread count (exp/run_lock_fasst.sh: `server 8`)
    with tempfile.TemporaryDirectory() as td:
        tp = os.path.join(td, "trace.bin")
        wire.as_bytes(rec).tofile(tp)
        srv = subprocess.Popen([_build.UDP_SERVER, "lock_fasst", "--bind", "127.0.0.1", "--port", str(port), "--sockets", str(n_sock)],
                               stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, start_new_session=True)
        try:
            t0 = time.time()
            os.set_blocking(srv.stderr.fileno(), False)
            banner = b""
            while b"sockets, batches" not in banner:                         # printed once the engine exists and the sockets are bound
                if srv.poll() is not None or time.time() - t0 > 90:
                    return {"unavailable": "server did not come up: " + banner.decode(errors="replace")[-200:]}
                time.sleep(0.2)
                try:
                    banner += srv.stderr.read() or b""
                except (BlockingIOError, TypeError):
                    pass
            exact = udp_verify(port, wire.as_bytes(rec[:8192]))       # on the fresh server, before the replayer mutates its state
            ct = max(8, min(32, cores // 4))
            r = subprocess.run([blast, tp, "9", str(port), str(ct), "64", str(seconds)], capture_output=True, timeout=seconds + 60)
            out = json.loads(r.stdout.decode().strip().splitlines()[-1])
        finally:
            try:
                os.killpg(srv.pid, signal.SIGTERM)          # exactly the process group we started
            except ProcessLookupError:
                pass
            try:
                srv.wait(timeout=20)
            except subprocess.TimeoutExpired:
                os.killpg(srv.pid, signal.SIGKILL)
                srv.wait()
    return {"req_per_s": out["req_per_s"], "lost_datagrams": out["lost"], "server_sockets": n_sock, "client_threads": out["client_threads"],
            "window": out["window"], "seconds": out["seconds"], "first_8192_replies_equal_oracle": exact,
            "note": "loopback UDP, one datagram per request, recvmmsg/sendmmsg front-end + dint_submit; same replayer as "
                    "cpu_baseline.udp_as_shipped (which serves the same trace with the unmodified reference server).  Both are bound by the "
                    "kernel's UDP path (two syscalls' worth of socket work per datagram on both ends), not by the handler; the first 8192 replies "
                    "of the fresh server are compared with the oracle here, every server kind by "
                    "tests/test_gpu_parity.py::test_udp_front_end_serves_the_wire_protocol_bit_exact"}


def run_store_get(args, torch, rank, steps, warmup):
    """The store lookup path: 100 % kRead, NURand keys over the reference's 24 M-key population."""
    from dint_b200 import Engine, wire
    from dint_b200.workloads import Workload
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    n = 1 << 22
    wl = Workload(wire.STORE, n_clients=n, seed=1 + rank)
    first = wl.next().copy()
    with Engine(wire.STORE, device=dev.index, chunk=args.chunk, populate=True) as eng:
        bufs = [torch.from_numpy(first).to(dev)] + [torch.from_numpy(wl.next().copy()).to(dev) for _ in range(steps + warmup - 1)]   # open-loop
        d_out = torch.empty_like(bufs[0])
        eng.submit_tensor(bufs[0], d_out)
        torch.cuda.synchronize(dev)
        first_resp = d_out.cpu().numpy().copy()
        bg = None
        if rank == 0:                                      # BASELINE.json configs[0]: the reference store server on the host CPU
            bg = Background(lambda: reference_check(wire.STORE, first, first_resp, 1.0, "the first step of the GET trace", timeout=300))
        for s in range(1, warmup):
            eng.submit_tensor(bufs[s], d_out)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(warmup, warmup + steps):
            eng.submit_tensor(bufs[s], d_out)
        e1.record()
        torch.cuda.synchronize(dev)
        cycles = max(1, int(np.ceil(min(TIMED_SECONDS, 0.5) * 1e3 / max(e0.elapsed_time(e1), 1e-3))))   # reads only: the state never changes
        eng.reset_stats()
        eng.profile(Engine.PROF_APPLY)
        e0.record()
        for _ in range(cycles):
            for s in range(warmup, warmup + steps):
                eng.submit_tensor(bufs[s], d_out)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        eng.profile(False)
        kt = eng.kernel_times()
        hits = int((d_out.view(-1, 53)[:, 0] == 3).sum().item())
    peak, how = peaks()
    l, t = kt["k_apply"]
    ach = STORE_GET_BYTES * n * steps * cycles / l / (t / l * 1e-3) / 1e9
    ach170 = ach * 170.0 / STORE_GET_BYTES
    res = {"workload": f"store kRead, NURand keys, 24,000,000-key table (reference population), device-resident, {steps} distinct 222 MB steps x {cycles} cycles",
           "get_per_s": n * steps * cycles / (ms * 1e-3), "timed_region_s": ms * 1e-3, "hit_fraction_last_step": hits / n,
           "roofline": {"kernel": "k_apply<store>", "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                        "frac": ach / peak, "peak_source": how, "avg_launch_us": t / l * 1e3,
                        "algorithmic_bytes_per_request": STORE_GET_BYTES,
                        "frac_with_this_engines_64B_entry": ach170 / peak,
                        "note": "186 B/GET is SURVEY 8(d)'s figure (reference 4-key entry); with this engine's one-key 64-byte entry the "
                                "minimum is 53 + 53 + 64 = 170 B/GET",
                        "traffic": load_static_traffic("k_apply<store>")}}
    if bg is not None:
        res["cpu_baseline"] = bg.get(timeout=400)
    return res


def run_txn(args, torch, rank, kind_name, rounds_timed=12, rounds_warm=8, clients=1 << 20):
    """Full transaction mixes driven by the reference's closed-loop client state machines
    (dint_b200/csrc/txn_workloads.cc) against THREE shard servers (primary key % 3 + 2 backups + log on all
    three, as {tatp,smallbank}/caladan/client_udp_shard.cc) -- here three engines resident on one GPU, each
    holding the reference's full population (tatp: 7,000,000 subscribers, mix 35/35/10/2/14/2/2; smallbank:
    24,000,000 accounts, 4 % hot accounts drawing 90 % of the transactions, mix 15/15/15/25/15/15)."""
    from dint_b200 import Engine, wire
    from dint_b200.txn_workloads import TxnWorkload, Cluster, partition_by_shard
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    kind = wire.TATP if kind_name == "tatp" else wire.SMALLBANK
    subscribers = 7_000_000 if kind == wire.TATP else 24_000_000
    msg, G = wire.MSG_SIZE[kind], 3
    t0 = time.time()

    def make():
        return [Engine(kind, device=dev.index, chunk=args.chunk, populate=True) for _ in range(G)]

    engs = make()
    t_pop = time.time() - t0
    wl = TxnWorkload(kind, n_clients=clients, n_shards=G, subscribers=subscribers, gid0=rank * clients)
    cl = Cluster([e.submit for e in engs], msg)
    rec, committed, nreq = [], [], []
    for r in range(rounds_warm + rounds_timed):
        before = wl.stats()["committed"]
        rq, dst = wl.next()
        rs = cl.submit(rq, dst)
        wl.feed(rs)
        parts = partition_by_shard(rq, dst, G, msg)[2]
        rparts = partition_by_shard(rs, dst, G, msg)[2]
        rec.append((parts, rparts))
        committed.append(wl.stats()["committed"] - before)
        nreq.append(int(dst.size))
    st = wl.stats()
    for e in engs:
        e.close()
    bg = None
    if rank == 0:                                          # shard 0's request stream from the start of the recording
        nchk = rounds_warm + 4
        s_req = np.concatenate([np.ascontiguousarray(parts[0]).reshape(-1) for parts, _ in rec[:nchk]])
        s_resp = np.concatenate([np.ascontiguousarray(rp[0]).reshape(-1) for _, rp in rec[:nchk]])
        bg = Background(lambda: reference_check(kind, s_req, s_resp, st["committed"] / max(1, st["requests"]),
                                                f"shard 0's first {nchk} rounds of the recorded closed loop", timeout=600))
    # device-resident replay from freshly populated shards
    engs = make()
    d = [[torch.from_numpy(np.ascontiguousarray(p)).to(dev) for p in parts] for parts, _ in rec]
    outs = [[torch.empty_like(x) for x in row] for row in d]
    for r in range(rounds_warm):
        for s_ in range(G):
            if d[r][s_].numel():
                engs[s_].submit_tensor(d[r][s_], outs[r][s_])
    torch.cuda.synchronize(dev)
    snaps = [e.snapshot() for e in engs]
    stream = torch.cuda.current_stream(dev)
    for e in engs:
        e.reset_stats()
    total_ms, cycles = 0.0, 0
    while total_ms < min(TIMED_SECONDS, 0.5) * 1e3 and cycles < 200:
        for e, sn in zip(engs, snaps):
            e.restore(sn, stream.cuda_stream)                  # outside the timed region (GBs of tables)
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for r in range(rounds_warm, rounds_warm + rounds_timed):
            for s_ in range(G):
                if d[r][s_].numel():
                    engs[s_].submit_tensor(d[r][s_], outs[r][s_])
        e1.record()
        torch.cuda.synchronize(dev)
        total_ms += e0.elapsed_time(e1)
        cycles += 1
    ok = all(bool((outs[r][s_].cpu().numpy() == rec[r][1][s_]).all()) for r in range(rounds_warm, rounds_warm + rounds_timed) for s_ in range(G))
    launches = sum(e.stats()["kernel_launches"] for e in engs)
    conflicted = sum(e.stats()["conflicted"] for e in engs)
    for e, sn in zip(engs, snaps):
        e.free_snapshot(sn)
        e.close()
    tc = sum(committed[rounds_warm:]) * cycles
    tr = sum(nreq[rounds_warm:]) * cycles
    res = {"workload": f"{kind_name} mix, {clients} closed-loop clients, 3 shard servers x {subscribers} "
                       f"{'subscribers' if kind == wire.TATP else 'accounts'} on one GPU, "
                       f"{rounds_timed} protocol rounds x {cycles} cycles timed (device-resident replay of the recorded closed-loop trace, state restored between cycles)",
           "abort_rate": 1.0 - st["committed"] / max(1, st["txns"]), "timed_region_s": total_ms * 1e-3,
           "txn_per_s": tc / (total_ms * 1e-3), "requests_per_s": tr / (total_ms * 1e-3), "requests_per_txn": st["requests"] / max(1, st["txns"]),
           "commit_rate_by_type": {k: round(v[1] / max(1, v[0]), 4) for k, v in st["by_type"].items()},
           "replies_bit_exact_vs_closed_loop_recording": ok, "gpu_launches": launches, "conflicted_fraction": conflicted / max(1, tr),
           "populate_s_per_3_shards": round(t_pop, 1)}
    if bg is not None:
        res["cpu_baseline"] = bg.get(timeout=600)
    return res


class Watchdog:
    """If the side measurements (which, at N > 1, are collective and cannot be run in a child process with a timeout) do not
    finish within `seconds`, rank 0 prints the headline line it already has and every rank exits: a stuck extra must not
    cost the headline."""

    def __init__(self, seconds, rank, fallback_line, out_fd):
        def fire():
            if rank == 0 and fallback_line is not None:
                os.write(out_fd, (json.dumps(fallback_line) + "\n").encode())
            os._exit(0)
        self.t = threading.Timer(seconds, fire)
        self.t.daemon = True
        self.t.start()

    def cancel(self):
        self.t.cancel()


def load_static_traffic(name):
    """dram__bytes_read + dram__bytes_write per launch of the named kernel from the committed ncu capture (profiles/):
    a STATIC figure measured once per round, not by this run."""
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(tp):
        return None
    return json.load(open(tp)).get(name)


# ----------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="dint_b200", choices=["dint_b200", "reference"])
    ap.add_argument("--chunk", type=int, default=1 << 20)
    ap.add_argument("--no-extra", action="store_true", help="skip the side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the replies of the last timed step to DIR/*.npy (float64; at N > 1 rank 0's)")
    ap.add_argument("--extra-only", default=None, help=argparse.SUPPRESS)     # child-process mode for a side measurement
    args = ap.parse_args()
    if args.extra_only:
        import torch
        print(json.dumps(run_closed_loop_extra(args, torch, 0, args.extra_only)), flush=True)
        return
    args.warmup = max(args.warmup, 3) if args.impl == "dint_b200" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))

    if args.impl == "reference":
        return main_reference(args, rank, world)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (dint_b200 has no CPU fallback)")
    # stdout carries exactly one JSON line: libraries that print there (NCCL's version banner) go to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist_mod.init_process_group("nccl")
        dist = dist_mod
    from dint_b200.workloads import REF, HOT

    t_start = time.time()
    if world > 1:
        res = run_fasst_sharded(args, torch, dist, rank, world, True, args.steps, args.warmup, dump_dir=args.dump_outputs)
    else:
        res = run_fasst(args, torch, "REF", REF, args.steps, args.warmup, dump_dir=args.dump_outputs)

    # reduce over ranks: time = max, work = sum
    ms, committed, reqs = res["ms"], res["committed"], res["requests"]
    e2e_s, e2e_c, e2e_r = res.get("e2e_s"), res.get("e2e_committed", 0), res.get("e2e_requests", 0)
    launches = res["stats"]["kernel_launches"]
    parity = 1.0 if (res["parity_replay"] and res.get("e2e_parity", True)) else 0.0
    if dist is not None:
        t = torch.tensor([ms, e2e_s or 0.0], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        w = torch.tensor([committed, reqs, launches, e2e_c, e2e_r, parity, res["alg_bytes"]], device="cuda", dtype=torch.float64)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
        ms, e2e_s = float(t[0]), float(t[1]) or None
        committed, reqs, launches, e2e_c, e2e_r = int(w[0]), int(w[1]), int(w[2]), int(w[3]), int(w[4])
        parity_all = float(w[5]) == world
        alg_total = float(w[6])
    else:
        parity_all, alg_total = parity == 1.0, float(res["alg_bytes"])
    extra = {}
    fallback = None
    if rank == 0:
        fallback = {"metric": "committed txns/sec (lock_fasst)", "value": committed / (ms * 1e-3), "unit": "txn/s", "n_gpus": world,
                    "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / res["steps_timed"], "higher_is_better": True,
                    "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": {"workload": WORKLOAD},
                    "requests_per_s": reqs / (ms * 1e-3), "timed_region_s": ms * 1e-3,
                    "replies_bit_exact_vs_closed_loop_recording": bool(parity_all), "clocks": res["clocks"], "gpu_launches": launches,
                    "note": "the side measurements exceeded their deadline: this is the headline alone (no roofline, no extras)"}
        if e2e_s:
            fallback["e2e"] = {"value": e2e_c / e2e_s, "unit": "txn/s", "h2d_bytes_per_step": STEP_REQS * 9 * world,
                               "d2h_bytes_per_step": STEP_REQS * 9 * world}
    watchdog = Watchdog(float(os.environ.get("DINT_BENCH_EXTRA_DEADLINE", "1500")), rank, fallback, real_stdout)
    if not args.no_extra and world > 1:
        # the reference's fixed constants at N GPUs (contention rises with N), checked against the reference BINARY
        try:
            r2 = run_fasst_sharded(args, torch, dist, rank, world, False, max(4, args.steps // 4), 3, do_e2e=False)
            t = torch.tensor([r2["ms"]], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            w = torch.tensor([r2["committed"], r2["requests"], 1.0 if r2["parity_replay"] else 0.0], device="cuda", dtype=torch.float64)
            dist.all_reduce(w, op=dist.ReduceOp.SUM)
            if rank == 0:
                extra["lock_fasst_reference_constants"] = {
                    "workload": f"36,000,000 slots and 24,000,000 ids in total (the reference's constants) shared by {world} x 1048576 clients",
                    "txn_per_s": float(w[0]) / (float(t[0]) * 1e-3), "requests_per_s": float(w[1]) / (float(t[0]) * 1e-3),
                    "committed_per_request": float(w[0]) / max(1.0, float(w[1])), "replies_bit_exact_vs_closed_loop_recording": float(w[2]) == world,
                    "oracle_parity": r2.get("oracle_parity"), "timed_region_s": float(t[0]) * 1e-3}
        except Exception as ex:
            extra["lock_fasst_reference_constants"] = {"error": repr(ex)[:300]}
        if world >= 3:
            for kn in ("tatp", "smallbank"):
                try:
                    r3 = run_txn_sharded(args, torch, dist, rank, world, kn)
                    if rank == 0:
                        extra[kn] = r3
                except Exception as ex:
                    extra[kn] = {"error": repr(ex)[:300]}
    if rank != 0:
        watchdog.cancel()
        if dist is not None:
            dist.destroy_process_group()
        return
    peak, peak_how = peaks()
    kt = res["kernel_times"]
    nl, tot_ms = kt["k_apply"]
    avg_s = tot_ms / nl * 1e-3
    alg_per_launch = res["alg_bytes"] / nl
    achieved = alg_per_launch / avg_s / 1e9
    akt = res.get("all_kernel_times", kt)
    roof = {"kernel": "k_apply<lock_fasst>", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": load_static_traffic("k_apply<lock_fasst>"),
            "traffic_source": "static: profiles/ncu_traffic.json (one single-pass ncu capture per round, --cache-control none; not measured by this run)",
            "peak_source": peak_how, "avg_launch_us": avg_s * 1e6, "launches": nl, "algorithmic_bytes_per_launch": alg_per_launch,
            "timing": "CUDA events around every k_apply launch of the timed region",
            "whole_step": {"achieved": alg_total / (ms * 1e-3) / 1e9 / world, "frac": alg_total / (ms * 1e-3) / 1e9 / world / peak,
                           "note": "all algorithmic bytes of the timed region / its whole duration (every kernel, launch gaps, state restores), per GPU"},
            "all_kernels_ms_profiled_cycle": {k: round(v[1], 3) for k, v in akt.items()}}
    if "k_classify" in akt:
        l1, t1 = akt["k_classify"]
        ach1 = res["alg_bytes"] / max(1, l1) / (t1 / l1 * 1e-3) / 1e9 if world == 1 else None
        roof["k_classify"] = {"avg_launch_us": t1 / l1 * 1e3, "launches_profiled_cycle": l1,
                              "achieved_same_algorithmic_bytes": ach1, "frac": (ach1 / peak) if ach1 else None,
                              "note": "second pass over the same requests (conflict flags + replay of the previous chunk): it moves no algorithmic byte "
                                      "of its own, so its fraction is quoted against the step's algorithmic bytes; from the fully profiled cycle, not the timed one"}
    line = {
        "metric": "committed txns/sec (lock_fasst)", "value": committed / (ms * 1e-3), "unit": "txn/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / res["steps_timed"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": WORKLOAD + (f" -- per GPU; key space scaled with the GPU count: {36 * world},000,000 slots, {24 * world},000,000 ids in total "
                                           "(constant contention; the reference's fixed constants: extra.lock_fasst_reference_constants)" if world > 1 else ""),
                   "baseline_config": "BASELINE.json configs[1] (lock_fasst OCC validate/commit, 1 B200).  Its '4800 keys, "
                                      "Zipf-0.8, 24M-op' wording is, in the reference, 4800 trace FILES, read fraction 0.8 and 24 M "
                                      "uniform lock ids (BASELINE.md section 1 note, lock_fasst/caladan/trace_init.sh:9-27): the headline "
                                      "runs that reference shape; the literal reading (4800 ids, Zipf 0.8) is extra.lock_fasst_HOT",
                   "requests_per_step": STEP_REQS * world, "chunk": args.chunk,
                   "timed_region": f"{res['steps_timed']} recorded steps once, {ms * 1e-3:.3f} s, from the server state the warm-up steps left",
                   "cache": "every step replays a different 37.7 MB trace segment (K segments larger than L2; lock/version tables 148.5 MB > 126 MB L2)",
                   "parallelism": (f"key-space sharded x{world}: dispatch / engine / combine kernels over NVLink peer memory (owner = slot % {world}), "
                                   "one process per GPU") if world > 1 else "single GPU"},
        "requests_per_s": reqs / (ms * 1e-3),
        "timed_region_s": ms * 1e-3,
        "replies_bit_exact_vs_closed_loop_recording": bool(parity_all),
        "abort_stats": {k: res["wl_stats"][k] for k in ("committed", "validation_aborts", "lock_rejects")},
        "committed_per_request": committed / max(1, reqs),
        "conflicted_fraction": res["stats"]["conflicted"] / max(1, res["stats"]["requests"]),
        "clocks": res["clocks"],
        "gpu_launches": launches,
        "roofline": roof,
    }
    if "oracle_parity" in res:
        line["oracle_parity"] = res["oracle_parity"]
    if e2e_s:
        line["e2e"] = {"value": e2e_c / e2e_s, "unit": "txn/s", "h2d_bytes_per_step": STEP_REQS * 9 * world,
                       "d2h_bytes_per_step": STEP_REQS * 9 * world, "requests_per_s": e2e_r / e2e_s, "timed_region_s": e2e_s,
                       "steps_timed": res.get("e2e_steps"),
                       "path": ("dint_submit(): pinned host wire structs -> H2D -> kernels -> D2H, one call per step" if world == 1 else
                                "dint_shard_submit_host(): pinned host wire structs -> H2D | dispatch | engine | combine | D2H pipelined, one call per step")}
    if "cpu_baseline" in res:
        line["cpu_baseline"] = res["cpu_baseline"]
        if world == 1 and not args.no_extra:
            import oracle_lib as O
            rq0, _, tpr = res["first_step"]
            if O.ref_available(1):
                line["cpu_baseline"]["udp_as_shipped"] = udp_as_shipped(O, 1, rq0, tpr)
    elif world > 1:
        import oracle_lib as O
        rq0, rs0, tpr = res["first_step"]
        rb = CLIENTS * 9
        line["cpu_baseline"] = reference_check(1, rq0[:rb], rs0[:rb], tpr, "rank 0's first client round (timing only: the replies of a sharded run are "
                                               "checked in oracle_parity)")
        line["cpu_baseline"].pop("gpu_replies_equal_reference", None)
    if not args.no_extra and world == 1:
        try:
            hot = run_fasst(args, torch, "HOT", HOT, max(3, args.steps // 3), 3, do_e2e=False, do_ref=True)
            extra["lock_fasst_HOT"] = {
                "workload": "BASELINE.json literal: 4800 lock ids, Zipf 0.8, same clients/protocol",
                "txn_per_s": hot["committed"] / (hot["ms"] * 1e-3), "requests_per_s": hot["requests"] / (hot["ms"] * 1e-3),
                "timed_region_s": hot["ms"] * 1e-3,
                "abort_stats": {k: hot["wl_stats"][k] for k in ("committed", "validation_aborts", "lock_rejects")},
                "conflicted_fraction": hot["stats"]["conflicted"] / max(1, hot["stats"]["requests"]),
                "replies_bit_exact_vs_closed_loop_recording": bool(hot["parity_replay"]), "cpu_baseline": hot.get("cpu_baseline")}
            extra["on_gpu_closed_loop"] = run_gpu_clients(args, torch, REF)
            extra["store_get"] = run_store_get(args, torch, rank, max(3, args.steps // 2), 3)
            extra["tatp"] = run_txn(args, torch, rank, "tatp")
            extra["smallbank"] = run_txn(args, torch, rank, "smallbank")
        except Exception as ex:  # side measurements must never cost the headline line
            extra["error"] = repr(ex)[:300]
        for kn in ("lock_2pl", "log_server"):
            # side measurements in a child process with a deadline: whatever happens there, the headline stands
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--extra-only", kn, "--chunk", str(args.chunk)],
                                   capture_output=True, timeout=400)
                rows = [l for l in r.stdout.decode().splitlines() if l.startswith("{")]
                extra[kn] = json.loads(rows[-1]) if rows else {"error": f"exit {r.returncode}: {r.stderr.decode()[-300:]}"}
            except Exception as ex:
                extra[kn] = {"error": repr(ex)[:300]}
        try:
            torch.cuda.empty_cache()
            extra["udp_front_end"] = run_udp_front_end()
        except Exception as ex:
            extra["udp_front_end"] = {"error": repr(ex)[:300]}
    if extra:
        line["extra"] = extra
    line["bench_wall_s"] = round(time.time() - t_start, 1)
    watchdog.cancel()
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main_reference(args, rank, world):
    """--impl reference: the reference's own lock_fasst server (oracle/_ref, built from /root/reference unmodified) on
    the host cores, handler only (replay shim: no UDP syscalls), on the GPU arm's workload: the same 1,048,576-client
    closed-loop trace (same seed; recorded here against the CPU restatement, whose replies are the GPU's bit for bit).
    A step = the first 4 trace steps (16.8 M requests) x `repeat` passes through `server <all cores>`."""
    if rank != 0:
        return
    import oracle_lib as O
    from dint_b200 import wire
    from dint_b200.workloads import Workload, REF
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    ora = O.Oracle(wire.FASST)
    wl = Workload(wire.FASST, n_clients=CLIENTS, seed=20230, **REF)
    n_rec = 4
    reqs, _, _ = record_closed_loop(ora.process, wl, n_rec, 9)
    st = wl.stats()
    # committed / request of the GPU arm's window (steps W.. of the same closed loop) is a little higher than of the first
    # 4 steps (transactions take >= 11 rounds to complete): use a longer CPU-side recording for the conversion factor
    for _ in range(8 * ROUNDS_PER_STEP):
        wl.feed(ora.process(wl.next()))
    st2 = wl.stats()
    txn_per_req = (st2["committed"] - st["committed"]) / max(1, st2["requests"] - st["requests"])
    sample = reqs.reshape(-1)
    n = sample.size // 9
    kind = "reference" if O.ref_available(wire.FASST) else "port"

    def one(threads, repeat):
        if kind == "reference":
            _, stt = O.run_ref(wire.FASST, sample, threads=threads, repeat=repeat, want_out=False, spread=True)
            return stt["requests"] / stt["seconds"]
        t0 = time.perf_counter()
        O.Oracle(wire.FASST).process(sample)
        return n / (time.perf_counter() - t0)

    rows = {}
    if kind == "reference":                          # scaling rows: 1 thread, 8 threads (the reference's own setting), all cores
        for th in sorted({1, min(8, cores), cores}):
            rep = max(1, min(400, int(2.0 * one(th, 2) / n)))          # about two seconds per repeat
            rates = [one(th, rep) for _ in range(3)]
            rows[str(th)] = {"req_per_s_median": sorted(rates)[1], "req_per_s_min": min(rates), "req_per_s_max": max(rates), "repeat": rep}
    # a step = `rep_all` passes over the sample, sized from a short calibration run to take about three seconds whatever the box
    cal = one(cores if kind == "reference" else 1, 4)
    rep_all = max(1, min(400, int(3.0 * cal / n)))
    times, rates = [], []
    for s in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        r = one(cores if kind == "reference" else 1, rep_all)
        if s >= args.warmup:
            rates.append(r)
            times.append(time.perf_counter() - t0)
    rate = float(np.median(rates))
    val = rate * txn_per_req
    line = {"impl": "reference", "metric": "committed txns/sec (lock_fasst)", "value": val, "unit": "txn/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(times)) * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "note": "handler only: the reference server.cc under the LD_PRELOAD replay shim (no UDP syscalls), "
                               f"`server {cores}` re-pinned one thread per host core; a step = the first {n_rec} steps of the same closed-loop trace "
                               f"({n} requests) x {rep_all} passes; value = median over the {args.steps} steps (min {min(rates) * txn_per_req:.3g}, max {max(rates) * txn_per_req:.3g} txn/s)"},
            "requests_per_s": rate, "committed_per_request": txn_per_req,
            "spread": {"min_over_median": min(rates) / rate, "max_over_median": max(rates) / rate},
            "thread_scaling": rows,
            "cpu_baseline": {"value": val, "unit": "txn/s", "cores": cores if kind == "reference" else 1, "kind": kind,
                             "sample": f"{n}-request closed-loop trace x {rep_all} passes per step"},
            "e2e": {"value": val, "unit": "txn/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
