#!/usr/bin/env python
"""Live TATP / SmallBank closed loop with the clients on the GPU (GpuTxnClients, dint_txn_clients_*).

bench.py's run_txn configuration: 2^20 clients, 3 shard engines on one GPU, each holding the reference population
(tatp 7,000,000 subscribers / smallbank 24,000,000 accounts).  Per kind:
  1. checks the first 8 rounds at scale: a host TxnWorkload (same gid0) fed the GPU round's replies must emit the GPU
     clients' next round, record for record;
  2. warms up (--warm rounds in all), then times at least --seconds of rounds with device events;
  3. in separate profiled runs: engine kernel time (Engine.profile) and client kernel time (torch.profiler); the rest of
     a round is the host's wait on the per-shard counts plus the launch gap.
Prints one JSON line per kind, with the device name and power limit read in the same run.

    python tools/txn_clients_bench.py [--kinds tatp,smallbank] [--clients 1048576] [--seconds 1.0]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def device_info(torch):
    d = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        d["power_limit_and_max_sm_clock"] = q.stdout.strip() or "not available"
    except (OSError, subprocess.TimeoutExpired):
        d["power_limit_and_max_sm_clock"] = "not available"
    return d


def check_at_scale(kind, gc, n_clients, subscribers, gid0, rounds):
    """Feed a host TxnWorkload the GPU's replies for `rounds` rounds; every next round must be the GPU's."""
    from dint_b200.txn_workloads import TxnWorkload
    from dint_b200.wire import MSG_SIZE
    msg = MSG_SIZE[kind]
    wl = TxnWorkload(kind, n_clients=n_clients, n_shards=3, subscribers=subscribers, gid0=gid0)
    records = 0
    for r in range(rounds + 1):
        want_rq, want_dst = wl.next()
        got_rq, got_dst, _ = gc.peek()
        if not (np.array_equal(got_dst, want_dst) and np.array_equal(got_rq, want_rq)):
            bad = np.flatnonzero((got_rq.reshape(-1, msg) != want_rq.reshape(-1, msg)).any(1)) if got_rq.size == want_rq.size else []
            raise SystemExit(f"round {r}: GPU clients differ from the host clients (first differing record {bad[:1]})")
        records += want_dst.size
        if r == rounds:
            break
        gc.run(1)
        wl.feed(gc.peek()[2])
    ok = wl.stats()
    wl.close()
    return {"rounds_checked": rounds, "records_checked": records, "host_stats_equal": ok == gc.stats()}


def run_kind(torch, kind_name, args):
    from dint_b200 import Engine, GpuTxnClients, wire
    kind = wire.TATP if kind_name == "tatp" else wire.SMALLBANK
    subscribers = 7_000_000 if kind == wire.TATP else 24_000_000
    t0 = time.time()
    engs = [Engine(kind, device=0, populate=True) for _ in range(3)]
    t_pop = time.time() - t0
    stream = torch.cuda.current_stream()
    gc = GpuTxnClients(engs, args.clients, subscribers=subscribers, gid0=0)
    res = {"workload": f"{kind_name} mix, {args.clients} closed-loop clients on the GPU, 3 shard engines x {subscribers} "
                       f"{'subscribers' if kind == wire.TATP else 'accounts'} on one GPU, live (no replay)",
           "populate_s_per_3_shards": round(t_pop, 1)}
    res["check"] = check_at_scale(kind, gc, args.clients, subscribers, 0, args.check_rounds)
    done = args.check_rounds
    t = time.perf_counter()
    gc.run(max(1, args.warm - done), stream.cuda_stream)
    per_round = (time.perf_counter() - t) / max(1, args.warm - done)
    k = max(20, math.ceil(args.seconds * 1.1 / per_round))
    # timed window
    s0 = gc.stats()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    gc.run(k, stream.cuda_stream)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    s1 = gc.stats()
    d = {key: s1[key] - s0[key] for key in ("requests", "txns", "committed", "rounds")}
    by = {n: (s1["by_type"][n][0] - s0["by_type"][n][0], s1["by_type"][n][1] - s0["by_type"][n][1]) for n in s1["by_type"]}
    sec = ms * 1e-3
    res.update({"timed_rounds": d["rounds"], "timed_region_s": round(sec, 4),
                "txn_per_s": d["committed"] / sec, "requests_per_s": d["requests"] / sec,
                "us_per_round": ms * 1e3 / d["rounds"], "requests_per_round": d["requests"] / d["rounds"],
                "abort_rate": 1.0 - d["committed"] / max(1, d["txns"]),
                "commit_rate_by_type": {n: round(c / max(1, b), 4) for n, (b, c) in by.items()}})
    # split of a round, each part from its own run of args.prof_rounds rounds
    pr = args.prof_rounds
    for e in engs:
        e.profile(True)
    gc.run(pr, stream.cuda_stream)
    torch.cuda.synchronize()
    eng_ms = 0.0
    for e in engs:
        e.sync(check=False)
        eng_ms += sum(ms_ for _, ms_ in e.kernel_times().values())
        e.profile(False)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gc.run(pr, stream.cuda_stream)
        torch.cuda.synchronize()
    cli_us, cli = 0.0, {}
    for ev in prof.key_averages():
        if "k_txn_" in ev.key:
            us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
            cli_us += us
            name = ev.key.split("<")[0].split("(")[0].replace("void ", "").replace("dint::", "")
            cli[name] = cli.get(name, 0.0) + us / pr
    us_round = res["us_per_round"]
    eng_us = eng_ms * 1e3 / pr
    res["round_split_us"] = {"engine_kernels": round(eng_us, 1), "client_kernels": round(cli_us / pr, 1),
                             "client_kernels_by_name": {k_: round(v, 1) for k_, v in cli.items()},
                             "host_wait_and_launch_gap": round(us_round - eng_us - cli_us / pr, 1),
                             "note": "engine and client kernel times come from separate profiled runs of "
                                     f"{pr} rounds; the gap is the timed round minus both"}
    gc.close()
    for e in engs:
        e.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kinds", default="tatp,smallbank")
    ap.add_argument("--clients", type=int, default=1 << 20)
    ap.add_argument("--warm", type=int, default=50, help="rounds before the timed window (the checked rounds included)")
    ap.add_argument("--check-rounds", type=int, default=8)
    ap.add_argument("--seconds", type=float, default=1.0, help="least length of the timed window")
    ap.add_argument("--prof-rounds", type=int, default=100)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement runs on the GPU only")
    info = device_info(torch)
    for kind_name in args.kinds.split(","):
        res = run_kind(torch, kind_name, args)
        res.update(info)
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
