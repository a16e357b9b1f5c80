"""bench.py's own plumbing without a GPU: the JSON line is assembled from a canned headline result and stubbed side
measurements (no number here means anything); what is checked is the contract -- ONE JSON line on stdout with the keys
the driver reads -- and the watchdog that prints the headline alone when the side measurements exceed their deadline."""
import json
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HARNESS = textwrap.dedent('''
    import os, sys, time, types
    sys.path.insert(0, %r)
    sys.argv = ["bench.py", "--steps", "4", "--warmup", "3"]
    import torch
    torch.cuda.is_available = lambda: True
    torch.cuda.empty_cache = lambda: None
    import bench as B
    res = dict(ms=1113.0, kernel_times={"k_apply": (160, 5.0)}, stats={"kernel_launches": 500, "conflicted": 10, "requests": 1000},
               clocks={"sm_mhz": 1965, "sm_max_mhz": 1965, "reasons": [], "samples": 5}, parity_replay=True,
               all_kernel_times={"k_classify": (40, 1.06), "k_apply": (40, 1.25), "k_ordered": (40, 0.2)}, committed=650000000, requests=16000000000,
               steps_timed=40, alg_bytes=3.8e9, reply_mix={}, e2e_s=1.0, e2e_steps=40, e2e_parity=True, e2e_committed=150000000, e2e_requests=4000000000,
               wl_stats={"committed": 1, "validation_aborts": 2, "lock_rejects": 3, "requests": 30},
               cpu_baseline={"value": 1.0, "unit": "txn/s", "cores": 1, "kind": "reference", "req_per_s": 1.0, "sample": "x", "gpu_replies_equal_reference": True},
               first_step=(None, None, 0.04))
    B.run_fasst = lambda *a, **k: dict(res)
    slow = float(os.environ.get("MOCK_SLOW", "0"))
    def extra(name):
        def f(*a, **k):
            time.sleep(slow)
            return {"name": name}
        return f
    B.run_gpu_clients = extra("clients"); B.run_store_get = extra("store"); B.run_txn = extra("txn"); B.run_udp_front_end = extra("udp")
    B.udp_as_shipped = lambda *a, **k: {"req_per_s": 1}
    B.subprocess.run = lambda *a, **k: types.SimpleNamespace(stdout=b'{"requests_per_s": 1}\\n', stderr=b"", returncode=0)
    import oracle_lib
    oracle_lib.ref_available = lambda *a, **k: False
    B.main()
''') % ROOT

KEYS = ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
        "config", "clocks", "gpu_launches", "e2e"]


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    r = subprocess.run([sys.executable, "-c", HARNESS], env=env, capture_output=True, timeout=120)
    lines = [l for l in r.stdout.decode().splitlines() if l.strip()]
    assert r.returncode == 0 and len(lines) == 1, (r.returncode, r.stdout[-500:], r.stderr[-800:])
    return json.loads(lines[0])


def test_bench_prints_one_json_line_with_the_contract_keys():
    d = _run({})
    for k in KEYS + ["roofline", "cpu_baseline", "extra"]:
        assert k in d, k
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    assert set(d["cpu_baseline"]) >= {"value", "unit", "cores", "kind", "sample"}
    assert set(d["e2e"]) >= {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert "workload" in d["config"] and d["scaling"] == "weak" and d["vs_baseline"] is None


def test_bench_watchdog_prints_the_headline_when_the_extras_hang():
    d = _run({"MOCK_SLOW": "3", "DINT_BENCH_EXTRA_DEADLINE": "2"})
    for k in KEYS:
        assert k in d, k
    assert "exceeded their deadline" in d["note"] and "extra" not in d


def test_dump_outputs_write_a_fixed_exact_sample_of_the_replies(tmp_path):
    import numpy as np
    import bench as B
    from dint_b200 import wire
    rec = np.zeros(B.STEP_REQS, dtype=wire.MSG_DTYPE[wire.FASST])
    idx = np.arange(rec.size, dtype=np.uint64)
    rec["type"] = 4 + idx % 5
    rec["lid"] = idx
    rec["ver"] = (idx * 2654435761) % 2**32
    for d in ("a", "b"):
        B.dump_replies(str(tmp_path / d), wire.as_bytes(rec))
    names = ["lock_fasst_reply_lid.npy", "lock_fasst_reply_type.npy", "lock_fasst_reply_ver.npy"]
    assert sorted(p.name for p in (tmp_path / "a").iterdir()) == names
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 << 20
    got = {}
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float64 and np.array_equal(a, b)         # the same sample in every run
        got[n.split("_")[-1][:-4]] = a.astype(np.uint64)
    lid = got["lid"]
    assert 0 < lid.size < rec.size and (np.diff(lid) > 0).all()
    assert np.array_equal(got["type"], 4 + lid % 5) and np.array_equal(got["ver"], (lid * 2654435761) % 2**32)
