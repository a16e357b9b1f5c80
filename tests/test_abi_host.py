"""CPU tests of the product's host side: the C-ABI library loads and exports every symbol that
include/dint_b200.h declares, the host/device-shared arithmetic is exact, and the compute entry points
fail loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import conftest
from dint_b200 import engine as E, wire

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "dint_b200.h")).read()
    declared = set(re.findall(r"\b(dint_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(E.ABI_SYMBOLS), declared ^ set(E.ABI_SYMBOLS)
    L = E.lib()
    for s in declared:
        assert hasattr(L, s), s


def test_msg_sizes_match_reference_structs():
    L = E.lib()
    assert [L.dint_msg_size(k) for k in range(6)] == [6, 9, 53, 53, 55, 23] == wire.MSG_SIZE
    assert [L.dint_log_entry_size(k) for k in range(6)] == wire.LOG_ENTRY_SIZE


def test_fasthash_and_fastmod_are_exact():
    import test_oracle_golden as TG
    L = E.lib()
    for (x, ln), h in TG.KAT.items():
        assert L.dint_test_fasthash64(x, ln) == h
    rng = np.random.default_rng(1)
    divisors = [1, 2, 3, 5, 7, 8, 4800, 2625000, 9000000, 10500000, 26250000, 36000000, 39375000,
                (1 << 31) - 1, 1 << 31, (1 << 32) - 1, 12345678]
    divisors += [int(d) for d in rng.integers(1, 2**32, size=40)]
    ns = [0, 1, 2**32 - 1, 2**32, 2**63, 2**64 - 1, 2**64 - 2] + [int(x) for x in rng.integers(0, 2**64, size=400, dtype=np.uint64)]
    for d in divisors:
        for n in ns + [d - 1, d, d + 1, 2 * d, 2 * d - 1, (2**64 - 1) // d * d, (2**64 - 1) // d * d - 1]:
            n &= 2**64 - 1
            assert L.dint_test_fastmod(n, d) == n % d, (n, d)


def test_host_slice_schedule_covers_every_call_exactly():
    """dint_submit's slice schedule (pure host logic): the slices sum to n, none exceeds a device buffer,
    small slices sit only at the two ends (a pyramid), and tiny calls are not split."""
    import ctypes as C
    L = E.lib()
    L.dint_test_host_slices.restype = C.c_uint32
    L.dint_test_host_slices.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, C.POINTER(C.c_uint32), C.c_uint32]
    buf = (C.c_uint32 * 4096)()
    rng = np.random.default_rng(7)
    cases = [(1, 131072, 262144), (1000, 131072, 262144), (131072, 131072, 262144), (262144, 131072, 262144),
             (1 << 20, 131072, 262144), ((1 << 20) + 5, 131072, 262144), (4 << 20, 65536, 1 << 20), (10**8, 65536, 262144)]
    cases += [(int(rng.integers(1, 3 * 10**7)), int(rng.choice([128, 4096, 65536, 1 << 20])), int(rng.choice([128, 65536, 262144, 1 << 20])))
              for _ in range(300)]
    for n, mn, mx in cases:
        for ramp_up in (0, 1):
            k = L.dint_test_host_slices(n, mn, mx, ramp_up, buf, 4096)
            assert k <= 4096 or n > 4096 * mx
            sl = list(buf[:min(k, 4096)])
            if k <= 4096:
                assert sum(sl) == n, (n, mn, mx, ramp_up)
            assert all(0 < c <= mx for c in sl), (n, mn, mx, ramp_up, sl[:8])
            if n < min(mn, mx):
                assert sl == [n]
            if mn < mx and n >= 2 * mn and k <= 4096:
                assert sl[-1] == mn, (n, mn, mx, sl)                    # the call ends on its smallest slice


def test_default_cfg_is_the_reference_constants():
    c = E.default_cfg(wire.TATP)
    assert (c.lock_slots, c.log_ring, c.subs_sizing, c.accts_sizing, c.n_shards) == (36000000, 1000000, 7000000, 24000000, 1)
    assert E.default_cfg(wire.STORE).subs_sizing == 2000000


@pytest.mark.skipif(conftest.HAS_GPU, reason="only meaningful without a GPU")
def test_no_cpu_fallback():
    with pytest.raises(E.DintError) as ei:
        E.Engine(wire.FASST)
    assert ei.value.code == -19        # DINT_ENODEV


@pytest.mark.skipif(conftest.HAS_GPU, reason="only meaningful without a GPU")
def test_udp_front_end_builds_and_fails_loudly_without_a_gpu():
    """dint_udp_server (the reference's UDP server shape over the C ABI) has no CPU path either."""
    import subprocess
    from dint_b200 import _build
    E.lib()
    assert os.path.exists(_build.UDP_SERVER)
    r = subprocess.run([_build.UDP_SERVER, "lock_fasst", "--port", "29731"], capture_output=True, timeout=60)
    assert r.returncode == 1 and b"dint_create failed" in r.stderr
    assert subprocess.run([_build.UDP_SERVER, "no_such_server"], capture_output=True, timeout=60).returncode == 2


def test_stats_struct_layout():
    """dint_stats is 12 u64 wide; fallback_chunks took the first reserved slot, so the layout did not move."""
    assert C.sizeof(E.DintStats) == 12 * 8
    assert E.DintStats.kv_rebuilds.offset == 8 * 8 and E.DintStats.fallback_chunks.offset == 9 * 8
