"""GPU: the live hook on a real B200 -- device accounting vs host sum, gpu_mem cap with real allocations,
burst-edge token renewals, and accumulated GPU-ms against the reference stack's ledger (+-1 %).  What the reference
stack did on a B200 was recorded by tests/golden/make_live_golden.py into tests/golden/ref_live_b200.json."""
import ctypes as C
import glob
import json
import os
import subprocess as sp
import tempfile
import time

import pytest

import kubeshare_b200 as kb
import orc
import wireproto as wp

pytestmark = pytest.mark.gpu
GIB8 = 8589934592
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live_b200.json")


def env_pool(tmp, pod="bench/c0", quota=None, **kw):
    quota = quota or "1\nbench/c0 1.0 1.0 %d\n" % GIB8
    with open(os.path.join(tmp, "quota.txt"), "w") as f:
        f.write(quota)
    env = {k: v for k, v in os.environ.items() if not k.startswith("GEMHOOK_") and k != "LD_PRELOAD"}
    env.update(LD_PRELOAD=kb.LIB_PATH, GEMHOOK_POOL=os.path.join(tmp, "pool"), GEMHOOK_QUOTA_FILE=os.path.join(tmp, "quota.txt"),
               POD_NAME=pod, GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"))
    env.update({k: str(v) for k, v in kw.items()})
    return env


def storm(env, *args, timeout=300):
    p = sp.run([kb.STORM_PATH, *map(str, args)], env=env, stdout=sp.PIPE, stderr=sp.PIPE, timeout=timeout)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return json.loads(p.stdout)


def stats(tmp):
    return [json.load(open(f)) for f in sorted(glob.glob(os.path.join(tmp, "stats.*.json")))]


def golden(key):
    with open(GOLDEN) as f:
        return json.load(f)[key]


def start_arbiter(tmp, cfg, pool):
    """gem-arbiter (the native gem-pmgr + gem-schd) on a fresh port, gem-schd's defaults; returns (process, port)."""
    with open(os.path.join(tmp, "cfg.txt"), "w") as f:
        f.write(cfg)
    port, log = wp.free_port(), os.path.join(tmp, "arbiter.log")
    with open(log, "w") as f:
        arb = sp.Popen([os.path.join(kb.HERE, "bin", "gem-arbiter"), "--pool", pool, "-p", tmp, "-f", "cfg.txt", "-P", str(port),
                        "-q", "300", "-m", "20", "-w", "10000"], stderr=f)
    deadline = time.time() + 10
    while time.time() < deadline and "listening" not in open(log).read():
        time.sleep(0.05)
    return arb, port


def pool_spans(pool):
    """[(start_ms, end_ms)] of every token in the pool's ledger, oldest first."""
    L = kb.lib()
    p = L.gemhook_pool_open(pool.encode(), 0, 0, 0, 0, 0)
    n = L.gemhook_pool_history(p, None, None, None, 0)
    sl, a, b = (C.c_int * n)(), (C.c_double * n)(), (C.c_double * n)()
    n = min(n, L.gemhook_pool_history(p, sl, a, b, n))
    L.gemhook_pool_close(p)
    return [(a[i], b[i]) for i in range(n)]


@pytest.mark.parametrize("seg", [0, 256])
def test_device_reduced_sm_time_equals_host_sum(seg):
    with tempfile.TemporaryDirectory() as tmp:
        res = storm(env_pool(tmp, GEMHOOK_SEG_LAUNCHES=seg, GEMHOOK_FLUSH_RECORDS=16), "--mode", "storm", "--steps", 4,
                    "--warmup", 1, "--step-launches", 16384, "--sync-every", 1024)
        st = stats(tmp)[0]
        assert st["launches"] == 5 * 16384
        assert st["segments"] >= (20 if seg == 0 else 300)   # bursts younger than GEMHOOK_SEG_MIN_US merge
        assert st["acct_kernels"] >= 2
        assert st["gpu_ns"] == st["gpu_ns_host"] > 0          # sm_100a reduction == host-side sum, bit-exact
        # the bursts cover the storm: SM-time within the wall time, and most of it
        assert 0.5 * res["event_ms"] < st["gpu_ns"] / 1e6 * 4 / 5 < 1.02 * res["event_ms"]


def test_config4_real_allocations_bit_exact_oom_point():
    O = orc.load()
    with tempfile.TemporaryDirectory() as tmp:
        res = storm(env_pool(tmp), "--mode", "memsweep")
    limit, used, first_fail = GIB8, 0, -1
    for row in res["sweep1"]:
        ok = O.orc_mem_prehook_allows(row["bytes"], used, limit)
        assert row["rc"] == (0 if ok else 2), row
        used += row["bytes"] if ok else 0
        if not ok and first_fail < 0:
            first_fail = row["i"]
        assert (row["free"], row["total"]) == (limit - used, limit)
    assert res["first_fail"] == first_fail == 8
    used = 0
    for sz, rc, free in res["sweep2"]:
        ok = O.orc_mem_prehook_allows(sz, used, limit)
        assert rc == (0 if ok else 2)
        used += sz if ok else 0
        assert free == limit - used
    assert res["free_end"] == limit


def test_config3_bursty_tokens_renew_only_at_burst_edges():
    with tempfile.TemporaryDirectory() as tmp:
        quota = "4\n" + "".join("bench/c%d 0.25 1.0 %d\n" % (i, GIB8) for i in range(4))
        procs = []
        for i in range(4):
            env = env_pool(tmp, pod="bench/c%d" % i, quota=quota)
            procs.append(sp.Popen([kb.STORM_PATH, "--mode", "bursty", "--rounds", "150", "--client-id", str(i), "--nclients", "4",
                                   "--barrier-dir", tmp, "--out", os.path.join(tmp, "out%d.json" % i)], env=env, stderr=sp.PIPE))
        for p in procs:
            _, err = p.communicate(timeout=600)
            assert p.returncode == 0, err.decode()[-1000:]
        st = stats(tmp)
        outs = [json.load(open(os.path.join(tmp, "out%d.json" % i))) for i in range(4)]
        assert len(st) == 4
        for s in st:
            o = [x for x in outs if x["launches"] == s["launches"]]
            assert o, "every launch intercepted"
            assert s["slow_path"] <= 150 + s["token_requests"] + 2   # one slow path per burst (+ tracker-forced edges)
            assert s["token_requests"] <= s["slow_path"] + 1          # renewals happen only on the slow path
            assert s["gpu_ns"] == s["gpu_ns_host"] > 0
        # 4 clients x ~150 bursts x ~2000 launches x 5 us: everybody got GPU time, nobody starved
        busy = [s["gpu_ns"] for s in st]
        assert min(busy) > 0.3 * max(busy)


def test_accumulated_gpu_ms_within_1pct_of_reference_ledger():
    """Same storm through (a) the reference hook against UNMODIFIED gem-pmgr + gem-schd(_DEBUG), as recorded on a B200
    (gem-schd's own ledger dump, scheduler.cpp:693-714, is the judge: sum(end-start)), (b) our hook over TCP to
    gem-arbiter and (c) our hook on the credit pool, both judged by the pool's ledger."""
    ref = golden("accumulated")
    totals = {"reference": ref}
    for which in ("ours", "pool"):
        with tempfile.TemporaryDirectory() as tmp:
            pool, arb = os.path.join(tmp, "pool"), None
            try:
                if which == "ours":
                    arb, port = start_arbiter(tmp, "1\nbench/c0 1.0 1.0 %d\n" % GIB8, pool)
                    env = {k: v for k, v in os.environ.items() if not k.startswith("GEMHOOK_") and k != "LD_PRELOAD"}
                    env.update(POD_NAME="bench/c0", POD_MANAGER_PORT=str(port), LD_PRELOAD=kb.LIB_PATH, GEMHOOK_SCHEDULER_IP="127.0.0.1",
                               GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"))
                else:
                    env = env_pool(tmp)
                res = storm(env, "--mode", "storm", "--steps", 30, "--warmup", 2, "--step-launches", 65536)
                time.sleep(0.2)
                spans = pool_spans(pool)
                totals[which] = {"tokens": len(spans), "closed_ms": sum(e - s_ for s_, e in spans[:-1]), "wall_ms": res["wall_s"] * 1e3,
                                 "stats": stats(tmp)[0] if which == "ours" else {}}
            finally:
                if arb is not None:
                    arb.kill()
                    arb.wait()
    ours, pool = totals["ours"], totals["pool"]
    print("ledger totals:", json.dumps(totals))
    # closed tokens only (the last, still-held token is clipped at exit by the pool but kept at full quota by
    # gem-schd): same number of tokens, same closed time within 1 %
    assert pool["tokens"] == ref["tokens"] == ours["tokens"]
    assert abs(pool["closed_ms"] - ref["closed_ms"]) <= 0.01 * ref["closed_ms"], totals
    # identical launch trace, identical policy: the TCP path's ledger agrees within 1 % as well
    assert abs(ours["closed_ms"] - ref["closed_ms"]) <= 0.01 * ref["closed_ms"], totals
    # and our own per-token view of the same quantity matches what the ledger recorded for us (within 1 %)
    assert abs(ours["stats"]["accumulated_token_ms"] - ours["closed_ms"]) <= 0.01 * ours["closed_ms"], ours


def test_reference_hook_served_by_gem_arbiter_next_to_a_native_client():
    """Drop-in in the other direction: the UNMODIFIED reference hook speaks TCP to gem-arbiter while a native hook
    arbitrates in the same pool; both finish, both appear in one ledger.  The reference hook's side is its recorded
    conversation replayed: every request it sent, no earlier than it sent it, on its own connection."""
    rec = golden("legacy_hook_vs_arbiter")
    with tempfile.TemporaryDirectory() as tmp:
        pool = os.path.join(tmp, "pool")
        arb, port = start_arbiter(tmp, "2\nbench/native 0.5 1.0 %d\nbench/legacy 0.5 1.0 %d\n" % (GIB8, GIB8), pool)
        try:
            base = {k: v for k, v in os.environ.items() if not k.startswith("GEMHOOK_") and k != "LD_PRELOAD"}
            e_native = dict(base, LD_PRELOAD=kb.LIB_PATH, GEMHOOK_POOL=pool, POD_NAME="bench/native",
                            GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"))
            native = sp.Popen([kb.STORM_PATH, "--mode", "storm", "--steps", "6", "--warmup", "1", "--step-launches", "65536", "--out",
                               os.path.join(tmp, "o0.json")], env=e_native, stderr=sp.PIPE)
            t0 = time.monotonic()
            conns = [wp.Client("127.0.0.1", port, c["name"], timeout=60) for c in rec["conns"]]
            calls = sorted((t, n, k, kind, args, answer) for n, c in enumerate(rec["conns"]) for k, (t, kind, args, answer) in enumerate(c["calls"]))
            for t, n, k, kind, args, answer in calls:
                time.sleep(max(0.0, t0 + t - time.monotonic()))
                c = conns[n]
                assert c.next_id == k
                if kind == wp.REQ_QUOTA:
                    assert c.quota(*args) > 0
                elif kind == wp.REQ_MEM_LIMIT:
                    assert list(c.mem_limit()) == answer
                else:
                    assert [c.mem_update(*args)] == answer
            time.sleep(max(0.0, t0 + rec["legacy_wall_s"] - time.monotonic()))   # the hook held its last token until it exited
            for c in conns:
                c.close()
            _, err = native.communicate(timeout=300)
            assert native.returncode == 0, err.decode()[-1500:]
            assert json.load(open(os.path.join(tmp, "o0.json")))["launches"] == 6 * 65536
            L = kb.lib()
            p = L.gemhook_pool_open(pool.encode(), 0, 0, 0, 0, 0)
            acc = {n: L.gemhook_pool_accumulated_ms(p, L.gemhook_pool_find(p, n.encode())) for n in ("bench/native", "bench/legacy")}
            L.gemhook_pool_close(p)
            print("ledger:", acc, "replayed %d requests" % len(calls))
            assert all(v > 100.0 for v in acc.values()), acc
        finally:
            arb.kill()
            arb.wait()


def test_modern_entry_points_on_real_driver():
    """cuLaunchKernelEx + cuMemAllocAsync/cuMemFreeAsync + cuStreamSynchronize against the real libcuda."""
    with tempfile.TemporaryDirectory() as tmp:
        res = storm(env_pool(tmp, quota="1\nbench/c0 1.0 1.0 5000\n", GEMHOOK_EXTRA_HOOKS=1), "--mode", "modern")
        st = stats(tmp)[0]
    assert st["launches"] == 100 and res["rc"] == [0, 0, 2]
    assert (res["free"], res["free_after"], res["total"]) == (2000, 4000, 5000)
    assert st["slow_path"] >= 5 and st["gpu_ns"] == st["gpu_ns_host"]
    # virtual memory management (PyTorch expandable segments): cuMemCreate is charged, cuMemRelease gives it back
    cap = 64 << 20
    with tempfile.TemporaryDirectory() as tmp:
        res = storm(env_pool(tmp, quota="1\nbench/c0 1.0 1.0 %d\n" % cap), "--mode", "modern")
    g = res["vmm"]["gran"]
    assert g >= 4096 and res["vmm"]["rc"] == [0, 2]                 # one granule fits, 4096 granules do not
    assert res["vmm"]["free_held"] == cap - 1000 - 3000 - g        # a (1000) and c (3000) are still allocated
    assert res["vmm"]["free_released"] == cap - 1000 - 3000


def test_pytorch_application_under_the_hook():
    """A real cudart application (PyTorch): cudart binds the driver through dlsym + cuGetProcAddress_v2, both
    interposed.  The gpu_mem cap shows up as torch's OOM, mem_get_info is virtualised, every kernel passes the gate."""
    import sys

    script = r'''
import json, sys, torch
x = torch.ones(1 << 20, device="cuda")
for _ in range(1500):
    x = x + 1
torch.cuda.synchronize()
free, total = torch.cuda.mem_get_info()
big = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")      # 1 GiB fits under the 2 GiB cap
oom = False
try:
    torch.empty(3 << 30, dtype=torch.uint8, device="cuda")          # 3 GiB does not
except torch.cuda.OutOfMemoryError:
    oom = True
print(json.dumps({"x0": float(x[0]), "total": total, "free_le_total": free <= total, "oom": oom}))
'''
    with tempfile.TemporaryDirectory() as tmp:
        env = env_pool(tmp, quota="1\nbench/c0 1.0 1.0 %d\n" % (2 << 30))
        p = sp.run([sys.executable, "-c", script], env=env, stdout=sp.PIPE, stderr=sp.PIPE, timeout=300)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        res = json.loads(p.stdout.decode().strip().splitlines()[-1])
        st = stats(tmp)[0]
    assert res["x0"] == 1501.0 and res["oom"] is True
    assert res["total"] == 2 << 30 and res["free_le_total"]
    assert st["launches"] >= 1500 and st["allocs_denied"] >= 1
    assert st["gpu_ns"] == st["gpu_ns_host"] > 0


def test_binding_paths_on_real_driver():
    """direct symbol, dlsym, cuGetProcAddress (legacy stream and per-thread stream) against the real libcuda."""
    with tempfile.TemporaryDirectory() as tmp:
        res = storm(env_pool(tmp, quota="1\nbench/c0 1.0 1.0 5000\n"), "--mode", "resolve")
        st = stats(tmp)[0]
    assert st["launches"] == 40 and res["gpa_is_hooked"] == 1 and res["ptsz_distinct"] == 1
    assert res["rc"] == [0, 0, 2] and (res["free"], res["total"]) == (2000, 5000)
