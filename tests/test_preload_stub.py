"""CPU: libgemhook.so.1 under LD_PRELOAD against the stub driver (tests/stub/libcuda.so.1).

BASELINE.json configs[0] (dry run: 1000 launches, quota-file parse), the three binding paths (direct
symbol, dlsym, cuGetProcAddress), the token protocol on the wire -- against a scripted fake pod manager
AND against the reference gem-pmgr + gem-schd, replayed from a recording of them serving this hook --, the gpu_mem
cap (config 4 sweep, bit-exact vs the oracle rule) and two co-resident clients arbitrating through the shared credit pool.
"""
import glob
import json
import os
import socket
import subprocess as sp
import tempfile
import threading
import time

import pytest

import kubeshare_b200 as kb
import orc
import wireproto as wp

LIVE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live_cpu.json")
GIB8 = 8589934592


def base_env(tmp, **kw):
    env = dict(os.environ)
    for k in list(env):
        if k.startswith("GEMHOOK_") or k in ("LD_PRELOAD", "POD_NAME", "POD_MANAGER_PORT"):
            env.pop(k)
    env["LD_LIBRARY_PATH"] = kb.STUB_DIR + ":" + env.get("LD_LIBRARY_PATH", "")
    env["STUB_REPORT"] = os.path.join(tmp, "stub.json")
    env.update({k: str(v) for k, v in kw.items()})
    return env


def hooked_env(tmp, pod="bench/c0", quota="1\nbench/c0 1.0 1.0 %d\n" % GIB8, **kw):
    with open(os.path.join(tmp, "quota.txt"), "w") as f:
        f.write(quota)
    return base_env(tmp, LD_PRELOAD=kb.LIB_PATH, GEMHOOK_POOL=os.path.join(tmp, "pool"),
                    GEMHOOK_QUOTA_FILE=os.path.join(tmp, "quota.txt"), POD_NAME=pod,
                    GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"), **kw)


def run_storm(env, *args, timeout=60):
    p = sp.run([kb.STORM_PATH, *map(str, args)], env=env, stdout=sp.PIPE, stderr=sp.PIPE, timeout=timeout)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return json.loads(p.stdout)


def stats_files(tmp):
    out = []
    for fn in sorted(os.listdir(tmp)):
        if fn.startswith("stats."):
            out.append(json.load(open(os.path.join(tmp, fn))))
    return out


def test_config1_dry_run_1000_launches():
    """configs[0]: single process, hook loaded, 1000 empty-kernel launches on the CPU-side stub."""
    with tempfile.TemporaryDirectory() as tmp:
        env = hooked_env(tmp, GEMHOOK_DRY_RUN=1)
        res = run_storm(env, "--mode", "storm", "--steps", 1, "--warmup", 0, "--step-launches", 1000, "--sync-every", 100)
        assert res["launches"] == 1000
        st = stats_files(tmp)[0]
        stub = json.load(open(os.path.join(tmp, "stub.json")))
        assert stub["launches"] == 1000           # every launch reached the driver exactly once
        assert st["launches"] == 1000 and st["pod"] == "bench/c0"
        assert st["slow_path"] == 10 and st["fast_path"] == 990   # one burst edge per sync interval
        assert st["token_requests"] >= 2          # the discarded first token + the first launch's (hook.cpp:766-768)
        assert st["mem_limit"] == GIB8            # quota-file parse
        assert st["acct_kernels"] == 0 and stub["event_records"] == 2  # dry run: only the app's own two events


def test_unknown_pod_exits_like_the_reference():
    with tempfile.TemporaryDirectory() as tmp:
        env = hooked_env(tmp, pod="bench/not-in-file")
        p = sp.run([kb.STORM_PATH, "--mode", "storm", "--steps", "1", "--warmup", "0", "--step-launches", "10"], env=env,
                   stdout=sp.PIPE, stderr=sp.PIPE, timeout=30)
        assert p.returncode != 0 and b"not in the quota file" in p.stderr
        env["GEMHOOK_EXIT_ON_FAILURE"] = "0"  # opt-out: run un-gated
        res = run_storm(env, "--mode", "storm", "--steps", 1, "--warmup", 0, "--step-launches", 10)
        assert res["launches"] == 10


def test_all_three_binding_paths_are_hooked():
    with tempfile.TemporaryDirectory() as tmp:
        env = hooked_env(tmp, quota="1\nbench/c0 1.0 1.0 5000\n")
        res = run_storm(env, "--mode", "resolve")
        st = stats_files(tmp)[0]
        assert st["launches"] == 40               # direct + dlsym + cuGetProcAddress_v2 (legacy and per-thread stream)
        assert res["gpa_is_hooked"] == 1 and res["ptsz_distinct"] == 1
        # cap 5000 B: 1000 ok, 2000 ok, 3000 denied (1000+2000+3000 > 5000) on the cuGetProcAddress path
        assert res["rc"] == [0, 0, 2]             # CUDA_ERROR_OUT_OF_MEMORY == 2
        assert (res["free"], res["total"]) == (2000, 5000)   # virtualised cuMemGetInfo
        assert st["allocs_denied"] == 1


def test_disabled_hook_is_transparent():
    with tempfile.TemporaryDirectory() as tmp:
        env = hooked_env(tmp, GEMHOOK_DISABLE=1)
        res = run_storm(env, "--mode", "resolve")
        assert res["rc"] == [0, 0, 0] and res["total"] == 180 << 30   # interposed, but every call passes straight through


# ------------------------------------------------------------------------------------------ wire / TCP
class FakePodManager(threading.Thread):
    """Scripted gem-pmgr: records every raw 80-byte request, answers like pod-manager.cpp would."""

    def __init__(self, limit, quota_ms):
        super().__init__(daemon=True)
        self.limit, self.quota_ms, self.used = limit, quota_ms, 0
        self.raw = []
        self.lsock = socket.socket()
        self.lsock.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
        self.lsock.bind(("127.0.0.1", 0))
        self.lsock.listen(4)
        self.port = self.lsock.getsockname()[1]

    def run(self):
        try:
            c, _ = self.lsock.accept()
            while True:
                buf = wp.recv_exact(c, wp.REQ_LEN)
                self.raw.append(buf)
                r = wp.unpack_request(buf)
                if r["type"] == wp.REQ_QUOTA:
                    c.sendall(wp.pack_response(wp.REQ_QUOTA, r["id"], quota=self.quota_ms))
                elif r["type"] == wp.REQ_MEM_LIMIT:
                    c.sendall(wp.pack_response(wp.REQ_MEM_LIMIT, r["id"], used=self.used, total=self.limit))
                else:
                    ok = 1
                    if r["alloc"]:
                        if self.used + r["bytes"] > self.limit:
                            ok = 0
                        else:
                            self.used += r["bytes"]
                    else:
                        self.used -= r["bytes"]
                    c.sendall(wp.pack_response(wp.REQ_MEM_UPDATE, r["id"], verdict=ok))
        except (ConnectionError, OSError):
            pass


def test_token_protocol_bytes_on_the_wire():
    pm = FakePodManager(limit=8192, quota_ms=50.0)
    pm.start()
    with tempfile.TemporaryDirectory() as tmp:
        env = base_env(tmp, LD_PRELOAD=kb.LIB_PATH, GEMHOOK_SCHEDULER_IP="127.0.0.1", POD_MANAGER_PORT=pm.port,
                       POD_NAME="default/mnist-pod-0123456789", GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"))
        res = run_storm(env, "--mode", "resolve")
        assert res["rc"] == [0, 0, 0] and res["total"] == 8192
    reqs = [wp.unpack_request(b) for b in pm.raw]
    assert all(len(b) == 80 for b in pm.raw)
    assert [r["id"] for r in reqs] == list(range(len(reqs)))          # per-process counter from 0 (comm.cpp:29, 62)
    assert all(r["name"] == "default/mnist-pod-0123456789" for r in reqs)
    # byte-identical to the reference layout (codec pinned against the reference's own bytes in test_oracle_golden)
    for raw, r in zip(pm.raw, reqs):
        assert raw == wp.pack_request(r["name"], r["id"], r["type"], r.get("overuse", 0.0), r.get("burst", 0.0),
                                      r.get("bytes", 0), r.get("alloc", 0))
    quotas = [r for r in reqs if r["type"] == wp.REQ_QUOTA]
    assert (quotas[0]["overuse"], quotas[0]["burst"]) == (0.0, 0.0)  # initialize(): first token, discarded
    assert (quotas[1]["overuse"], quotas[1]["burst"]) == (0.0, 0.0)  # first launch: nothing measured yet
    mem = [(r["bytes"], r["alloc"]) for r in reqs if r["type"] == wp.REQ_MEM_UPDATE]
    assert mem == [(1000, 1), (2000, 1), (3000, 1), (3000, 0), (2000, 0), (1000, 0)] or \
        mem[:3] == [(1000, 1), (2000, 1), (3000, 1)]


class ReplayPodManager(threading.Thread):
    """The reference gem-pmgr (+ gem-schd) as recorded serving this hook (tests/golden/ref_live_cpu.json, written by
    tests/golden/make_live_golden.py): the n-th connection replays the n-th recorded one.  Every memory request must be
    the one the reference daemons were sent at that point, with the id the hook's counter gives it, and gets the answer
    they gave.  Token renewals depend on timing, so one the recording lacks gets the last recorded quota and a recorded
    one the hook does not send is skipped."""

    FIELDS = {wp.REQ_QUOTA: ("quota",), wp.REQ_MEM_LIMIT: ("used", "total"), wp.REQ_MEM_UPDATE: ("verdict",)}

    def __init__(self, conns):
        super().__init__(daemon=True)
        self.conns, self.errors, self.served = conns, [], 0
        self.lsock = socket.socket()
        self.lsock.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
        self.lsock.bind(("127.0.0.1", 0))
        self.lsock.listen(4)
        self.port = self.lsock.getsockname()[1]

    def run(self):
        for rec in self.conns:
            try:
                c, _ = self.lsock.accept()
            except OSError:
                return
            with c:
                self._serve(c, rec)

    def _serve(self, c, rec):
        calls, k, n, quota = rec["calls"], 0, 0, None
        while True:
            try:
                r = wp.unpack_request(wp.recv_exact(c, wp.REQ_LEN))
            except (ConnectionError, OSError):
                break
            if r["name"] != rec["name"] or r["id"] != n:
                self.errors.append(("request %d" % n, r))
                return
            n += 1
            if r["type"] == wp.REQ_QUOTA:
                if k < len(calls) and calls[k][1] == wp.REQ_QUOTA:
                    quota = calls[k][3][0]
                    k += 1
                if quota is None:
                    self.errors.append(("token request the recording never answered", r))
                    return
                c.sendall(wp.pack_response(wp.REQ_QUOTA, r["id"], quota=quota))
                continue
            while k < len(calls) and calls[k][1] == wp.REQ_QUOTA:
                quota = calls[k][3][0]
                k += 1
            want = calls[k] if k < len(calls) else None
            got = [r["type"], [r["bytes"], r["alloc"]] if r["type"] == wp.REQ_MEM_UPDATE else []]
            if want is None or got != want[1:3]:
                self.errors.append(("memory request %d: sent %s, the reference daemons were sent %s" % (n - 1, got, want and want[1:3])))
                return
            c.sendall(wp.pack_response(r["type"], r["id"], **dict(zip(self.FIELDS[r["type"]], want[3]))))
            k += 1
        left = [x for x in calls[k:] if x[1] != wp.REQ_QUOTA]
        if left:
            self.errors.append("%d recorded memory requests never sent" % len(left))
        self.served += 1

    def check(self):
        self.lsock.close()
        self.join(timeout=10)
        assert not self.errors, self.errors
        assert self.served == len(self.conns), (self.served, len(self.conns))


def replayed(key, run):
    with open(LIVE) as f:
        rec = json.load(f)[key]["runs"][run]
    pm = ReplayPodManager(rec["conns"])
    pm.start()
    return pm, rec


def test_drop_in_against_live_reference_daemons():
    """Our hook speaking TCP to the UNMODIFIED gem-pmgr + gem-schd (recorded): tokens and the pod-wide memory cap."""
    with tempfile.TemporaryDirectory() as tmp:
        pm, rec = replayed("drop_in", 0)
        env = base_env(tmp, LD_PRELOAD=kb.LIB_PATH, GEMHOOK_SCHEDULER_IP="127.0.0.1", POD_MANAGER_PORT=pm.port,
                       POD_NAME="bench/c0", GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"))
        res = run_storm(env, *rec["args"])
        pm.check()
        assert res == rec["result"]
        assert res["rc"] == [0, 0, 2] and (res["free"], res["total"]) == (2000, 5000)
        pm, rec = replayed("drop_in", 1)
        env["POD_MANAGER_PORT"] = str(pm.port)
        res = run_storm(env, *rec["args"])
        pm.check()
        assert res["launches"] == rec["result"]["launches"] == 4000
        st = stats_files(tmp)[-1]
        assert st["token_requests"] >= 2 and st["quota_ms"] > 0


# ------------------------------------------------------------------------------------------ gpu_mem cap
def expected_sweep(limit, total_target):
    """Oracle rule applied to gem-storm's memsweep trace: allow iff bytes <= limit - used."""
    O = orc.load()
    used, first_fail, rows = 0, -1, []
    total, i = 0, 1
    while total < total_target and i < 512:
        sz = (256 << 20) * i
        ok = O.orc_mem_prehook_allows(sz, used, limit)
        if ok:
            used += sz
        elif first_fail < 0:
            first_fail = i
        rows.append((i, sz, 0 if ok else 2, limit - used))
        total += sz
        i += 1
    return rows, first_fail


def check_memsweep(res, limit):
    rows, first_fail = expected_sweep(limit, 40 << 30)
    got = [(r["i"], r["bytes"], r["rc"], r["free"]) for r in res["sweep1"]]
    assert got == rows
    assert res["first_fail"] == first_fail == 8        # 256 MiB * (1+..+7) = 7 GiB fits, +2 GiB does not
    assert all(r["total"] == limit for r in res["sweep1"])
    assert res["free_after_release"] == limit
    # sweep 2: 1000 odd sizes, never freed: replay the rule on the sizes the client reports
    O = orc.load()
    used = 0
    denied = 0
    for sz, rc, free in res["sweep2"]:
        ok = O.orc_mem_prehook_allows(sz, used, limit)
        assert rc == (0 if ok else 2)
        used += sz if ok else 0
        denied += 0 if ok else 1
        assert free == limit - used
    assert denied > 100 and res["free_end"] == limit


def test_config4_memory_cap_sweep_pool():
    with tempfile.TemporaryDirectory() as tmp:
        env = hooked_env(tmp)
        res = run_storm(env, "--mode", "memsweep")
        check_memsweep(res, GIB8)
        assert stats_files(tmp)[0]["mem_used"] == 0


def test_config4_memory_cap_sweep_against_live_gem_pmgr():
    with tempfile.TemporaryDirectory() as tmp:
        pm, rec = replayed("memsweep", 0)
        env = base_env(tmp, LD_PRELOAD=kb.LIB_PATH, GEMHOOK_SCHEDULER_IP="127.0.0.1", POD_MANAGER_PORT=pm.port,
                       POD_NAME="bench/c0")
        res = run_storm(env, *rec["args"])
        pm.check()
        assert res == rec["result"]
        check_memsweep(res, GIB8)


# ------------------------------------------------------------------------------------------ co-resident clients
def test_two_clients_share_one_token_through_the_pool():
    with tempfile.TemporaryDirectory() as tmp:
        quota = "2\nbench/c0 0.5 1.0 %d\nbench/c1 0.5 1.0 %d\n" % (GIB8, GIB8)
        procs = []
        for i in range(2):
            env = hooked_env(tmp, pod="bench/c%d" % i, quota=quota, GEMHOOK_BASE_QUOTA_MS=30, GEMHOOK_MIN_QUOTA_MS=5,
                             STUB_REPORT=os.path.join(tmp, "stub%d.json" % i))
            procs.append(sp.Popen([kb.STORM_PATH, "--mode", "storm", "--steps", "4", "--warmup", "1", "--step-launches", "20000",
                                   "--sync-every", "500", "--client-id", str(i), "--nclients", "2", "--barrier-dir", tmp,
                                   "--out", os.path.join(tmp, "out%d.json" % i)], env=env, stderr=sp.PIPE))
        for p in procs:
            _, err = p.communicate(timeout=120)
            assert p.returncode == 0, err.decode()[-1000:]
        st = stats_files(tmp)
        assert len(st) == 2 and all(s["launches"] == 100000 for s in st)
        assert all(s["token_requests"] >= 3 for s in st)       # both had to renew: the token really moved
        assert sum(s["token_wait_ms"] for s in st) > 10.0      # somebody waited while the other held it
        L = kb.lib()
        p = L.gemhook_pool_open(os.path.join(tmp, "pool").encode(), 0, 0, 0, 0, 0)
        assert p and L.gemhook_pool_nslots(p) == 2
        acc = [L.gemhook_pool_accumulated_ms(p, k) for k in range(2)]
        assert all(a > 0 for a in acc)
        L.gemhook_pool_close(p)


def test_modern_entry_points_are_gated_and_capped():
    """SURVEY.md 8f-2: cuLaunchKernelEx passes the token gate, stream-ordered allocations count against gpu_mem,
    cuStreamSynchronize is a burst edge only when GEMHOOK_EXTRA_HOOKS=1."""
    for extra, min_syncs, max_syncs in ((0, 0, 1), (1, 6, 12)):
        with tempfile.TemporaryDirectory() as tmp:
            env = hooked_env(tmp, quota="1\nbench/c0 1.0 1.0 5000\n", GEMHOOK_EXTRA_HOOKS=extra)
            res = run_storm(env, "--mode", "modern")
            st = stats_files(tmp)[0]
            assert st["launches"] == 100
            assert res["rc"] == [0, 0, 2] and (res["free"], res["total"]) == (2000, 5000)
            assert res["free_after"] == 4000        # cuMemFreeAsync gave the 2000 bytes back
            # cuMemCreate (stub granularity 1000 B): 1000 more fits (used 2000 of 5000), 4096 x 1000 does not
            assert res["vmm"]["rc"] == [0, 2] and res["vmm"]["free_held"] == 3000 and res["vmm"]["free_released"] == 4000
            assert st["allocs_denied"] == 2 and st["mem_used"] == 0
            assert min_syncs <= st["host_syncs"] <= max_syncs, st["host_syncs"]
            assert (st["slow_path"] >= 5) == bool(extra)   # every burst edge seen only with the extra hooks


def test_multithreaded_client_no_lost_launches_no_deadlock():
    """8 application threads launching on their own streams, syncing and allocating concurrently."""
    with tempfile.TemporaryDirectory() as tmp:
        env = hooked_env(tmp, GEMHOOK_BASE_QUOTA_MS=10, GEMHOOK_MIN_QUOTA_MS=2, GEMHOOK_SEG_MIN_US=100)
        res = run_storm(env, "--mode", "mt", "--nclients", 8, "--step-launches", 20000, timeout=120)
        st = stats_files(tmp)[0]
        stub = json.load(open(os.path.join(tmp, "stub.json")))
        assert res["launches"] == st["launches"] == 160000
        assert stub["launches"] >= 160000          # + our own reduce launches
        assert st["mem_used"] == 0 and st["allocs_denied"] == 0
        assert st["token_requests"] >= 3


def test_pitch_and_array_charges_follow_the_reference_byte_rules():
    """hook.cpp:629-680: pitch allocations are charged pitch*height with the REAL pitch, arrays W*H*[D*]C*fmt."""
    O = orc.load()
    with tempfile.TemporaryDirectory() as tmp:
        res = run_storm(hooked_env(tmp, quota="1\nbench/c0 1.0 1.0 5000\n"), "--mode", "arrays")
    pitch_bytes = res["pitch"] * 7
    a2 = O.orc_array_bytes(16, 8, 0, 4, 0x20, 0)
    a3 = O.orc_array_bytes(8, 4, 2, 2, 0x10, 1)
    assert (res["pitch"], pitch_bytes, a2, a3) == (512, 3584, 2048, 256)
    # 3584 fits in 5000; +2048 does not (denied, the driver is never asked); +256 fits
    assert res["rc"] == [0, 2, 0]
    assert res["free"] == [5000, 5000 - 3584, 5000 - 3584, 5000 - 3584 - 256, 5000 - 3584, 5000] and res["total"] == 5000


def test_yield_on_idle_hands_the_token_over_at_syncs():
    """Work-conserving option: with GEMHOOK_YIELD_ON_IDLE=1 a client that reaches a sync while another one waits
    returns the token instead of sitting on it until the quota expires (reference behaviour, default)."""
    results = {}
    for y in (0, 1):
        with tempfile.TemporaryDirectory() as tmp:
            quota = "2\nbench/c0 0.5 1.0 %d\nbench/c1 0.5 1.0 %d\n" % (GIB8, GIB8)
            procs = []
            for i in range(2):
                env = hooked_env(tmp, pod="bench/c%d" % i, quota=quota, GEMHOOK_YIELD_ON_IDLE=y, GEMHOOK_BASE_QUOTA_MS=200,
                                 GEMHOOK_MIN_QUOTA_MS=200, STUB_REPORT=os.path.join(tmp, "stub%d.json" % i))
                procs.append(sp.Popen([kb.STORM_PATH, "--mode", "bursty", "--rounds", "40", "--sleep-mean-ms", "3", "--client-id", str(i),
                                       "--nclients", "2", "--barrier-dir", tmp, "--out", os.path.join(tmp, "out%d.json" % i)],
                                      env=env, stderr=sp.PIPE))
            for p in procs:
                _, err = p.communicate(timeout=180)
                assert p.returncode == 0, err.decode()[-1000:]
            st = stats_files(tmp)
            wall = max(json.load(open(os.path.join(tmp, "out%d.json" % i)))["wall_s"] for i in range(2))
            results[y] = (wall, sum(s["yields"] for s in st), sum(s["token_requests"] for s in st))
    assert results[0][1] == 0 and results[1][1] >= 10          # tokens really changed hands at sync points
    assert results[1][2] > results[0][2]                         # ... which costs more (cheap) renewals
    assert results[1][0] < results[0][0] * 1.05                  # and never makes the pair slower


def test_two_processes_of_one_pod_share_the_pods_token():
    """Two processes with the SAME POD_NAME (one pod): gem-pmgr's pod-level token, one slot, one mailbox --
    neither may starve or hang when their requests collide."""
    with tempfile.TemporaryDirectory() as tmp:
        procs = []
        for i in range(2):
            env = hooked_env(tmp, pod="bench/c0", GEMHOOK_BASE_QUOTA_MS=5, GEMHOOK_MIN_QUOTA_MS=2,
                             STUB_REPORT=os.path.join(tmp, "stub%d.json" % i))
            procs.append(sp.Popen([kb.STORM_PATH, "--mode", "storm", "--steps", "6", "--warmup", "0", "--step-launches", "20000",
                                   "--sync-every", "250", "--out", os.path.join(tmp, "out%d.json" % i)], env=env, stderr=sp.PIPE))
        for p in procs:
            _, err = p.communicate(timeout=120)
            assert p.returncode == 0, err.decode()[-1000:]
        st = stats_files(tmp)
        assert len(st) == 2 and all(s["launches"] == 120000 for s in st)
        assert sum(s["token_requests"] for s in st) >= 4


def test_first_renewal_already_reports_a_doubled_burst():
    """A client that launches without idle gaps reports 2 x its measured burst from its first renewal on
    (estimate_full_burst, hook.cpp:402-417: the window predictor is below SCHD_OVERHEAD), so a lone tenant's quota grows
    by the x1.5 law of gem-schd's EMA (300 -> 448 -> 671 ... on the B200 with the reference hook).  The hook's own
    first-use initialisation -- which, unlike the reference's, runs at the first *launch*, after the application's first
    synchronising call opened a window -- must not be mistaken for application idle time: it once sat in the window
    predictor for 3 s and kept the estimate un-doubled (six 296 ms tokens where the reference had already reached 1 s).
    (Up to three attempts: on a busy machine the client can be descheduled for over 2 ms between a sync and the next launch,
    which IS an idle window and legitimately switches the doubling off for 3 s; the defect failed every time.)"""
    last = None
    for attempt in range(3):
        with tempfile.TemporaryDirectory() as tmp:
            env = hooked_env(tmp, GEMHOOK_BASE_QUOTA_MS=50, GEMHOOK_MIN_QUOTA_MS=20, GEMHOOK_TOKEN_TRACE=os.path.join(tmp, "trace.%d.jsonl"),
                             STUB_KERNEL_US=2, STUB_MODULE_LOAD_US=5000)   # a real driver loads the hook's cubin in milliseconds
            # the application synchronises once before its first launch (warm-up 0: barrier + cuCtxSynchronize, then launches)
            run_storm(env, "--mode", "storm", "--steps", 4, "--warmup", 0, "--step-launches", 65536, "--sync-every", 1024)
            tr = [json.loads(l) for f in glob.glob(os.path.join(tmp, "trace.*.jsonl")) for l in open(f)]
        assert len(tr) >= 4, tr
        # request 0: initialisation (burst 0); request 1: first launch (burst 0); request 2: after the first token was used up
        assert tr[0]["burst_ms"] == 0 and tr[1]["burst_ms"] == 0
        first = tr[2]
        assert first["quota_ms"] == pytest.approx(0.5 * first["burst_ms"] + 0.5 * 50, rel=1e-9)   # get_quota, scheduler.cpp:84-97
        last = tr[:4]
        if 1.8 * 50 <= first["burst_ms"] <= 2.1 * 50 and tr[3]["burst_ms"] > first["burst_ms"]:   # 2 x (a 50 ms token's worth)
            return
    raise AssertionError("burst estimate never doubled: %s" % (last,))


def test_ledger_time_covers_the_clients_own_unblocked_run_time():
    """The quantity the B200 parity tests compare between the stacks (tests/test_gpu_parity.py), on the CPU stub: per client,
    token time in the pool's ledger (last entry clipped at the client's own end stamp) over the time the client itself was
    not blocked in a launch (gem-storm --track-blocked: launch calls longer than 5 ms).  On hardware 0.995-1.002 in all three
    stacks; the stub's events report no overuse, so the drain after every expiry (~1 % here) is missing from the ledger."""
    import ctypes as C
    with tempfile.TemporaryDirectory() as tmp:
        quota = "2\nbench/c0 0.5 1.0 %d\nbench/c1 0.5 1.0 %d\n" % (GIB8, GIB8)
        procs = []
        for i in range(2):
            env = hooked_env(tmp, pod="bench/c%d" % i, quota=quota, GEMHOOK_BASE_QUOTA_MS=100, GEMHOOK_MIN_QUOTA_MS=20,
                             STUB_KERNEL_US=2, STUB_REPORT=os.path.join(tmp, "stub%d.json" % i))
            procs.append(sp.Popen([kb.STORM_PATH, "--mode", "storm", "--steps", "6", "--warmup", "0", "--step-launches", "65536",
                                   "--sync-every", "1024", "--track-blocked", "--client-id", str(i), "--nclients", "2",
                                   "--start-barrier-dir", tmp, "--out", os.path.join(tmp, "out%d.json" % i)], env=env, stderr=sp.PIPE))
        for p in procs:
            _, err = p.communicate(timeout=180)
            assert p.returncode == 0, err.decode()[-1000:]
        outs = [json.load(open(os.path.join(tmp, "out%d.json" % i))) for i in range(2)]
        L = kb.lib()
        p = L.gemhook_pool_open(os.path.join(tmp, "pool").encode(), 0, 0, 0, 0, 0)
        t0 = time.monotonic() - L.gemhook_pool_now_ms(p) / 1e3          # origin of the ledger's clock on CLOCK_MONOTONIC
        k = L.gemhook_pool_history(p, None, None, None, 0)
        sl, a, b = (C.c_int * k)(), (C.c_double * k)(), (C.c_double * k)()
        L.gemhook_pool_history(p, sl, a, b, k)
        for i in range(2):
            slot = L.gemhook_pool_find(p, ("bench/c%d" % i).encode())
            spans = [(a[j], b[j]) for j in range(k) if sl[j] == slot]
            exit_ms = (outs[i]["t_last"] - t0) * 1e3
            delivered = L.gemhook_pool_accumulated_ms(p, slot) - max(0.0, spans[-1][1] - max(exit_ms, spans[-1][0]))
            busy = (outs[i]["t_last"] - outs[i]["t_first"] - outs[i]["blocked_s"]) * 1e3
            assert outs[i]["blocked_s"] > 0.1, outs[i]["blocked_s"]              # it did wait for its peer's tokens
            assert 0.95 <= delivered / busy <= 1.03, (i, delivered, busy)
        L.gemhook_pool_close(p)
