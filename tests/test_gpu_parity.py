"""GPU: parity on the configurations the numbers are quoted on (VERDICT r1 items 1-2).

 * configs[1] (2 clients 0.5/0.5 storm) and configs[4] (4 clients 0.1/0.1/0.4/0.4 MNIST-shaped conv) through
   (a) the UNMODIFIED reference hook + gem-pmgr + gem-schd(_DEBUG) -- recorded on a B200 into
   tests/golden/ref_live_b200.json by tests/golden/make_live_golden.py, which runs this module's run_arm('reference') --,
   (b) our hook over TCP to gem-arbiter (the native gem-pmgr + gem-schd), (c) our hook on the credit pool; gem-schd's own
   ledger dump (scheduler.cpp:693-714) / gemhook_pool_history is the judge: per-client sum(end - start).
   HOW THE RELEASE-AT-EXIT DEVIATION IS EXCLUDED: a client that exits holding a token keeps it until the quota times
   out in the reference (scheduler.cpp:507-510) but hands it back in ours (DESIGN.md 4 (i)); that only ever affects
   the LAST token of a client, so in every arm a client's last ledger entry is clipped at the moment the client itself
   finished (its own CLOCK_MONOTONIC stamp; gem-schd's ledger counts from its process start on the same clock) -- what is compared
   is the token time each client was actually delivered while it ran.  (Dropping the last token instead does not
   work: adaptive quotas grow to ~1 s in a launch storm, so the used part of the last token varies by that much.)
   WHAT IS ASSERTED AT 1 %: ledger time delivered / the client's own un-blocked run time (gem-storm --track-blocked), stack
   against stack.  Absolute token time for a fixed amount of work also depends on how fast the device happened to serve
   that work (launch-queue regime, stalls while a token is held): +-7 % for the storm and single-client excursions of
   +2.7 % for the conv workload were seen in every stack, the reference included; the ratio is 0.994-0.997 (storm) and
   0.999-1.002 (conv) in all three stacks.  Clients are pinned to cores of their own and pass a barrier before the first
   interceptable call.
 * configs[2] (4 clients 0.25, bursty): every quota the scheduler policy granted equals the oracle's replay of
   get_quota (scheduler.cpp:160-174) over the (overuse, burst) sequence the client sent -- == on doubles.
 * the device-reduced SM-time against an independent truth: kernels that time themselves with %globaltimer.
"""
import ctypes as C
import glob
import json
import os
import signal
import subprocess as sp
import tempfile
import time

import pytest

import kubeshare_b200 as kb
import orc
import wireproto as wp
from test_gpu_hook import env_pool, stats, storm

pytestmark = pytest.mark.gpu
REF = os.path.join(kb.ROOT, "oracle", "_ref")   # the reference stack, where it is built (fixture generation only)
GIB8 = 8589934592
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live_b200.json")
CONFIG2 = ([0.5, 0.5], ["--mode", "storm", "--steps", 32, "--warmup", 0, "--step-launches", 65536, "--sync-every", 1024, "--track-blocked"])
CONFIG5 = ([0.1, 0.1, 0.4, 0.4], ["--mode", "mnist", "--iters", 400, "--track-blocked"])


def _kubeshare_dirs():
    """The reference hook reads its pod manager's address from /kubeshare/library/schedulerIP.txt (reference hook.cpp:162,
    233-237); oracle/ref_compat.h lets REF_KUBESHARE_ROOT stand in for /kubeshare, so no root is needed."""
    if "REF_KUBESHARE_ROOT" not in os.environ:
        root = tempfile.mkdtemp(prefix="ref_kubeshare_")
        os.makedirs(os.path.join(root, "library"))
        os.makedirs(os.path.join(root, "log"))
        with open(os.path.join(root, "library", "schedulerIP.txt"), "w") as f:
            f.write("127.0.0.1\n")
        os.environ["REF_KUBESHARE_ROOT"] = root


def _delivered(spans_by_client, outs, schd_t0):
    """Per client: token time delivered = sum(end - start) over its ledger entries, the LAST one clipped at the moment
    the client finished.  gem-schd counts milliseconds since its own process start on steady_clock (scheduler.cpp:97,
    107-109) = CLOCK_MONOTONIC, the clock of the clients' stamps and of time.monotonic(): `schd_t0` is the monotonic time
    at which the test started gem-schd (good to a few ms, on totals of seconds)."""
    out = {}
    for c, v in spans_by_client.items():
        exit_ms = (outs[c]["t_last"] - schd_t0) * 1e3
        out[c] = sum(e - s for s, e in v[:-1]) + max(0.0, min(v[-1][1], exit_ms) - v[-1][0]) if v else 0.0
    return out, {c: len(v) for c, v in spans_by_client.items()}


def _core_sets():
    """Hyper-thread sibling sets of the physical cores this process may use: every client gets a core of its own (both
    siblings, so the hook's tracker thread has somewhere to run); two launch storms sharing a core slow each other."""
    seen, out = set(), []
    for c in sorted(os.sched_getaffinity(0)):
        try:
            sib = open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c).read().strip()
        except OSError:
            sib = str(c)
        if sib in seen:
            continue
        seen.add(sib)
        cpus = set()
        for part in sib.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        out.append(cpus & set(os.sched_getaffinity(0)) or {c})
    return out


def run_arm(which, fracs, wargs, timeout=900, extra_env=None):
    """One co-resident run.  which: 'reference' (the reference stack from oracle/_ref) | 'ours-tcp' (our hook over TCP to
    gem-arbiter) | 'pool'.  Returns {client: [(start_ms, end_ms)...]}, per-client outputs, hook stats."""
    n = len(fracs)
    quota = "%d\n" % n + "".join("bench/c%d %r 1.0 %d\n" % (i, f, GIB8) for i, f in enumerate(fracs))
    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "quota.txt"), "w") as f:
            f.write(quota)
        base = {k: v for k, v in os.environ.items() if not k.startswith("GEMHOOK_") and k not in ("LD_PRELOAD", "POD_NAME")}
        daemons, ports, schd, schd_t0 = [], [], None, None
        try:
            if which == "ours-tcp":
                aport = wp.free_port()
                alog = os.path.join(tmp, "arbiter.log")
                with open(alog, "w") as f:
                    daemons.append(sp.Popen([os.path.join(kb.HERE, "bin", "gem-arbiter"), "--pool", os.path.join(tmp, "pool"), "-p", tmp,
                                             "-f", "quota.txt", "-P", str(aport), "-q", "300", "-m", "20", "-w", "10000"], stderr=f))
                deadline = time.time() + 10
                while time.time() < deadline and "listening" not in open(alog).read():
                    time.sleep(0.05)
                ports = [aport] * n
            elif which == "reference":
                _kubeshare_dirs()
                sport = wp.free_port()
                t_before = time.monotonic()
                schd = sp.Popen([os.path.join(REF, "gem-schd-dbg"), "-p", tmp, "-f", "quota.txt", "-P", str(sport), "-q", "300", "-m", "20",
                                 "-w", "10000", "-v", "1"], cwd=tmp, stdout=sp.DEVNULL, stderr=sp.DEVNULL)
                schd_t0 = 0.5 * (t_before + time.monotonic()) + 0.001   # its static initialisers run ~1 ms after exec
                daemons.append(schd)
                time.sleep(0.5)
                for i in range(n):
                    ports.append(wp.free_port())
                    daemons.append(sp.Popen([os.path.join(REF, "gem-pmgr")], stdout=sp.DEVNULL, stderr=sp.DEVNULL,
                                            env=dict(base, POD_NAME="bench/c%d" % i, POD_MANAGER_PORT=str(ports[i]),
                                                     SCHEDULER_IP="127.0.0.1", SCHEDULER_PORT=str(sport))))
                time.sleep(0.5)
            procs = []
            for i in range(n):
                e = dict(base, POD_NAME="bench/c%d" % i)
                if which == "reference":
                    e.update(LD_PRELOAD=os.path.join(REF, "libgemhook_ref.so.1"), POD_MANAGER_PORT=str(ports[i]))
                elif which == "ours-tcp":
                    e.update(LD_PRELOAD=kb.LIB_PATH, GEMHOOK_SCHEDULER_IP="127.0.0.1", POD_MANAGER_PORT=str(ports[i]),
                             GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"), GEMHOOK_TOKEN_TRACE=os.path.join(tmp, "trace.%d.jsonl"))
                else:
                    e.update(LD_PRELOAD=kb.LIB_PATH, GEMHOOK_POOL=os.path.join(tmp, "pool"), GEMHOOK_QUOTA_FILE=os.path.join(tmp, "quota.txt"),
                             GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json"), GEMHOOK_TOKEN_TRACE=os.path.join(tmp, "trace.%d.jsonl"))
                    e.update({k: str(v) for k, v in (extra_env or {}).items()})
                # No barrier once tokens exist: a client that waits at a barrier sits on its token (up to a whole quota) while
                # its peer cannot move -- idle-hold time that varies from run to run and is not what is being compared.  But
                # one BEFORE the first call any hook intercepts: a peer that is still creating its context stalls the device
                # for the client that already runs on a token (50-120 ms of ledger time without progress, in any stack).
                cores = _core_sets()
                cpus = cores[(1 + i) % len(cores)] if len(cores) > n + 1 else None
                procs.append(sp.Popen([kb.STORM_PATH, *map(str, wargs), "--client-id", str(i), "--nclients", str(n),
                                       "--start-barrier-dir", tmp, "--out", os.path.join(tmp, "out%d.json" % i)], env=e, stderr=sp.PIPE,
                                      preexec_fn=(lambda c=cpus: os.sched_setaffinity(0, c)) if cpus else None))
            for p in procs:
                _, err = p.communicate(timeout=timeout)
                assert p.returncode == 0, err.decode()[-1500:]
            outs = [json.load(open(os.path.join(tmp, "out%d.json" % i))) for i in range(n)]
            spans = {i: [] for i in range(n)}
            if which != "reference":   # the credit pool's ledger (gem-arbiter keeps its ledger in the same pool)
                L = kb.lib()
                p = L.gemhook_pool_open(os.path.join(tmp, "pool").encode(), 0, 0, 0, 0, 0)
                k = L.gemhook_pool_history(p, None, None, None, 0)
                sl, a, b = (C.c_int * k)(), (C.c_double * k)(), (C.c_double * k)()
                L.gemhook_pool_history(p, sl, a, b, k)
                names = {L.gemhook_pool_find(p, ("bench/c%d" % i).encode()): i for i in range(n)}
                acc = {i: L.gemhook_pool_accumulated_ms(p, s_) for s_, i in names.items()}
                schd_t0 = time.monotonic() - L.gemhook_pool_now_ms(p) / 1e3   # the pool ledger's origin on CLOCK_MONOTONIC
                L.gemhook_pool_close(p)
                for j in range(k):
                    spans[names[sl[j]]].append((a[j], b[j]))
                spans["accumulated_ms"] = acc   # full history (the ledger proper is pruned to the 10 s window)
            else:
                time.sleep(0.2)
                schd.send_signal(signal.SIGINT)
                schd.wait(timeout=20)
                dumps = [d for d in glob.glob(os.path.join(tmp, "*.json")) if os.path.basename(d)[0].isdigit()]
                assert dumps, "gem-schd did not dump its ledger"
                for e in json.load(open(dumps[0])):
                    spans[int(e["container"].rsplit("c", 1)[1])].append((e["start"] * 1e3, e["end"] * 1e3))
            trace = [json.loads(l) for f in sorted(glob.glob(os.path.join(tmp, "trace.*.jsonl"))) for l in open(f)]
            if schd_t0 is not None:
                spans["schd_t0"] = schd_t0
            return spans, outs, stats(tmp), trace
        finally:
            for d in daemons:
                if d.poll() is None:
                    d.kill()
                d.wait()


def arm_result(which, fracs, wargs):
    """run_arm + the per-client figures the parity tests compare (lists indexed by client)."""
    spans, outs, st, _ = run_arm(which, fracs, wargs)
    acc = spans.pop("accumulated_ms", None)
    t0_ = spans.pop("schd_t0")
    n = len(outs)
    if acc is not None:
        # pool: a client hands its token back when its process exits -- after its own end stamp by however long the
        # teardown (context destroy, with peers still running) takes.  Same clipping as for the gem-schd ledgers: the
        # part of the client's last entry that lies after its own end stamp is not token time "while it ran".
        delivered, tokens = {}, {c: None for c in acc}
        for c in acc:
            exit_ms = (outs[c]["t_last"] - t0_) * 1e3
            over = max(0.0, spans[c][-1][1] - max(exit_ms, spans[c][-1][0])) if spans[c] else 0.0
            delivered[c] = acc[c] - over
        print("ledger %s: overhang after the client's own end" % which, {c: round(acc[c] - delivered[c], 1) for c in acc})
    else:
        delivered, tokens = _delivered(spans, outs, t0_)
        print("ledger %s:" % which, {c: [(round(s_), round(e_)) for s_, e_ in v] for c, v in spans.items()},
              "exits", [round((o["t_last"] - t0_) * 1e3) for o in outs], "first launches", [round((o["t_first"] - t0_) * 1e3) for o in outs])
    res = {"delivered_ms": [delivered[c] for c in range(n)], "tokens": [tokens[c] for c in range(n)],
           "wall_s": [round(o["wall_s"], 3) for o in outs], "launches": [o["launches"] for o in outs]}
    if "--track-blocked" in wargs:   # gem-storm --track-blocked: the client's own un-blocked run time
        busy = [(o["t_last"] - o["t_first"] - o["blocked_s"]) * 1e3 for o in outs]
        res["busy_ms"] = [round(b, 1) for b in busy]
        res["coverage"] = [delivered[c] / busy[c] for c in range(n)]
    return res


def _three_arms(key, fracs, wargs):
    """The reference stack's figures as recorded on a B200, next to our two stacks run now."""
    res = {"reference": json.load(open(GOLDEN))[key]}
    for which in ("ours-tcp", "pool"):
        res[which] = arm_result(which, fracs, wargs)
    print("ledgers:", json.dumps(res))
    return res


def test_config2_two_client_ledger_split_matches_reference():
    """configs[1], the headline config: 2 x 0.5, 32 x 65536 noop launches each, sync every 1024.

    WHAT IS COMPARED.  A noop storm is bound by the driver's launch queue, and how fast that queue is served depends on how
    the launching thread is paced: the same un-hooked storm runs at 486.8 K launches/s when it outruns the GPU front end
    and at 506-524 K/s with 160-240 ns of extra host time per launch (profiles/r02_launch_rate_vs_host_pace.txt).  The
    reference hook adds about that much, ours 2 ns, so "token time needed for 2^21 launches" differs between the stacks by
    up to 7 % from run to run for a reason that has nothing to do with either ledger.  Each client therefore also measures
    on its own clock the time it was NOT blocked waiting for a token (gem-storm --track-blocked: launch calls over 5 ms);
    per client and stack, ledger time delivered / un-blocked run time is the figure of merit -- what fraction of the time
    the client really ran is covered by tokens in that stack's ledger -- and it has to agree within 1 % between the
    reference stack and ours (measured: 0.9947-0.9970 in all three stacks, 3 repetitions)."""
    res = _three_arms("config2", *CONFIG2)
    # The two clients are identical (same fraction, same work); which of them wins the very first token is a coin toss,
    # so the comparison is between the SORTED per-client figures, not between labels.
    ref = sorted(res["reference"]["coverage"])
    for arm in ("ours-tcp", "pool"):
        got = sorted(res[arm]["coverage"])
        for g, r in zip(got, ref):
            assert abs(g - r) <= 0.01, (arm, got, ref)           # same share of the run covered by ledger time, within 1 %
            assert 0.98 <= g <= 1.01 and 0.98 <= r <= 1.01       # and the ledger neither invents nor loses run time
    # (absolute token time is printed, not asserted: on one box and in one stack it moved between 4140 and 4750 ms from run
    #  to run with the launch rate the driver's queue happened to settle at -- 441 to 507 K launches/s)


def test_config5_four_client_mixed_fraction_ledger_matches_reference():
    """configs[4] on one device: min-fractions 0.1/0.1/0.4/0.4, MNIST-shaped conv, 400 iterations x 100 launches.
    40 000 launches per client (~5.4 s of GPU work each, 22 s per arm).  GPU-bound, so here absolute token time is
    comparable between the stacks; but in every stack (the reference included: 5547 ms next to 5413-5428) one client in a
    few runs is delivered 70-130 ms more than its peers for the same work -- the device made no progress for it while it
    held a token.  As in the storm test the client's own un-blocked run time tells the two apart: ledger time / un-blocked
    time agrees within 1 % between the stacks (the strict assertion); absolute time within 5 % per client and 2.5 % in
    total (the largest excursion seen in 14 runs: +2.7 % for one client, in the reference stack)."""
    res = _three_arms("config5", *CONFIG5)
    # Clients of one fraction class are interchangeable (first-token coin toss), so classes are compared sorted.
    ref = res["reference"]
    tot_ref = sum(ref["delivered_ms"])
    for arm in ("ours-tcp", "pool"):
        got = res[arm]
        tot = sum(got["delivered_ms"])
        assert abs(tot - tot_ref) <= 0.025 * tot_ref, (arm, tot, tot_ref)   # the same work holds the GPU equally long
        for cls in ((0, 1), (2, 3)):
            g = sorted(got["delivered_ms"][c] for c in cls)
            r = sorted(ref["delivered_ms"][c] for c in cls)
            for a, b in zip(g, r):
                assert abs(a - b) <= 0.05 * b, (arm, cls, g, r)
            gc = sorted(got["coverage"][c] for c in cls)
            rc = sorted(ref["coverage"][c] for c in cls)
            for a, b in zip(gc, rc):
                assert abs(a - b) <= 0.01, (arm, cls, gc, rc)           # ledger time per un-blocked run time: within 1 %
                assert 0.98 <= a <= 1.02 and 0.98 <= b <= 1.02
        # and the shares bite the same way: the 0.4 clients are done well before the 0.1 clients in every arm
        assert max(got["wall_s"][2:]) < min(got["wall_s"][:2]) and max(ref["wall_s"][2:]) < min(ref["wall_s"][:2])


def test_config3_quota_sequence_equals_oracle_ema_replay():
    """configs[2]: 4 x 0.25 bursty trace.  For every request the pool forwarded to the scheduler policy the granted
    quota must equal get_quota (scheduler.cpp:160-174) replayed by the ORACLE over the same (overuse, burst) sequence."""
    O = orc.load()
    spans, outs, st, trace = run_arm("pool", [0.25] * 4, ["--mode", "bursty", "--rounds", 150])
    assert len(st) == 4 and len(trace) >= 8
    checked = 0
    for pod in sorted({t["pod"] for t in trace}):
        seq = [t for t in trace if t["pod"] == pod]
        h = O.orc_schd_new(300.0, 20.0, 10000.0)
        O.orc_schd_set_client(h, pod.encode(), 0.25, 1.0, GIB8)
        try:
            fwd = [t for t in seq if t["forwarded"] == 1]
            assert len(fwd) >= 2
            for k, t in enumerate(fwd):
                O.orc_schd_request(h, pod.encode(), float(k), t["overuse_ms"], t["burst_ms"])
                want = O.orc_schd_grant(h, pod.encode(), float(k))
                assert t["quota_ms"] == want, (pod, k, t, want)      # == on doubles
                checked += 1
            # requests the pod-level rule answered locally got the REMAINING pod quota: below the last full quota
            last = None
            for t in seq:
                if t["forwarded"] == 1:
                    last = t["quota_ms"]
                elif last is not None:
                    assert t["quota_ms"] <= last
        finally:
            O.orc_schd_free(h)
    for s in st:   # token renewals happen only at burst edges
        assert s["token_requests"] <= s["slow_path"] + 1 and s["slow_path"] <= 150 + s["token_requests"] + 2
    print("EMA replay: %d forwarded requests equal the oracle" % checked)


def test_yield_on_idle_keeps_the_ledger_rules():
    """GEMHOOK_YIELD_ON_IDLE=1 (off by default) changes WHEN tokens move, not the rules they move by: every quota the
    policy grants still equals the oracle's get_quota replay, tokens never overlap, nobody starves, and each client is
    delivered at least the SM-time it actually used."""
    O = orc.load()
    spans, outs, st, trace = run_arm("pool", [0.25] * 4, ["--mode", "bursty", "--rounds", 150], extra_env={"GEMHOOK_YIELD_ON_IDLE": 1})
    acc = spans.pop("accumulated_ms")
    spans.pop("schd_t0", None)
    assert sum(s["yields"] for s in st) >= 20, "the option never fired: %s" % [s["yields"] for s in st]
    for pod in sorted({t["pod"] for t in trace}):
        h = O.orc_schd_new(300.0, 20.0, 10000.0)
        O.orc_schd_set_client(h, pod.encode(), 0.25, 1.0, GIB8)
        try:
            for k, t in enumerate(x for x in trace if x["pod"] == pod and x["forwarded"] == 1):
                O.orc_schd_request(h, pod.encode(), float(k), t["overuse_ms"], t["burst_ms"])
                assert t["quota_ms"] == O.orc_schd_grant(h, pod.encode(), float(k)), (pod, k, t)
        finally:
            O.orc_schd_free(h)
    # one outstanding token: entries overlap only by a client's overuse (the scheduler splits that overlap, scheduler.cpp:342-367)
    flat = sorted((s, e) for c, v in spans.items() for s, e in v)
    overlap = sum(max(0.0, flat[i][1] - flat[i + 1][0]) for i in range(len(flat) - 1))
    assert overlap <= 0.02 * sum(e - s for s, e in flat), (overlap, len(flat))
    by_pod = {s["pod"]: s for s in st}
    for i in range(4):
        used_ms = by_pod["bench/c%d" % i]["gpu_ns"] / 1e6
        assert acc[i] >= 0.98 * used_ms, (i, acc[i], used_ms)              # token time covers the SM-time consumed
    busy = [s["gpu_ns"] for s in st]
    assert min(busy) > 0.3 * max(busy)
    print("yield-on-idle: %d yields, delivered %s ms, used %s ms" % (sum(s["yields"] for s in st), [round(acc[i]) for i in range(4)],
                                                                    [round(by_pod["bench/c%d" % i]["gpu_ns"] / 1e6) for i in range(4)]))


# ------------------------------------------------------------------------------------------------ SM-time truth
TRUTH_CASES = [
    # (name, env, rounds, launches/burst, spin us, idle ms, streams)
    ("merged: 1.5 ms bursts, 0.3 ms idle gaps, SEG_MIN 4 ms", {}, 300, 150, 10, 0.3, 1),
    ("merged: back-to-back 1 ms bursts", {}, 400, 100, 10, 0.0, 1),
    ("SEG_LAUNCHES=256 inside 8 ms bursts", {"GEMHOOK_SEG_LAUNCHES": 256}, 80, 1024, 8, 0.2, 1),
    ("two non-blocking streams", {}, 200, 400, 10, 0.3, 2),
    ("unmerged: every burst its own segment", {"GEMHOOK_SEG_MIN_US": 0}, 200, 200, 10, 0.3, 1),
]


@pytest.mark.parametrize("case", TRUTH_CASES, ids=[c[0] for c in TRUTH_CASES])
def test_device_sm_time_within_1pct_of_in_kernel_globaltimer_truth(case):
    """The kernels measure themselves: every spin kernel folds its own %globaltimer start/end into the bounds of its
    burst; truth = sum over bursts of (latest end - earliest start).  The hook never sees those numbers; its gpu_ns
    comes from event pairs, host-measured idle subtraction and the sm_100a reduction."""
    name, extra, rounds, per, spin, idle, streams = case
    with tempfile.TemporaryDirectory() as tmp:
        res = storm(env_pool(tmp, GEMHOOK_FLUSH_RECORDS=8, **extra), "--mode", "truth", "--rounds", rounds, "--step-launches", per,
                    "--spin-us", spin, "--sleep-mean-ms", idle, "--nclients", streams)
        st = stats(tmp)[0]
    truth, got = res["truth_ns"], st["gpu_ns"]
    print("truth %s: truth %.3f ms, hook %.3f ms, ratio %.5f, segments %d" % (name, truth / 1e6, got / 1e6, got / truth, st["segments"]))
    assert st["gpu_ns"] == st["gpu_ns_host"]
    assert abs(got - truth) <= 0.01 * truth, (name, got, truth, got / truth)


def test_live_scrape_sees_growing_gpu_seconds():
    """f3: gem-poolctl prom WHILE a storm runs shows a growing gemhook_gpu_seconds_total that ends within 1 % of the
    client's own final figure (published on every flush, not only at exit; no GEMHOOK_STATS_FILE needed for it)."""
    poolctl = os.path.join(kb.HERE, "bin", "gem-poolctl")
    with tempfile.TemporaryDirectory() as tmp:
        env = env_pool(tmp, GEMHOOK_FLUSH_RECORDS=8)
        p = sp.Popen([kb.STORM_PATH, "--mode", "storm", "--steps", "40", "--warmup", "1", "--step-launches", "65536"], env=env,
                     stdout=sp.PIPE, stderr=sp.PIPE)
        seen = []
        while p.poll() is None:
            if os.path.exists(os.path.join(tmp, "pool")):
                q = sp.run([poolctl, os.path.join(tmp, "pool"), "prom"], stdout=sp.PIPE, stderr=sp.DEVNULL)
                for line in q.stdout.decode().splitlines():
                    if line.startswith("gemhook_gpu_seconds_total{"):
                        seen.append(float(line.split()[-1]))
            time.sleep(0.25)
        out, err = p.communicate()
        assert p.returncode == 0, err.decode()[-1000:]
        final = stats(tmp)[0]["gpu_ns"] / 1e9
        q = sp.run([poolctl, os.path.join(tmp, "pool"), "prom"], stdout=sp.PIPE)
        end = [float(l.split()[-1]) for l in q.stdout.decode().splitlines() if l.startswith("gemhook_gpu_seconds_total{")][0]
        led = sp.run([poolctl, os.path.join(tmp, "pool"), "ledger"], stdout=sp.PIPE)
        ledger = json.loads(led.stdout)
    live = sorted(set(v for v in seen if v > 0))
    print("live scrape:", live[:3], "...", live[-3:], "final", final)
    assert len(live) >= 4 and seen == sorted(seen), "gpu seconds must grow while the client runs"
    assert live[0] < 0.5 * final
    assert abs(end - final) <= 0.01 * final
    # the alternative output: gem-schd's _DEBUG dump shape (scheduler.cpp:693-714)
    assert ledger and set(ledger[0]) == {"container", "start", "end"} and ledger[0]["container"] == "bench/c0"


def test_cuda_graph_capture_and_replay_under_the_hook():
    """ADVICE r1 (medium): a capture must never see our events.  Driver API (gem-storm --mode graph, tokens expiring
    during the capture) and torch.cuda.graph()."""
    import sys

    with tempfile.TemporaryDirectory() as tmp:
        env = env_pool(tmp, GEMHOOK_BASE_QUOTA_MS=5, GEMHOOK_MIN_QUOTA_MS=2, GEMHOOK_SEG_MIN_US=100, GEMHOOK_SEG_LAUNCHES=16)
        res = storm(env, "--mode", "graph", "--step-launches", 64, "--rounds", 20, "--spin-us", 20)
        st = stats(tmp)[0]
    assert [res[k] for k in ("begin", "launch", "end", "instantiate", "replay", "sync", "destroy")] == [0] * 7, res
    assert res["nodes"] == 64, "our events must not become nodes of the application's graph: %s" % res
    print("graph replays: app-side events %.3f ms, hook %.3f ms" % (res["replay_ms"], st["gpu_ns"] / 1e6))
    assert st["gpu_ns"] == st["gpu_ns_host"] >= 0.95 * res["replay_ms"] * 1e6   # the replays were accounted
    script = r'''
import json, torch
x = torch.zeros(1 << 16, device="cuda")
s = torch.cuda.Stream()
with torch.cuda.stream(s):
    for _ in range(3):
        x += 1
torch.cuda.current_stream().wait_stream(s)
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    for _ in range(50):
        x += 1
for _ in range(40):
    g.replay()
torch.cuda.synchronize()
print(json.dumps({"x0": float(x[0])}))
'''
    with tempfile.TemporaryDirectory() as tmp:
        env = env_pool(tmp, GEMHOOK_BASE_QUOTA_MS=5, GEMHOOK_MIN_QUOTA_MS=2, GEMHOOK_SEG_MIN_US=100)
        p = sp.run([sys.executable, "-c", script], env=env, stdout=sp.PIPE, stderr=sp.PIPE, timeout=300)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        assert json.loads(p.stdout.decode().strip().splitlines()[-1])["x0"] == 3 + 40 * 50   # (captured launches do not execute)
        assert stats(tmp)[0]["gpu_ns"] > 0
