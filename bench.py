#!/usr/bin/env python
"""bench.py -- hook overhead % and launches/s at 1/2/4/8 co-resident clients vs un-hooked (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # our hook (libgemhook.so.1, credit pool)
    python bench.py --impl reference --gpus N ...            # the UNMODIFIED reference hook + gem-pmgr + gem-schd
                                                             # (oracle/_ref, built from /root/reference)
    python bench.py --workload bursty|mnist ...              # BASELINE configs[2] / configs[4], same one-line schema
    python bench.py ... --dump-outputs DIR                   # + what the timed path computed in its last step, as .npy

A "step" is one pass of the hot path over one batch of synthetic input: every co-resident client issues
STEP_LAUNCHES (65536) launches of noop<<<1,32>>> on the default stream with cuCtxSynchronize every 1024
(SURVEY.md 8d config 2).  The headline workload is BASELINE.json configs[1]: 2 clients, gpu_request 0.5 each, on
one B200; the 1/2/4/8 client sweep is reported under "clients".  Each client is a separate process
(kubeshare_b200/bin/gem-storm, CUDA driver API) -- exactly how pods share a GPU -- pinned to its own host core.

  value      aggregate hooked launches/s, timed on the device with CUDA events around the K timed steps in
             every client (max over clients and ranks); median over --reps repetitions of the K-step run
  e2e        the same launches through the LD_PRELOAD boundary timed on the host clock from the first
             client's start to the last client's end, including the accounting traffic inside the steps
  roofline   the sm_100a accounting kernel (gemhook_acct_reduce) on a 2^26-record (1 GiB > L2) device-resident
             ring, CUDA events on the accounting stream, algorithmic bytes = 16 B/record
  cpu_baseline        the reference hook stack on the same box, same workload, same K/W, same timing
  cpu_baseline_debug  the reference as KubeShare ships it (DEBUG=1 hook, _DEBUG gem-schd), bounded sample, with
                      the per-client ledger split gem-schd dumps (scheduler.cpp:693-714)

Multi-GPU: the path does not shard (one gem-scheduler + hook set per device, SURVEY.md 8e): --gpus N runs N
independent replicas, one rank per GPU, no collective in the data path; value sums the replicas' launches
over the slowest replica's time.  The reference arm runs on rank 0 alone (contract) and drives its N replicas
from that one process.

The JSON line stays small: per-process hook statistics go to a side file, bench_detail_*.json in the --dump-outputs
directory (or in a fresh temporary directory, named on stderr), and the line carries only a summary.  The benchmark
runs from the tree as __graft_entry__.build() left it and writes nothing into it.

--dump-outputs DIR writes, after the timed steps, what a caller of the timed path receives from its last step:
  acct_totals_<ring>.npy     float64 [nslots, 3] (SM-time ns, launches, records per client slot) that the last timed
                             gemhook_acct_reduce launch added on each roofline ring (inputs are a fixed function of the
                             ring index, identical from run to run)
  hooked_launches.npy        float64 [clients]: launches the hook intercepted in each client of the headline run
                             (median repetition), warm-up included
"""
import argparse
import glob
import json
import os
import shutil
import signal
import statistics
import subprocess as sp
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
STORM = os.path.join(ROOT, "kubeshare_b200", "bin", "gem-storm")
HOOK = os.environ.get("GEMBENCH_HOOK") or os.path.join(ROOT, "kubeshare_b200", "lib", "libgemhook.so.1")  # (override: A/B runs)
REFDIR = os.path.join(ROOT, "oracle", "_ref")
STEP_LAUNCHES = int(os.environ.get("GEMBENCH_STEP_LAUNCHES", "65536"))  # override only for the CPU stub tests
SYNC_EVERY = 1024
GIB8 = 8589934592
SCHD_ARGS = ["-q", "300", "-m", "20", "-w", "10000"]  # reference launcher.py:77-80 defaults


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling DURING the timed regions (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu = gpu
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = sp.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                  "--format=csv,noheader,nounits", "-lms", "200"], stdout=sp.PIPE, stderr=sp.DEVNULL,
                                 text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except sp.TimeoutExpired:
                self.proc.kill()

    def summary(self, windows):
        sm, mx, reasons = [], 0.0, set()
        for ts, line in self.rows:
            if windows and not any(a <= ts <= b for a, b in windows):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------- host cores
def free_ports(n):
    """n distinct currently-free TCP ports (fresh per run: gem-schd binds without SO_REUSEADDR)."""
    import socket

    socks = []
    for _ in range(n):
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        socks.append(s)
    ports = [s.getsockname()[1] for s in socks]
    for s in socks:
        s.close()
    return ports


_PHYS = None


def physical_cores():
    """One logical CPU per physical core (first hyper-thread sibling), so pinned clients never share a core."""
    global _PHYS
    if _PHYS is None:
        seen, out = set(), []
        try:
            avail = sorted(os.sched_getaffinity(0))
        except AttributeError:
            avail = list(range(os.cpu_count() or 1))
        for c in avail:
            try:
                sib = open("/sys/devices/system/cpu/cpu%d/topology/thread_siblings_list" % c).read().strip()
            except OSError:
                sib = str(c)
            if sib not in seen:
                seen.add(sib)
                out.append(c)
        _PHYS = out or avail
    return _PHYS


def pin(core):
    """`core` is an index into the list of physical cores (wraps around)."""
    phys = physical_cores()
    cpu = phys[core % len(phys)]

    def f():
        try:
            os.sched_setaffinity(0, {cpu})
        except OSError:
            pass
    return f


# --------------------------------------------------------------------------------------------- workloads
def workload_spec(name, nclients, steps, warmup, step_launches=None):
    """-> (fractions per client, gem-storm arguments, human description).  Quota files are written in the order
    gem-schd READS them: name request(min) limit(max) mem (SURVEY.md 8b trap)."""
    sl = step_launches or STEP_LAUNCHES
    if name == "storm":
        fr = [1.0 / nclients] * nclients
        return fr, ["--mode", "storm", "--steps", str(steps), "--warmup", str(warmup), "--step-launches", str(sl),
                    "--sync-every", str(SYNC_EVERY)], (
            "configs[1]: %d co-resident clients per B200, gpu_request %.3g each / gpu_limit 1.0, each %d x %d noop<<<1,32>>> "
            "launches on the default stream, cuCtxSynchronize every %d; quota file in gem-schd column order; base/min "
            "quota 300/20 ms, window 10 s" % (nclients, 1.0 / nclients, steps, sl, SYNC_EVERY))
    if name == "bursty":
        fr = [0.25] * 4
        rounds = steps * 25
        return fr, ["--mode", "bursty", "--rounds", str(rounds)], (
            "configs[2]: 4 clients per B200, gpu_request 0.25 / gpu_limit 1.0, bursty trace seed 0xB200: %d rounds (= %d steps "
            "x 25) of {U{16..4096} launches of a ~5 us spin kernel; sync; sleep Exp(2 ms)}" % (rounds, steps))
    if name == "mnist":
        fr = [0.1, 0.1, 0.4, 0.4]  # K8s priority 0/0/100/100 never reaches Gemini; SURVEY.md 8d models it as min-fraction
        iters = steps * 2
        return fr, ["--mode", "mnist", "--iters", str(iters)], (
            "configs[4]: 4 clients per B200, min-fractions 0.1/0.1/0.4/0.4 (priority 0/0/100/100), limit 1.0, MNIST-shaped "
            "conv (N=64, 1->32->64 ch, 28x28, 3x3): %d iterations (= %d steps x 2) x 100 launches + one DtoH" % (iters, steps))
    raise ValueError(name)


def quota_text(fracs):
    rows = ["bench/c%d %s 1.0 %d" % (i, repr(f), GIB8) for i, f in enumerate(fracs)]
    return "%d\n%s\n" % (len(fracs), "\n".join(rows))


def ledger_split_from_dump(path, nclients):
    """gem-schd(_DEBUG)'s ledger dump (scheduler.cpp:693-714): [{container,start,end} (seconds)] -> per-client ms."""
    led = json.load(open(path))
    out = [0.0] * nclients
    for e in led:
        try:
            i = int(e["container"].rsplit("c", 1)[1])
        except (ValueError, IndexError, KeyError):
            continue
        if 0 <= i < nclients:
            out[i] += (e["end"] - e["start"]) * 1e3
    return out, len(led)


def pool_ledger_split(pool_path, nclients):
    """-> (per-client token ms over the full history, hand-over gaps in the ledger window: count / total ms / longest ms)"""
    import ctypes as C

    import kubeshare_b200 as kb

    L = kb.lib()
    p = L.gemhook_pool_open(pool_path.encode(), 0, 0, 0, 0, 0)
    if not p:
        return None, None
    try:
        acc = [L.gemhook_pool_accumulated_ms(p, L.gemhook_pool_find(p, ("bench/c%d" % i).encode())) for i in range(nclients)]
        k = L.gemhook_pool_history(p, None, None, None, 0)
        sl, a, b = (C.c_int * k)(), (C.c_double * k)(), (C.c_double * k)()
        k = min(k, L.gemhook_pool_history(p, sl, a, b, k))
        gaps = [a[i + 1] - b[i] for i in range(k - 1) if a[i + 1] > b[i]]
        return acc, {"tokens": k, "gaps": len(gaps), "gap_ms_total": round(sum(gaps), 3), "gap_ms_max": round(max(gaps), 3) if gaps else 0.0}
    finally:
        L.gemhook_pool_close(p)


def run_clients(workload, nclients, steps, warmup, gpu, mode, core_base, step_launches=None, timeout=900, extra_env=None):
    """mode: 'unhooked' | 'ours' | 'reference' | 'reference-dbg'.  One run of `workload` with all clients co-resident
    on `gpu`.  Returns per-client results and aggregates (device-timed and host-timed)."""
    fracs, wargs, _ = workload_spec(workload, nclients, steps, warmup, step_launches)
    nclients = len(fracs)
    tmp = tempfile.mkdtemp(prefix="gembench_")
    daemons = []
    schd = None
    try:
        env0 = {k: v for k, v in os.environ.items() if not k.startswith("GEMHOOK_") and k not in ("LD_PRELOAD", "POD_NAME")}
        env0["CUDA_VISIBLE_DEVICES"] = str(gpu)
        env0.update(extra_env or {})
        with open(os.path.join(tmp, "quota.txt"), "w") as f:
            f.write(quota_text(fracs))
        ports = []
        dbg = mode == "reference-dbg"
        if mode.startswith("reference"):
            # the reference hook hard-codes /kubeshare/library/schedulerIP.txt (reference hook.cpp:162, 233-237)
            os.makedirs("/kubeshare/library", exist_ok=True)
            os.makedirs("/kubeshare/log", exist_ok=True)
            with open("/kubeshare/library/schedulerIP.txt", "w") as f:
                f.write("127.0.0.1\n")
            sport = free_ports(1)[0]
            schd_bin = os.path.join(REFDIR, "gem-schd-dbg" if dbg else "gem-schd")
            schd = sp.Popen([schd_bin, "-p", tmp, "-f", "quota.txt", "-P", str(sport)] + SCHD_ARGS + (["-v", "1"] if dbg else []),
                            cwd=tmp, stdout=sp.DEVNULL, stderr=sp.DEVNULL, preexec_fn=pin(core_base + 2 * nclients))
            daemons.append(schd)
            time.sleep(0.4)
            for i, port in enumerate(free_ports(nclients)):
                ports.append(port)
                e = dict(env0, POD_NAME="bench/c%d" % i, POD_MANAGER_PORT=str(port), SCHEDULER_IP="127.0.0.1",
                         SCHEDULER_PORT=str(sport))
                daemons.append(sp.Popen([os.path.join(REFDIR, "gem-pmgr")], env=e, stdout=sp.DEVNULL, stderr=sp.DEVNULL,
                                        preexec_fn=pin(core_base + nclients + i)))
            time.sleep(0.4)
        procs = []
        for i in range(nclients):
            e = dict(env0)
            if mode == "ours":
                e.update(LD_PRELOAD=HOOK, GEMHOOK_POOL=os.path.join(tmp, "pool"), GEMHOOK_QUOTA_FILE=os.path.join(tmp, "quota.txt"),
                         POD_NAME="bench/c%d" % i, GEMHOOK_STATS_FILE=os.path.join(tmp, "stats.%d.json" % i))
            elif mode.startswith("reference"):
                e.update(LD_PRELOAD=os.path.join(REFDIR, "libgemhook_ref_dbg.so.1" if dbg else "libgemhook_ref.so.1"),
                         POD_NAME="bench/c%d" % i, POD_MANAGER_PORT=str(ports[i]))
            cmd = [STORM] + wargs + ["--client-id", str(i), "--nclients", str(nclients), "--barrier-dir", tmp, "--out",
                                     os.path.join(tmp, "out.%d.json" % i)]
            procs.append(sp.Popen(cmd, env=e, stdout=sp.DEVNULL, stderr=sp.PIPE, preexec_fn=pin(core_base + i)))
        wall0 = time.time()
        errs = []
        for p in procs:
            try:
                _, err = p.communicate(timeout=timeout)
            except sp.TimeoutExpired:
                p.kill()
                _, err = p.communicate()
                errs.append("timeout")
            if p.returncode != 0:
                errs.append("rc=%s %s" % (p.returncode, (err or b"").decode()[-300:]))
        wall1 = time.time()
        if errs:
            raise RuntimeError("%s clients failed: %s" % (mode, errs))
        res = [json.load(open(os.path.join(tmp, "out.%d.json" % i))) for i in range(nclients)]
        stats, ledger, gaps = [], None, None
        if mode == "ours":
            for i in range(nclients):
                try:
                    stats.append(json.load(open(os.path.join(tmp, "stats.%d.json" % i))))
                except (OSError, ValueError):
                    stats.append({})
            try:
                ledger, gaps = pool_ledger_split(os.path.join(tmp, "pool"), nclients)
            except Exception as e:  # noqa: BLE001 -- a diagnostic, never fatal
                log("pool ledger unavailable: %r" % (e,))
        elif dbg and schd is not None:
            time.sleep(0.2)
            schd.send_signal(signal.SIGINT)  # the _DEBUG build dumps its ledger on SIGINT (scheduler.cpp:693-714)
            try:
                schd.wait(timeout=20)
            except sp.TimeoutExpired:
                pass
            dumps = [d for d in glob.glob(os.path.join(tmp, "*.json")) if os.path.basename(d)[0].isdigit()]
            if dumps:
                ledger, _ = ledger_split_from_dump(dumps[0], nclients)
        launches = sum(r["launches"] for r in res)
        dev_s = max(r["event_ms"] for r in res) / 1e3
        if all("t0" in r for r in res):
            host_s = max(r["t1"] for r in res) - min(r["t0"] for r in res)
        else:
            host_s = max(r["wall_s"] for r in res)
        return {"clients": nclients, "fracs": fracs, "launches": launches, "device_s": dev_s, "host_s": host_s,
                "step_s": [r.get("step_s") for r in res],
                "launches_per_s_device": launches / dev_s, "launches_per_s_host": launches / host_s,
                "per_client_wall_s": [r["wall_s"] for r in res], "per_client_launches": [r["launches"] for r in res],
                "stats": stats, "ledger_ms": ledger, "ledger_gaps": gaps, "window": (wall0, wall1)}
    finally:
        for d in daemons:
            if d.poll() is None:
                d.kill()
            d.wait()
        shutil.rmtree(tmp, ignore_errors=True)


def run_replicas(ngpu, fn):
    """Reference arm under torchrun: rank 0 alone drives one replica per GPU (threads only wait on subprocesses)."""
    out, errs = [None] * ngpu, []

    def work(g):
        try:
            out[g] = fn(g)
        except Exception as e:  # noqa: BLE001
            errs.append(e)

    th = [threading.Thread(target=work, args=(g,)) for g in range(ngpu)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if errs:
        raise errs[0]
    return out


def jain(xs):
    s, s2 = sum(xs), sum(x * x for x in xs)
    return s * s / (len(xs) * s2) if s2 else 0.0


def fairness(run):
    """Jain's index of rate/entitlement, the same basis in both arms: rate = the client's completion rate (launches per
    second of its own wall time), entitlement = its min-fraction.  (The ledger share is no basis for a fixed-work run: every
    client needs the same token time for the same work, whatever its fraction -- 0.735 by construction for
    0.1/0.1/0.4/0.4; it is reported next to it where the arm has a ledger.)"""
    return jain([l / w / f for l, w, f in zip(run["per_client_launches"], run["per_client_wall_s"], run["fracs"])]), \
        "completion_rate/min_fraction"


def fairness_ledger(run):
    if run.get("ledger_ms") and all(v is not None for v in run["ledger_ms"]) and sum(run["ledger_ms"]) > 0:
        return round(jain([d / f for d, f in zip(run["ledger_ms"], run["fracs"])]), 4)
    return None


# --------------------------------------------------------------------------------------------- roofline
def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        return None


def roofline_kernel(steps, warmup, nslots=2, sizes=(("ring_2p26", 1 << 26), ("ring_2p20", 1 << 20), ("ring_64", 64)), cpu=True,
                    last=None):
    """Time gemhook_acct_reduce on a device-resident ring through the C ABI (events on its own stream).  With a dict
    `last`, last[label] = the totals the last timed launch added (read back before it, outside its timed window)."""
    import numpy as np
    import torch

    import kubeshare_b200 as kb

    torch.cuda.init()
    torch.zeros(1, device="cuda")
    out = {}
    acct = kb.Acct(nslots)
    try:
        for label, n in sizes:
            rec = torch.empty((n, 4), dtype=torch.int32, device="cuda")
            idx = torch.arange(n, device="cuda", dtype=torch.int64)
            rec[:, 0] = ((idx * 2654435761) >> 7).remainder(nslots).to(torch.int32)
            rec[:, 1] = 1024
            rec[:, 2] = (2_000_000 + (idx % 4096)).to(torch.int32)
            rec[:, 3] = 0
            del idx
            torch.cuda.synchronize()
            flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if n < (1 << 24) else None
            times = []
            for i in range(warmup + steps):
                if flush is not None:
                    flush.fill_(i & 0xFF)  # write 256 MiB > 126 MB L2 between timed launches of the small rings
                    torch.cuda.synchronize()
                if last is not None and i == warmup + steps - 1:
                    before = acct.totals()[0].copy()
                ms = acct.reduce_device(rec.data_ptr(), n, timed=True)
                if i >= warmup:
                    times.append(ms)
            tot, _ = acct.totals()
            if last is not None:
                last[label] = (tot - before).astype(np.float64)
            expect = (warmup + steps) * n
            assert int(tot[:, 2].sum()) == expect, "accounting kernel lost records: %s vs %d" % (tot[:, 2], expect)
            acct.reset()
            avg_ms = sum(times) / len(times)
            out[label] = {"records": n, "bytes": 16 * n, "avg_ms": avg_ms, "min_ms": min(times),
                          "gbps": 16 * n / (avg_ms * 1e-3) / 1e9, "grid": acct.grid_for(n), "launches": len(times)}
            del rec
        if cpu:
            # CPU path of the same reduction (oracle), bounded sample: 2^24 records
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import orc

            OL = orc.load()
            n_cpu = 1 << 24
            r = np.zeros(n_cpu, np.dtype([("slot", "<u4"), ("launches", "<u4"), ("elapsed_ns", "<u8")]))
            r["slot"] = np.arange(n_cpu, dtype=np.uint32) % nslots
            r["launches"] = 1024
            r["elapsed_ns"] = 2_000_000
            t = time.time(); orc.acct_reduce(OL, r, nslots); t1 = time.time() - t
            threads = min(os.cpu_count() or 1, 64)
            t = time.time(); orc.acct_reduce(OL, r, nslots, threads=threads); tn = time.time() - t
            out["cpu_oracle"] = {"records": n_cpu, "gbps_1_thread": 16 * n_cpu / t1 / 1e9, "threads": threads,
                                 "gbps_all_threads": 16 * n_cpu / tn / 1e9}
        out["kernel_launches"] = acct.kernel_launches
    finally:
        acct.close()
    return out


# --------------------------------------------------------------------------------------------- main
def med(xs):
    return statistics.median(xs) if xs else None


def summarise_stats(stats):
    """min / median / max over the co-resident client processes for the counters that explain the number."""
    out = {}
    for k in ("token_requests", "token_wait_ms", "slow_path", "segments", "acct_kernels", "gpu_ns"):
        v = [s.get(k) for s in stats if s.get(k) is not None]
        if v:
            out[k] = [min(v), med(v), max(v)]
    return out


def dump_outputs(outdir, acct_last, hooked_launches):
    """--dump-outputs: the last timed step's outputs as float64 .npy files (a few KB: far below the 64 MB bound)."""
    import numpy as np

    if not outdir:
        return
    for label, tot in sorted((acct_last or {}).items()):
        np.save(os.path.join(outdir, "acct_totals_%s.npy" % label), np.asarray(tot, np.float64))
    if hooked_launches is not None:
        np.save(os.path.join(outdir, "hooked_launches.npy"), np.asarray(hooked_launches, np.float64))
    log("outputs in", outdir)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="storm", choices=["storm", "bursty", "mnist"])
    ap.add_argument("--clients", default="1,2,4,8", help="co-resident client counts to sweep (storm)")
    ap.add_argument("--headline-clients", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5, help="repetitions of the headline K-step run; value = median")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--skip-other", action="store_true", help="skip the bounded configs[2] / configs[4] samples of the default run")
    ap.add_argument("--skip-baseline", action="store_true", help="skip the reference cpu_baseline legs")
    ap.add_argument("--only-roofline", action="store_true", help="run just the accounting-kernel leg (for ncu)")
    ap.add_argument("--nslots", type=int, default=2, help="slot count of the roofline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.warmup < 3:
        log("warm-up raised to 3 (timing rules)")
        args.warmup = 3
    args.reps = max(1, args.reps)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    ngpu = world  # GPUs this job covers (replicas)
    ref_arm = args.impl == "reference"
    if ref_arm and world > 1:
        # contract: under torchrun the reference arm runs on rank 0 alone; the other ranks exit without work
        if rank != 0:
            return
        world = 1
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("gloo")  # host-side gather only: there is no collective in the data path
    gpu = local
    if not ref_arm:
        os.environ["CUDA_VISIBLE_DEVICES"] = str(gpu)  # this rank (and torch below) sees only its own GPU

    missing = [p for p in (STORM, HOOK) if not os.path.exists(p)]
    if missing:
        raise SystemExit("bench.py: %s missing -- run `python __graft_entry__.py` (build()) first" % ", ".join(missing))
    outdir = args.dump_outputs
    if outdir and rank == 0:
        os.makedirs(outdir, exist_ok=True)
    last = {} if outdir else None

    if args.only_roofline:
        print(json.dumps(roofline_kernel(args.steps, args.warmup, nslots=args.nslots, cpu=False, last=last)))
        if rank == 0:
            dump_outputs(outdir, last, None)
        return

    if ref_arm and not os.path.exists(os.path.join(REFDIR, "libgemhook_ref.so.1")):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (needs /root/reference at build time)"}))
        return

    ncpu = os.cpu_count() or 1
    nphys = len(physical_cores())
    cores_per_gpu = max(1, nphys // max(ngpu, 1))
    mode = "reference" if ref_arm else "ours"
    storm = args.workload == "storm"
    hc = args.headline_clients if storm else 4
    sweep = sorted({int(c) for c in args.clients.split(",") if c} | {hc}) if storm else [hc]
    my_gpus = list(range(ngpu)) if ref_arm else [gpu]

    def core_base(g):
        return g * cores_per_gpu + 1  # indices into physical_cores(): replicas never share a physical core

    def one(c, m, **kw):
        """one K-step run of the workload with c clients in mode m on every GPU this process drives"""
        if len(my_gpus) == 1:
            return [run_clients(args.workload, c, args.steps, args.warmup, my_gpus[0], m, core_base(my_gpus[0]), **kw)]
        return run_replicas(len(my_gpus), lambda g: run_clients(args.workload, c, args.steps, args.warmup, g, m, core_base(g), **kw))

    sampler = ClockSampler(gpu)
    sampler.start()
    windows = []
    results = {}
    t_start = time.time()
    for c in sweep:
        reps = args.reps if c == hc else 1
        runs = {"unhooked": [], "hooked": []}
        for _ in range(reps):
            for which, m in (("unhooked", "unhooked"), ("hooked", mode)):
                if dist:
                    dist.barrier()
                rr = one(c, m)
                windows += [r["window"] for r in rr]
                runs[which].append(rr)
        results[c] = runs
        log("rank %d clients=%d unhooked %s/s hooked(%s) %s/s (device-timed, per rep)" % (
            rank, c, ["%.0f" % sum(r["launches_per_s_device"] for r in rr) for rr in runs["unhooked"]], mode,
            ["%.0f" % sum(r["launches_per_s_device"] for r in rr) for rr in runs["hooked"]]))

    # bounded samples of BASELINE configs[2] (bursty) and configs[4] (MNIST-shaped, mixed fractions) on this rank's GPU, same
    # arm: un-hooked vs hooked aggregate launches/s and Jain fairness (full runs: --workload bursty|mnist)
    other = {}
    if storm and rank == 0 and not args.skip_other:
        for wl, k_o in (("bursty", 5), ("mnist", 30)):
            try:
                w0 = time.time()
                un_o = run_clients(wl, 4, k_o, args.warmup, my_gpus[0], "unhooked", core_base(my_gpus[0]))
                hk_o = run_clients(wl, 4, k_o, args.warmup, my_gpus[0], mode, core_base(my_gpus[0]))
                windows.append((w0, time.time()))
                jf, how = fairness(hk_o)
                other["configs[2] bursty" if wl == "bursty" else "configs[4] mnist"] = {
                    "sample": workload_spec(wl, 4, k_o, args.warmup)[2].split(": ", 1)[1][:160],
                    "unhooked_launches_per_s": round(un_o["launches_per_s_device"], 1),
                    "hooked_launches_per_s": round(hk_o["launches_per_s_device"], 1),
                    "overhead_pct": round((un_o["launches_per_s_device"] / hk_o["launches_per_s_device"] - 1.0) * 100.0, 3),
                    "jain_fairness": round(jf, 4), "fairness_of": how, "jain_ledger_share": fairness_ledger(hk_o)}
            except Exception as e:  # noqa: BLE001 -- a side sample must not take the headline down
                log("%s sample failed: %r" % (wl, e))

    roof = None
    base_runs = {}
    if not ref_arm and rank == 0:
        if not args.skip_roofline:
            w0 = time.time()
            roof = roofline_kernel(args.steps, args.warmup, nslots=args.nslots, last=last)
            try:  # the same kernel with the slot table full (GEMHOOK_MAX_SLOTS = 64 clients): bins crowd shared memory
                last64 = {} if last is not None else None
                r64 = roofline_kernel(args.steps, args.warmup, nslots=64, sizes=(("ring_2p26", 1 << 26),), cpu=False, last=last64)
                if last64:
                    last["ring_2p26_slots_64"] = last64["ring_2p26"]
                roof["slots_64"] = r64["ring_2p26"]
                roof["kernel_launches"] += r64["kernel_launches"]
            except Exception as e:  # noqa: BLE001
                log("64-slot roofline leg failed: %r" % (e,))
            windows.append((w0, time.time()))
        if os.path.exists(os.path.join(REFDIR, "libgemhook_ref.so.1")) and not args.skip_baseline:
            for key, m, k_steps in (("cpu_baseline", "reference", args.steps), ("cpu_baseline_debug", "reference-dbg", min(args.steps, 6))):
                if m == "reference-dbg" and not os.path.exists(os.path.join(REFDIR, "libgemhook_ref_dbg.so.1")):
                    continue
                try:
                    w0 = time.time()
                    # the reference stack is bimodal at 2 clients (370 K and 441 K launches/s in consecutive runs on one
                    # box): the baseline is the median of three runs, not a single draw
                    runs = [run_clients(args.workload, hc, k_steps, args.warmup, gpu, m, core_base(gpu))
                            for _ in range(3 if key == "cpu_baseline" else 1)]
                    runs.sort(key=lambda x: x["launches_per_s_device"])
                    r = runs[len(runs) // 2]
                    r["sample_steps"] = k_steps
                    r["runs"] = [round(x["launches_per_s_device"], 1) for x in runs]
                    base_runs[key] = r
                    windows.append((w0, time.time()))
                except Exception as e:  # noqa: BLE001 -- a baseline leg must not take the product arm down
                    log("%s leg failed: %r" % (key, e))
    sampler.stop()
    clocks = sampler.summary(windows)

    # ---- gather replicas: per client count and arm, per repetition, (launches, device_s, host_s) of every replica
    def slim(rr):
        return [{k: r.get(k) for k in ("launches", "device_s", "host_s", "stats", "ledger_ms", "ledger_gaps", "fracs", "per_client_wall_s",
                                       "per_client_launches", "step_s")} for r in rr]

    mine = {c: {which: [slim(rr) for rr in reps] for which, reps in runs.items()} for c, runs in results.items()}
    allr = [mine]
    if dist:
        allr = [None] * world
        dist.all_gather_object(allr, mine)
    if rank != 0:
        return

    def agg(c, which, rep):
        reps = [r for ranks in allr for r in ranks[c][which][rep]]  # every replica of this repetition
        launches = sum(r["launches"] for r in reps)
        return launches, max(r["device_s"] for r in reps), max(r["host_s"] for r in reps)

    def rate(c, which, host=False):
        n = len(allr[0][c][which])
        v = []
        for rep in range(n):
            l, d, h = agg(c, which, rep)
            v.append(l / (h if host else d))
        return v

    sweep_out = {}
    for c in sweep:
        un, hk = med(rate(c, "unhooked")), med(rate(c, "hooked"))
        un_h, hk_h = med(rate(c, "unhooked", True)), med(rate(c, "hooked", True))
        sweep_out[str(c)] = {"unhooked_launches_per_s": round(un, 1), "hooked_launches_per_s": round(hk, 1),
                             "frac_of_unhooked": round(hk / un, 5), "overhead_pct": round((un / hk - 1.0) * 100.0, 4),
                             "hooked_launches_per_s_e2e": round(hk_h, 1), "overhead_pct_e2e": round((un_h / hk_h - 1.0) * 100.0, 4)}
    hk_rates, hk_rates_h = rate(hc, "hooked"), rate(hc, "hooked", True)
    value, e2e_value = med(hk_rates), med(hk_rates_h)
    mid = sorted(range(len(hk_rates)), key=lambda i: hk_rates[i])[len(hk_rates) // 2]  # the repetition the median comes from
    lh, dh, hh = agg(hc, "hooked", mid)
    head_runs = [r for ranks in allr for r in ranks[hc]["hooked"][mid]]
    stats = [s for r in head_runs for s in r.get("stats", [])]
    acct_kernels = sum(s.get("acct_kernels", 0) for s in stats)
    segments = sum(s.get("segments", 0) for s in stats)
    fracs, _, desc = workload_spec(args.workload, hc, args.steps, args.warmup)
    k_all = max(1, args.steps + args.warmup)
    line = {
        "metric": "hooked_launches_per_s", "value": value, "unit": "launches/s", "n_gpus": ngpu, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dh * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": desc, "clients": hc, "step_launches": STEP_LAUNCHES, "sync_every": SYNC_EVERY, "reps": args.reps,
                   "parallelism": "replicas x%d (path does not shard)" % ngpu,
                   "l2": "roofline ring 1 GiB > 126 MB L2; smaller rings timed after a 256 MiB L2 flush"},
        "reps_values": [round(v, 1) for v in hk_rates],
        "overhead_pct": sweep_out[str(hc)]["overhead_pct"],
        "clients": sweep_out,
        "e2e": {"value": e2e_value, "unit": "launches/s",
                "h2d_bytes_per_step": (16 * segments // k_all) if mode == "ours" else 0,
                "d2h_bytes_per_step": (acct_kernels * (32 + 24 * hc) // k_all) if mode == "ours" else 0},
        "gpu_launches": int(acct_kernels + (roof or {}).get("kernel_launches", 0)) if mode == "ours" else 0,
        "clocks": clocks,
        "host": {"cpus": ncpu, "physical_cores": nphys, "client_cores": "one pinned PHYSICAL core per client, daemons on their own cores"},
        "wall_s": round(time.time() - t_start, 1),
    }
    if storm:
        line["overhead_pct_single_client_quota_1"] = sweep_out.get("1", {}).get("overhead_pct")
        if other:
            line["other_configs"] = other
    else:
        jf, how = fairness(head_runs[0])
        line["unhooked_launches_per_s"] = sweep_out[str(hc)]["unhooked_launches_per_s"]
        line["jain_fairness"] = {"value": round(jf, 5), "of": how, "ledger_share": fairness_ledger(head_runs[0])}
    if head_runs[0].get("ledger_ms"):
        line["ledger_ms"] = [round(v, 3) for v in head_runs[0]["ledger_ms"]]
    if head_runs[0].get("ledger_gaps"):
        line["ledger_gaps"] = head_runs[0]["ledger_gaps"]  # time between one token's end and the next one's start (last 10 s)
    if mode == "ours":
        line["hook_summary"] = summarise_stats(stats)
        peaks = measured_peaks()
        peak = (peaks or {}).get("hbm_gbs", 6650.0)
        if roof:
            big = roof["ring_2p26"]
            traffic = None
            try:  # dram read+write bytes per launch of the same kernel/size from the committed ncu --set full capture
                tj = json.load(open(os.path.join(ROOT, "profiles", "acct_reduce_traffic.json")))
                if tj.get("records") == big["records"]:
                    traffic = tj["traffic_bytes_per_launch"]
            except (OSError, ValueError, KeyError):
                pass
            small = {k: {kk: (round(vv, 5) if isinstance(vv, float) else vv) for kk, vv in roof[k].items() if kk in ("records", "avg_ms", "gbps", "grid")}
                     for k in roof if k.startswith("ring_") and k != "ring_2p26" and isinstance(roof[k], dict)}
            line["roofline"] = {"bound": "hbm", "kernel": "gemhook_acct_reduce", "achieved": big["gbps"], "peak": peak,
                                "unit": "GB/s", "frac": big["gbps"] / peak,
                                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6.65 TB/s (of fallback)",
                                "traffic": traffic, "algorithmic_bytes": big["bytes"], "records": big["records"], "avg_ms": big["avg_ms"],
                                "grid": big["grid"], "nslots": args.nslots, "small_rings": small, "cpu_oracle": roof.get("cpu_oracle")}
            if roof.get("slots_64"):
                line["roofline"]["slots_64"] = {"achieved": round(roof["slots_64"]["gbps"], 1), "frac": round(roof["slots_64"]["gbps"] / peak, 4),
                                                "avg_ms": round(roof["slots_64"]["avg_ms"], 5), "grid": roof["slots_64"]["grid"]}
        for key in ("cpu_baseline", "cpu_baseline_debug"):
            r = base_runs.get(key)
            if not r:
                if key == "cpu_baseline":
                    line[key] = {"value": None, "unit": "launches/s", "kind": "reference", "cores": 0, "sample": "oracle/_ref unavailable"}
                continue
            flavour = "libgemhook_ref.so.1 (-O2) + gem-pmgr + gem-schd" if key == "cpu_baseline" else \
                "libgemhook_ref_dbg.so.1 (as shipped, DEBUG=1) + gem-pmgr + gem-schd(_DEBUG)"
            line[key] = {"value": r["launches_per_s_device"], "e2e_value": r["launches_per_s_host"], "unit": "launches/s", "kind": "reference",
                         "cores": 2 * hc + 1, "timing": "device (CUDA events in every client), like `value`",
                         "sample": "%d clients x (%d warm-up + %d timed) steps of the same workload through oracle/_ref %s%s" % (
                             hc, args.warmup, r["sample_steps"], flavour, "; median of %d runs" % len(r["runs"]) if len(r["runs"]) > 1 else ""),
                         "runs": r["runs"]}
            if r.get("ledger_ms"):
                line[key]["ledger_ms"] = [round(v, 3) for v in r["ledger_ms"]]
    else:
        line["impl"] = "reference"
        line["cpu_baseline"] = {"value": value, "unit": "launches/s", "kind": "reference", "cores": (2 * hc + 1) * ngpu,
                                "sample": "%d clients x (%d warm-up + %d timed) steps, %d repetition(s), %d replica(s)" % (
                                    hc, args.warmup, args.steps, args.reps, ngpu)}
        line["e2e"] = {"value": e2e_value, "unit": "launches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if outdir:
        dump_outputs(outdir, last, [s.get("launches", 0) for s in stats] if mode == "ours" else None)
    # everything per process goes to a side file, not onto the line
    try:
        side = os.path.join(outdir or tempfile.mkdtemp(prefix="gembench_"), "bench_detail_%s_%s_n%d.json" % (mode, args.workload, ngpu))
        with open(side, "w") as f:
            json.dump({"line": line, "runs": allr, "baselines": {k: {kk: vv for kk, vv in v.items() if kk != "window"} for k, v in base_runs.items()},
                       "roofline": roof}, f)
        log("details in", side)
    except OSError:
        pass
    print(json.dumps(line))


if __name__ == "__main__":
    try:
        main()
    except Exception as e:  # noqa: BLE001
        if "--impl" in sys.argv and "reference" in sys.argv and int(os.environ.get("RANK", "0")) == 0:
            # contract: the reference arm never fails the driver; say why it could not run
            print(json.dumps({"impl": "reference", "unavailable": "reference stack failed on this box: %r" % (e,)}))
            sys.exit(0)
        raise
