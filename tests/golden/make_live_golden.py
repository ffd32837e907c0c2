#!/usr/bin/env python
"""Record what the tests used to read from the running REFERENCE stack, as committed fixtures.

Needs the unmodified reference built into oracle/_ref/ (`make -C oracle ref`, where its sources are available);
the tests themselves never run it.

    python tests/golden/make_live_golden.py cpu    -> tests/golden/ref_live_cpu.json   (stub driver, no GPU)
    python tests/golden/make_live_golden.py b200   -> tests/golden/ref_live_b200.json  (on a B200)

cpu:   * the reference hook's interposed surface (`nm -D` on libgemhook_ref.so.1);
       * every request our hook sent to the live reference gem-pmgr (+ gem-schd) and every answer it got, for the
         drop-in and gpu_mem-sweep scenarios of tests/test_preload_stub.py.
b200:  * the reference arm of tests/test_gpu_hook.py's accumulated-GPU-ms test (gem-schd(_DEBUG)'s own ledger);
       * the reference arm of the two ledger-parity configurations of tests/test_gpu_parity.py;
       * the requests the reference hook sent to gem-arbiter (with their times) next to a native client.
"""
import glob
import json
import os
import signal
import socket
import subprocess as sp
import sys
import tempfile
import threading
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import wireproto as wp  # noqa: E402

REF = os.path.join(ROOT, "oracle", "_ref")
GIB8 = 8589934592


def compact(t, req, rsp):
    """One exchange as [seconds since the first request, type, request fields, response fields]; the request id is the
    exchange's index on its connection (checked), the pod name is stored once per connection."""
    kind = req["type"]
    args = {wp.REQ_QUOTA: ("overuse", "burst"), wp.REQ_MEM_LIMIT: (), wp.REQ_MEM_UPDATE: ("bytes", "alloc")}[kind]
    answer = {wp.REQ_QUOTA: ("quota",), wp.REQ_MEM_LIMIT: ("used", "total"), wp.REQ_MEM_UPDATE: ("verdict",)}[kind]
    return [round(t, 6), kind, [req[k] for k in args], [rsp[k] for k in answer]]


class RecordingProxy(threading.Thread):
    """Loopback proxy between a hook and its pod manager: forwards each 80-byte request and the 40-byte answer to it, and
    records both with the time the request arrived, per connection in accept order: {"name", "calls": [compact(...)]}."""

    def __init__(self, upstream_port):
        super().__init__(daemon=True)
        self.upstream = upstream_port
        self.lsock = socket.socket()
        self.lsock.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
        self.lsock.bind(("127.0.0.1", 0))
        self.lsock.listen(8)
        self.port = self.lsock.getsockname()[1]
        self.conns = []
        self.t0 = None

    def run(self):
        try:
            while True:
                c, _ = self.lsock.accept()
                log = {"name": None, "calls": []}
                self.conns.append(log)
                threading.Thread(target=self._serve, args=(c, log), daemon=True).start()
        except OSError:
            pass

    def _serve(self, c, log):
        up = socket.create_connection(("127.0.0.1", self.upstream))
        try:
            while True:
                req = wp.recv_exact(c, wp.REQ_LEN)
                t = time.monotonic()
                if self.t0 is None:
                    self.t0 = t
                r = wp.unpack_request(req)
                assert r["id"] == len(log["calls"]) and log["name"] in (None, r["name"]), r
                log["name"] = r["name"]
                up.sendall(req)
                rsp = wp.recv_exact(up, wp.RSP_LEN)
                c.sendall(rsp)
                log["calls"].append(compact(t - self.t0, r, wp.unpack_response(rsp, r["type"])))
        except (ConnectionError, OSError):
            pass
        finally:
            c.close()
            up.close()

    def close(self):
        self.lsock.close()


def daemons(tmp, cfg, schd_args=("-q", "300", "-m", "20", "-w", "10000"), schd="gem-schd", pod="bench/c0"):
    with open(os.path.join(tmp, "cfg.txt"), "w") as f:
        f.write(cfg)
    sport, pport = wp.free_port(), wp.free_port()
    s = sp.Popen([os.path.join(REF, schd), "-p", tmp, "-f", "cfg.txt", "-P", str(sport), *schd_args], cwd=tmp,
                 stdout=sp.DEVNULL, stderr=sp.DEVNULL)
    time.sleep(0.5)
    p = sp.Popen([os.path.join(REF, "gem-pmgr")], stdout=sp.DEVNULL, stderr=sp.DEVNULL,
                 env=dict(os.environ, POD_NAME=pod, POD_MANAGER_PORT=str(pport), SCHEDULER_IP="127.0.0.1", SCHEDULER_PORT=str(sport)))
    time.sleep(0.5)
    return s, p, pport


def stop(*procs):
    for p in procs:
        if p.poll() is None:
            p.kill()
        p.wait()


# ------------------------------------------------------------------------------------------------------------- cpu
def hook_surface():
    out = sp.check_output(["nm", "-D", "--defined-only", os.path.join(REF, "libgemhook_ref.so.1")], text=True)
    return sorted({line.split()[-1] for line in out.splitlines() if " T " in line})


def pmgr_session(cfg, runs, schd_args=("-q", "300", "-m", "20", "-w", "10000"), stats=True):
    """Our hook (stub driver) against fresh reference daemons through a recording proxy; one entry per gem-storm run,
    in the environment the test runs it in (with a stats file the hook asks for its usage once more at exit)."""
    import kubeshare_b200 as kb
    from test_preload_stub import base_env, run_storm

    out = []
    with tempfile.TemporaryDirectory() as tmp:
        s, p, pport = daemons(tmp, cfg, schd_args)
        try:
            for args in runs:
                px = RecordingProxy(pport)
                px.start()
                env = base_env(tmp, LD_PRELOAD=kb.LIB_PATH, GEMHOOK_SCHEDULER_IP="127.0.0.1", POD_MANAGER_PORT=px.port,
                               POD_NAME="bench/c0")
                if stats:
                    env["GEMHOOK_STATS_FILE"] = os.path.join(tmp, "stats.%d.json")
                res = run_storm(env, *args)
                time.sleep(0.2)
                px.close()
                out.append({"args": list(map(str, args)), "result": res, "conns": px.conns})
        finally:
            stop(p, s)
    return {"config": cfg, "schd_args": list(schd_args), "runs": out}


def make_cpu():
    g = {"_made_by": "tests/golden/make_live_golden.py cpu, reference built into oracle/_ref"}
    g["hook_surface"] = hook_surface()
    g["drop_in"] = pmgr_session("1\nbench/c0 1.0 1.0 5000\n", [
        ["--mode", "resolve"],
        ["--mode", "storm", "--steps", 2, "--warmup", 1, "--step-launches", 2000, "--sync-every", 200]])
    g["memsweep"] = pmgr_session("1\nbench/c0 1.0 1.0 %d\n" % GIB8, [["--mode", "memsweep"]], schd_args=(), stats=False)
    return g


# ------------------------------------------------------------------------------------------------------------ b200
def accumulated_reference_arm():
    """test_gpu_hook's storm (30 x 65536 launches) through the reference hook + gem-pmgr + gem-schd(_DEBUG)."""
    import kubeshare_b200 as kb  # noqa: F401
    from test_gpu_hook import storm

    with tempfile.TemporaryDirectory() as tmp:
        s, p, pport = daemons(tmp, "1\nbench/c0 1.0 1.0 %d\n" % GIB8, ("-q", "300", "-m", "20", "-w", "10000", "-v", "1"), "gem-schd-dbg")
        try:
            env = {k: v for k, v in os.environ.items() if not k.startswith("GEMHOOK_") and k != "LD_PRELOAD"}
            env.update(POD_NAME="bench/c0", POD_MANAGER_PORT=str(pport), LD_PRELOAD=os.path.join(REF, "libgemhook_ref.so.1"))
            res = storm(env, "--mode", "storm", "--steps", 30, "--warmup", 2, "--step-launches", 65536)
            time.sleep(0.2)
            s.send_signal(signal.SIGINT)
            s.wait(timeout=20)
            dumps = [d for d in glob.glob(os.path.join(tmp, "*.json")) if os.path.basename(d)[0].isdigit()]
            led = [e for e in json.load(open(dumps[0])) if e["container"] == "bench/c0"]
        finally:
            stop(p, s)
    return {"ledger_ms": sum(e["end"] - e["start"] for e in led) * 1e3, "closed_ms": sum(e["end"] - e["start"] for e in led[:-1]) * 1e3,
            "tokens": len(led), "wall_ms": res["wall_s"] * 1e3}


def legacy_transcript():
    """The reference hook (gem-storm, 6 x 65536 launches) speaking TCP to gem-arbiter next to a native client, recorded."""
    import kubeshare_b200 as kb

    with tempfile.TemporaryDirectory() as tmp:
        with open(os.path.join(tmp, "cfg.txt"), "w") as f:
            f.write("2\nbench/native 0.5 1.0 %d\nbench/legacy 0.5 1.0 %d\n" % (GIB8, GIB8))
        port, pool = wp.free_port(), os.path.join(tmp, "pool")
        arb = sp.Popen([os.path.join(kb.HERE, "bin", "gem-arbiter"), "--pool", pool, "-p", tmp, "-f", "cfg.txt", "-P", str(port),
                        "-q", "300", "-m", "20", "-w", "10000"], stderr=sp.DEVNULL)
        time.sleep(0.5)
        px = RecordingProxy(port)
        px.start()
        try:
            base = {k: v for k, v in os.environ.items() if not k.startswith("GEMHOOK_") and k != "LD_PRELOAD"}
            e_native = dict(base, LD_PRELOAD=kb.LIB_PATH, GEMHOOK_POOL=pool, POD_NAME="bench/native")
            e_legacy = dict(base, LD_PRELOAD=os.path.join(REF, "libgemhook_ref.so.1"), POD_NAME="bench/legacy", POD_MANAGER_PORT=str(px.port))
            args = ["--mode", "storm", "--steps", "6", "--warmup", "1", "--step-launches", "65536", "--nclients", "2", "--barrier-dir", tmp]
            procs = [sp.Popen([kb.STORM_PATH, *args, "--client-id", "0", "--out", os.path.join(tmp, "o0.json")], env=e_native),
                     sp.Popen([kb.STORM_PATH, *args, "--client-id", "1", "--out", os.path.join(tmp, "o1.json")], env=e_legacy)]
            for p in procs:
                p.wait(timeout=300)
                assert p.returncode == 0
            outs = [json.load(open(os.path.join(tmp, "o%d.json" % i))) for i in range(2)]
            time.sleep(0.2)
        finally:
            px.close()
            stop(arb)
    return {"conns": px.conns, "legacy_wall_s": outs[1]["wall_s"], "native_wall_s": outs[0]["wall_s"]}


def make_b200():
    import torch
    from test_gpu_parity import CONFIG2, CONFIG5, _kubeshare_dirs, arm_result

    _kubeshare_dirs()   # the reference hook reads /kubeshare/library/schedulerIP.txt (reference hook.cpp:162, 233-237)

    g = {"_made_by": "tests/golden/make_live_golden.py b200, reference built into oracle/_ref",
         "device": torch.cuda.get_device_name(0)}
    try:
        g["power_limit"] = sp.check_output(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], text=True).strip()
    except (OSError, sp.CalledProcessError):
        g["power_limit"] = None
    g["accumulated"] = accumulated_reference_arm()
    g["config2"] = arm_result("reference", *CONFIG2)
    g["config5"] = arm_result("reference", *CONFIG5)
    g["legacy_hook_vs_arbiter"] = legacy_transcript()
    return g


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else ""
    if which not in ("cpu", "b200"):
        sys.exit("usage: make_live_golden.py cpu|b200 [output path]")
    if not os.path.exists(os.path.join(REF, "gem-pmgr")):
        sys.exit("build the reference first: make -C oracle ref")
    g = make_cpu() if which == "cpu" else make_b200()
    path = sys.argv[2] if len(sys.argv) > 2 else os.path.join(HERE, "ref_live_%s.json" % which)
    with open(path, "w") as f:
        json.dump(g, f, separators=(",", ":"))
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
