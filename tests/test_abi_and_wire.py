"""CPU: the C ABI library loads and exports every symbol include/gemhook.h declares; wire codec parity."""
import ctypes as C
import json
import os
import subprocess

import kubeshare_b200 as kb

G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_golden.json")))

_SURVEYED_SURFACE = [  # SURVEY.md 8b: what `nm -D` showed on the reference libgemhook.so.1
    "dlsym", "cuGetProcAddress", "cuLaunchKernel", "cuLaunchCooperativeKernel", "cuMemAlloc_v2", "cuMemAllocManaged",
    "cuMemAllocPitch_v2", "cuMemFree_v2", "cuArrayCreate_v2", "cuArray3DCreate_v2", "cuArrayDestroy",
    "cuMipmappedArrayCreate", "cuMipmappedArrayDestroy", "cuMemGetInfo_v2", "cuDeviceTotalMem_v2", "cuCtxSynchronize",
    "cuMemcpyAtoH_v2", "cuMemcpyHtoA_v2", "cuMemcpyHtoD_v2"]


def reference_hook_surface():
    """The interposed symbols of the reference hook, as `nm -D` listed them on the reference build itself
    (tests/golden/ref_live_cpu.json, recorded by tests/golden/make_live_golden.py); plus the two the reference gets
    wrong / lacks: cuMemcpyDtoH_v2 (it exports it C++-mangled, hook.cpp:925-926) and cuGetProcAddress_v2 (CUDA >= 12
    resolves through it)."""
    with open(os.path.join(os.path.dirname(__file__), "golden", "ref_live_cpu.json")) as f:
        syms = set(json.load(f)["hook_surface"])
    names = sorted(x for x in syms if x == "dlsym" or (x.startswith("cu") and not x.startswith("cuda")))
    assert set(_SURVEYED_SURFACE) <= set(names), "the survey's list and the reference build disagree"
    assert any("cuMemcpyDtoH" in x and x.startswith("_Z") for x in syms) or "cuMemcpyDtoH_v2" in syms
    return sorted(set(names) | {"cuMemcpyDtoH_v2", "cuGetProcAddress_v2"})


REFERENCE_HOOK_SURFACE = reference_hook_surface()


def exported():
    out = subprocess.check_output(["nm", "-D", "--defined-only", kb.LIB_PATH], text=True)
    return {line.split()[-1] for line in out.splitlines() if " T " in line}


def test_every_declared_symbol_is_exported():
    syms = exported()
    missing = [s for s in kb.abi_symbols() if s not in syms]
    assert not missing, missing
    kb.lib()  # binds every function with ctypes; raises AttributeError if one is absent


def test_hook_surface_matches_reference():
    syms = exported()
    assert not [s for s in REFERENCE_HOOK_SURFACE if s not in syms]
    L = kb.lib()
    n = C.c_size_t()
    arr = L.gemhook_hooked_symbols(C.byref(n))
    names = [arr[i].decode() for i in range(n.value)]
    assert set(REFERENCE_HOOK_SURFACE) <= set(names)
    assert all(s in syms for s in names)


def test_no_cxx_runtime_leaks():
    """An LD_PRELOAD shim must not export libstdc++ symbols into the application's namespace."""
    assert not [s for s in exported() if s.startswith("_Z")]
    needed = subprocess.check_output(["readelf", "-d", kb.LIB_PATH], text=True)
    assert "libstdc++" not in needed and "libcudart" not in needed and "libcuda" not in needed


def test_wire_requests_match_reference_bytes():
    L = kb.lib()
    for case in G["wire"]:
        for r in case["requests"]:
            req = kb.Request(name=case["name"].encode(), req_id=r["id"], type=r["type"], overuse_ms=r["overuse"],
                             burst_ms=r["burst"], bytes=r["bytes"], is_alloc=r["alloc"])
            buf = (C.c_uint8 * 80)()
            assert L.gemhook_wire_pack_request(C.byref(req), buf) > 0
            assert bytes(buf).hex() == r["hex"]
            back = kb.Request()
            assert L.gemhook_wire_unpack_request(buf, C.byref(back)) == r["payload_off"] + (16 if r["type"] == 0 else 12 if r["type"] == 2 else 0)
            assert (back.name.decode(), back.req_id, back.type) == (r["parsed_name"], r["parsed_id"], r["parsed_type"])
            if r["type"] == 0:
                assert (back.overuse_ms, back.burst_ms) == (r["overuse"], r["burst"])
            if r["type"] == 2:
                assert (back.bytes, back.is_alloc) == (r["bytes"], r["alloc"])


def test_wire_responses_match_reference_bytes():
    L = kb.lib()
    for r in G["wire"][0]["responses"]:
        rsp = kb.Response(req_id=r["id"], quota_ms=r.get("quota", 0.0), mem_used=r.get("used", 0),
                          mem_total=r.get("total", 0), verdict=r.get("verdict", 0))
        buf = (C.c_uint8 * 40)()
        assert L.gemhook_wire_pack_response(r["type"], C.byref(rsp), buf) == r["len"]
        assert bytes(buf).hex() == r["hex"]
        back = kb.Response()
        L.gemhook_wire_unpack_response(r["type"], buf, C.byref(back))
        assert back.req_id == r["id"]
        assert (back.quota_ms, back.mem_used, back.mem_total, back.verdict) == (
            r.get("quota", 0.0), r.get("used", 0), r.get("total", 0), r.get("verdict", 0))


def test_overlong_pod_name_is_rejected_not_overflowed():
    """The reference writes past its 80-byte buffer (comm.cpp:42-60); we refuse."""
    L = kb.lib()
    buf = (C.c_uint8 * 96)(*([0xAA] * 96))
    req = kb.Request(name=b"x" * 48, req_id=1, type=kb.REQ_QUOTA)
    assert L.gemhook_wire_pack_request(C.byref(req), buf) == -1
    assert bytes(buf[80:]) == b"\xaa" * 16
    req = kb.Request(name=b"x" * 47, req_id=1, type=kb.REQ_QUOTA)
    assert L.gemhook_wire_pack_request(C.byref(req), buf) == 80
    req = kb.Request(name=b"x" * 52, req_id=1, type=kb.REQ_MEM_UPDATE)
    assert L.gemhook_wire_pack_request(C.byref(req), buf) == -1
