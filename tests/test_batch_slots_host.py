"""Host tier of the batch slots (dpgicp_slot_*): the library exports every slot entry point at ABI version 5, the ctypes
bindings agree with the prototypes in include/dpgicp.h, a NULL slot is refused before any device work, and the batch
runner refuses --inflight where it does not apply."""
import ctypes as C
import os
import re
import subprocess

from dpg_slam_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dpgicp.h")
RUNNER = os.path.join(ROOT, "dpg_slam_b200", "dpg_batch_runner")
E_INVALID = -1


def _slot_prototypes():
    """name -> list of parameter declarations of every dpgicp_slot_* prototype in the header"""
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    out = {}
    for m in re.finditer(r"\bint\s+(dpgicp_slot_\w+)\s*\(([^)]*)\)\s*;", text):
        out[m.group(1)] = [a.strip() for a in m.group(2).split(",")]
    return out


SCALARS = {"int32_t": C.c_int32, "int64_t": C.c_int64, "float": C.c_float}


def _ctypes_of(decl: str):
    """the ctypes types a C parameter declaration may bind to in _abi.py (a data pointer: void* or typed)"""
    if re.search(r"counters\[8\]$", decl):
        return (C.POINTER(C.c_uint64 * 8),)
    if "dpgicp_params" in decl:
        return (C.POINTER(_abi.Params),)
    if "**" in decl:
        return (C.POINTER(C.c_void_p),)
    base = decl.split("*")[0].replace("const", "").strip()
    if "*" in decl:
        return (C.c_void_p,) + ((C.POINTER(SCALARS[base]),) if base in SCALARS else ())
    return (SCALARS[decl.rsplit(" ", 1)[0].replace("const", "").strip()],)


def test_abi_version_is_5():
    lib = _abi.load_library()
    assert _abi.ABI_VERSION == 5 and lib.dpgicp_abi_version() == 5
    assert "#define DPGICP_ABI_VERSION 5" in open(HEADER).read()


def test_slot_symbols_exported_and_listed():
    protos = _slot_prototypes()
    assert len(protos) == 14, sorted(protos)
    lib = _abi.load_library()
    for name in protos:
        assert name in _abi.EXPORTS, name
        getattr(lib, name)
    assert sorted(n for n in _abi.EXPORTS if n.startswith("dpgicp_slot_")) == sorted(protos)


def test_slot_ctypes_signatures_match_header():
    lib = _abi.load_library()
    for name, params in _slot_prototypes().items():
        fn = getattr(lib, name)
        assert fn.restype is C.c_int, name
        want = [_ctypes_of(p) for p in params]
        assert len(fn.argtypes) == len(want), name
        for k, (got, ok) in enumerate(zip(fn.argtypes, want)):
            assert got in ok, f"{name} argument {k} ({params[k]}): {got} not in {ok}"


def test_null_slot_is_refused():
    lib = _abi.load_library()
    p = _abi.Params.defaults()
    h = C.c_void_p()
    assert lib.dpgicp_slot_create(None, C.byref(h)) == E_INVALID and not h.value
    assert lib.dpgicp_slot_destroy(None) == E_INVALID
    assert lib.dpgicp_slot_set_pairs(None, None, None, None, 0) == E_INVALID
    assert lib.dpgicp_slot_set_pair_cost_hints(None, None, 0) == E_INVALID
    assert lib.dpgicp_slot_run(None, C.byref(p)) == E_INVALID
    assert lib.dpgicp_slot_run_range(None, C.byref(p), 0, 0) == E_INVALID
    assert lib.dpgicp_slot_fetch_results(None, None, 0) == E_INVALID
    assert lib.dpgicp_slot_fetch_results_range(None, None, 0, 0) == E_INVALID
    assert lib.dpgicp_slot_fetch_factors(None, None, 0) == E_INVALID
    assert lib.dpgicp_slot_fetch_pairs(None, None, None, None, 0) == E_INVALID
    c = (C.c_uint64 * 8)()
    assert lib.dpgicp_slot_last_run_counters(None, C.byref(c)) == E_INVALID
    assert lib.dpgicp_slot_synchronize(None) == E_INVALID
    assert lib.dpgicp_slot_query(None) == E_INVALID
    n = C.c_int64(0)
    assert lib.dpgicp_slot_enumerate_pairs_device(None, 0, 5.0, 2.0, 0, 1, C.byref(n), C.byref(n)) == E_INVALID


def test_runner_refuses_inflight_where_it_does_not_apply():
    for extra in (["--replay"], ["--successive-only"], ["--gpus", "2"], ["--devices", "0,0"]):
        r = subprocess.run([RUNNER, "--inflight", "2", "--scans", "8", "--beams", "64"] + extra, capture_output=True, text=True)
        assert r.returncode == 2 and "--inflight" in r.stderr, (extra, r.stderr)
    for bad in (["--inflight", "0"], ["--inflight", "2", "--batch-pairs", "0"]):
        r = subprocess.run([RUNNER, "--scans", "8", "--beams", "64"] + bad, capture_output=True, text=True)
        assert r.returncode == 2 and "--inflight" in r.stderr, (bad, r.stderr)
