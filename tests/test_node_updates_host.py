"""Host tier of dpgicp_update_nodes: the library exports it and lists it, the ctypes binding agrees with the header
prototype, a NULL context is refused before any device work, and the batch runner refuses a bad --nodes value."""
import ctypes as C
import os
import re
import subprocess

from dpg_slam_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dpgicp.h")
RUNNER = os.path.join(ROOT, "dpg_slam_b200", "dpg_batch_runner")
E_INVALID = -1


def _prototype():
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    m = re.search(r"\bint\s+dpgicp_update_nodes\s*\(([^)]*)\)\s*;", text)
    assert m, "dpgicp_update_nodes is not declared"
    return [a.strip() for a in m.group(1).split(",")]


def test_update_nodes_exported_and_listed():
    assert "dpgicp_update_nodes" in _abi.EXPORTS
    getattr(_abi.load_library(), "dpgicp_update_nodes")


def test_update_nodes_ctypes_signature_matches_header():
    params = _prototype()
    assert params == ["dpgicp_ctx *ctx", "int32_t n_nodes", "const int32_t *ids", "const float *pose_xytheta",
                      "const int32_t *pass", "int32_t n_ids"]
    fn = _abi.load_library().dpgicp_update_nodes
    assert fn.restype is C.c_int
    assert fn.argtypes == [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]


def test_null_context_is_refused():
    lib = _abi.load_library()
    assert lib.dpgicp_update_nodes(None, 0, None, None, None, 0) == E_INVALID
    assert lib.dpgicp_update_nodes(None, 4, None, None, None, 4) == E_INVALID


def test_runner_refuses_a_bad_nodes_value():
    for extra in (["--replay", "--nodes", "partial"], ["--replay", "--nodes", ""], ["--nodes", "sync"]):
        r = subprocess.run([RUNNER, "--scans", "8", "--beams", "64"] + extra, capture_output=True, text=True)
        assert r.returncode == 2 and "--nodes" in r.stderr, (extra, r.stderr)
