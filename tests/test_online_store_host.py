"""Host tier of the online scan-store path: without a context the append entry points refuse the call, and the batch
runner's --replay mode fails loudly on a box without a GPU (there is no CPU fallback)."""
import os
import subprocess

import pytest

from dpg_slam_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "dpg_slam_b200", "dpg_batch_runner")


def test_append_entry_points_refuse_a_null_context():
    lib = _abi.load_library()
    assert lib.dpgicp_append_ranges(None, None, 1, 64, -1.0, 1.0, 30.0, 0.2, 0.0, 0.0) == -1
    assert lib.dpgicp_append_scans(None, None, 8, None, 1) == -1


def test_replay_runner_fails_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([RUNNER, "--replay", "--scans", "8", "--beams", "64"], capture_output=True, text=True)
    assert r.returncode == 1 and "no CPU fallback" in r.stderr


def test_replay_runner_refuses_several_gpus():
    for extra in (["--gpus", "2"], ["--devices", "0,0"]):
        r = subprocess.run([RUNNER, "--replay", "--scans", "8", "--beams", "64"] + extra, capture_output=True, text=True)
        assert r.returncode == 2 and "--replay" in r.stderr, r.stderr
