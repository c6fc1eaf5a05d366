"""CPU: bench.py's reference arm prints ONE JSON line with the contract's keys (the product arm needs a GPU: one test
marked gpu runs it); __graft_entry__.build() is idempotent and leaves every library in place; --dump-outputs writes the
records of the last timed step."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    env = dict(os.environ, DPGICP_BENCH_CPU_TARGET_S="0.5")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "icp_cov_scan_pairs_per_sec" and d["unit"] == "pairs/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_build_entry_point():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.build()
    for rel in ("dpg_slam_b200/libdpgicp.so", "dpg_slam_b200/libdpgsynth.so", "dpg_slam_b200/dpg_batch_runner",
                "oracle/libdpgoracle.so"):
        assert os.path.exists(os.path.join(ROOT, rel)), rel


def test_dump_outputs_files_and_budget(tmp_path):
    """--dump-outputs: every record field as float32/float64 .npy with the values of the records; a batch over the budget
    is cut to a sorted, seeded sample that is the same on every call and stays under 64 MB on disk."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from dpg_slam_b200._abi import RESULT_DTYPE
    assert np.array_equal(bench.dump_sample(1000), np.arange(1000))
    big = bench.dump_sample(200_000_000)
    assert np.array_equal(big, bench.dump_sample(200_000_000)) and np.all(np.diff(big) > 0) and big[-1] < 200_000_000
    rng = np.random.default_rng(5)
    rec = np.zeros(len(big), RESULT_DTYPE)
    for f in ("tx", "ty", "theta", "rot_c", "rot_s", "mse", "cov"):
        rec[f] = rng.normal(size=rec[f].shape)
    rec["iterations"], rec["n_correspondences"] = rng.integers(0, 500, len(rec)), rng.integers(0, 4096, len(rec))
    rec["status"] = rng.integers(0, 2 ** 32, len(rec), dtype=np.uint32)
    bench.dump_records(str(tmp_path), rec, big)
    files = sorted(os.listdir(tmp_path))
    assert files == sorted(["index.npy"] + [f"{f}.npy" for f in RESULT_DTYPE.names])
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    assert np.array_equal(np.load(tmp_path / "index.npy"), big.astype(np.float64))
    for f in RESULT_DTYPE.names:
        a = np.load(tmp_path / f"{f}.npy")
        assert a.dtype in (np.float32, np.float64) and a.shape == rec[f].shape, f
        assert np.array_equal(a, rec[f]), f


def test_dump_outputs_needs_the_product_arm_on_one_gpu():
    for extra in (["--impl", "reference"], ["--gpus", "2"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", "unused"] + extra,
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr, extra


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs writes the records the timed path returned: the same bits as the same seeded batch
    submitted through the C ABI."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from dpg_slam_b200.scanmatch import ScanMatcher
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--pairs", "300", "--steps", "2", "--warmup", "0",
                        "--no-cpu-baseline", "--no-latency", "--no-also", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert d["steps"] == 2 and d["config"]["global_pairs"] == 300
    wl = bench.make_host_workload("corridor", 300)
    with ScanMatcher(0) as sm:
        sm.upload_ranges(wl.ranges, wl.scanner)
        want = sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, bench.bench_params("corridor", "pruned"))
    assert np.array_equal(np.load(tmp_path / "index.npy"), np.arange(300, dtype=np.float64))
    for f in want.dtype.names:
        assert np.array_equal(np.load(tmp_path / f"{f}.npy"), want[f]), f


def test_roofline_helpers_definitions():
    """The two ceilings bench.py quotes: the FP32 peak is the LARGER of the two measured separately-rounded rates (scalar and
    packed chains run at the same rate; the packed probe once reported twice that, from fused instructions) and the
    shared-memory bound charges two write-back cycles per warp-level point evaluation."""
    sys.path.insert(0, ROOT)
    import bench
    peak, scalar, packed = bench.fp32_peak({"mul_add_ops_per_s": 36.2e12, "mul_add_packed_ops_per_s": 37.1e12, "fma_ops_per_s": 36e12}, 37.2)
    assert (peak, scalar, packed) == (37.1, 36.2, 37.1)
    assert bench.fp32_peak({"mul_add_ops_per_s": 0.0}, 37.2)[0] == 37.2            # no probe: nominal rate
    blk = bench.smem_block({"distance_evals": 32 * 1000}, k_ms=1.0, sm_mhz=1000.0, n_sm=2)
    assert blk["busy_cycles_per_launch"] == 2000.0 and blk["available_cycles"] == 2.0e6 and blk["frac"] == 1e-3
