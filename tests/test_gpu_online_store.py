"""GPU (B200): the scan store grown one node at a time (dpgicp_append_ranges / dpgicp_append_scans) and the reference's
online loop replayed on it.  An appended store holds the rows one upload of the same scans would hold, so every record
is independent of how the store was built; a failed append leaves the store as it was; a store write refused for its
arguments leaves the store and every batch as they were; appends are stream-ordered
behind a run already enqueued; the online replay (append -> set_nodes -> enumerate ONLINE -> run, reoptimize at each
pass boundary) equals the CPU oracle update by update, and the C++ runner's --replay writes the same records."""
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from dpg_slam_b200 import synth
from dpg_slam_b200._abi import COV_CENSI_CORR, COV_REFERENCE_LIVE, ENUM_ONLINE, ENUM_REOPTIMIZE, Params
from dpg_slam_b200.scanmatch import DpgIcpError, ScanMatcher, relative_guess
from oracle import oracle_py as O
from test_gpu_parity import assert_records_match

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "dpg_slam_b200", "dpg_batch_runner")
E_INVALID, E_RANGE, E_TOOBIG = -1, -5, -7


def _corridor(n, n_beams, passes, seed):
    wl = synth.config_corridor_passes(n, n_beams, passes, seed)
    return wl.ranges, wl.scanner, wl.poses_est, wl.passes


def _rows(sm, n):
    return [sm.download_scan(k) for k in range(n)]


def _assert_rows_equal(got, want, ctx=""):
    assert len(got) == len(want), ctx
    for k, (a, b) in enumerate(zip(got, want)):
        assert a.shape == b.shape and a.tobytes() == b.tobytes(), f"{ctx}: row {k} differs"


def _chunks(n, sizes=(1, 7, 64)):
    out, k, i = [], 0, 0
    while k < n:
        out.append((k, min(n, k + sizes[i % len(sizes)])))
        k, i = out[-1][1], i + 1
    return out


def _ragged_clouds(rng, n):
    """0 .. 1500 points; a short first cloud so that later, longer ones re-pitch the store"""
    counts = rng.integers(0, 1501, n)
    counts[0], counts[1], counts[n // 2] = 5, 0, 1500
    clouds = [rng.uniform(-30, 30, (int(c), 2)).astype(np.float32) for c in counts]
    return clouds


def _csr(clouds):
    off = np.zeros(len(clouds) + 1, np.int64)
    off[1:] = np.cumsum([c.shape[0] for c in clouds])
    pts = np.concatenate(clouds) if clouds else np.zeros((0, 2), np.float32)
    return np.ascontiguousarray(pts, np.float32), off


def _pairs(est, passes):
    src, tgt = O.enumerate_pairs(est[:, :2], passes, 5.0, 2.0)
    guess = np.stack([relative_guess(est[t], est[s]) for s, t in zip(src, tgt)])
    return src, tgt, guess


# ---- 1. append == upload ------------------------------------------------------------------------------------------
def test_append_ranges_rows_equal_one_upload():
    ranges, sc, _, _ = _corridor(300, 1081, 1, seed=31)
    with ScanMatcher(0) as bulk, ScanMatcher(0) as sm:
        bulk.upload_ranges(ranges, sc)
        want = _rows(bulk, 300)
        assert sm.scan_count == 0
        for a, b in _chunks(300):                     # 1, 8, 72, 73, 80, 144, ...: crosses every capacity doubling
            sm.append_ranges(ranges[a:b], sc)
            assert sm.scan_count == b
            _assert_rows_equal(_rows(sm, b), want[:b], f"after appending scans {a}..{b - 1}")


def test_append_scans_rows_equal_one_upload_with_repitch():
    rng = np.random.default_rng(32)
    clouds = _ragged_clouds(rng, 160)
    with ScanMatcher(0) as bulk, ScanMatcher(0) as sm:
        bulk.upload_scans(*_csr(clouds))
        want = _rows(bulk, len(clouds))
        for c, w in zip(clouds, want):
            assert c.tobytes() == w.tobytes()
        sm.upload_scans(np.zeros((0, 2), np.float32), np.zeros(1, np.int64))          # an emptied store is started again
        for a, b in _chunks(len(clouds)):
            sm.append_scans(*_csr(clouds[a:b]))
            assert sm.scan_count == b
            _assert_rows_equal(_rows(sm, b), want[:b], f"after appending clouds {a}..{b - 1}")
        # PointXYZ layout (16-byte stride) appends the same rows
        sm.append_scans(*_csr([np.pad(c, ((0, 0), (0, 2))) for c in clouds[:9]]))
        _assert_rows_equal(_rows(sm, len(clouds) + 9)[len(clouds):], want[:9], "PointXYZ layout")


# ---- 2. records do not depend on how the store was built ------------------------------------------------------------
def test_records_do_not_depend_on_how_the_store_was_built():
    ranges, sc, est, passes = _corridor(120, 1081, 2, seed=33)
    src, tgt, guess = _pairs(est, passes)
    with ScanMatcher(0) as bulk, ScanMatcher(0) as app, ScanMatcher(0) as rep:
        bulk.upload_ranges(ranges, sc)
        clouds = _rows(bulk, len(ranges))
        for a, b in _chunks(len(ranges), (1, 7, 64)):
            app.append_ranges(ranges[a:b], sc)
        # re-pitched store: every chunk ends just before a cloud longer than all before it, so the store's pitch grows
        # with the clouds, one re-pitch per new maximum
        counts = np.array([c.shape[0] for c in clouds])
        cuts = [k for k in range(1, len(counts)) if counts[k] > counts[:k].max()]
        assert cuts and counts[:cuts[0]].max() < counts.max()
        bounds = [0] + cuts + [len(clouds)]
        for a, b in zip(bounds[:-1], bounds[1:]):
            rep.append_scans(*_csr(clouds[a:b]))
        for sm in (app, rep):
            _assert_rows_equal(_rows(sm, len(clouds)), clouds)
        for div in (1, 5):
            for cov in (COV_CENSI_CORR, COV_REFERENCE_LIVE):
                p = Params.defaults(downsample_divisor=div, cov_mode=cov)
                want = bulk.submit_pairs(src, tgt, guess, p)
                want_f = bulk.fetch_factors()
                for name, sm in (("appended", app), ("re-pitched", rep)):
                    got = sm.submit_pairs(src, tgt, guess, p)
                    assert got.tobytes() == want.tobytes(), (name, div, cov)
                    assert sm.fetch_factors().tobytes() == want_f.tobytes(), (name, div, cov)


# ---- 3. failure is atomic -----------------------------------------------------------------------------------------
def test_failed_append_leaves_the_store_as_it_was():
    ranges, sc, est, passes = _corridor(50, 1081, 1, seed=34)
    src, tgt, guess = _pairs(est, passes)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    with ScanMatcher(0) as sm:
        sm.append_ranges(ranges[:30], sc)
        sm.append_ranges(ranges[30:], sc)
        before = _rows(sm, 50)
        want = sm.submit_pairs(src, tgt, guess, p)
        far = synth.Scanner(n_beams=1081, range_max=1e6)
        bad_nan = ranges[:3].copy()
        bad_nan[2, 10] = np.nan
        bad_far = np.ones((2, 1081), np.float32)
        bad_far[1, 500] = 2000.0                                     # a point beyond 1000 m
        long_cloud = np.random.default_rng(1).uniform(-20, 20, (1500, 2)).astype(np.float32)
        attempts = [
            (E_RANGE, lambda: sm.append_ranges(bad_nan, sc)),
            (E_RANGE, lambda: sm.append_ranges(bad_far, far)),
            # growth and a re-pitch happen before the bad point is found
            (E_RANGE, lambda: sm.append_scans(*_csr([long_cloud] * 40 + [np.array([[np.nan, 0.0]], np.float32)]))),
            (E_RANGE, lambda: sm.append_scans(*_csr([long_cloud, np.array([[1000.5, 0.0]], np.float32)]))),
            (E_INVALID, lambda: sm.append_ranges(np.zeros((1, 1), np.float32), sc)),                  # n_beams < 2
            (E_INVALID, lambda: sm._check(sm._lib.dpgicp_append_ranges(sm._h, None, 1, 1081, sc.angle_min, sc.angle_max,
                                                                       sc.range_max, 0.2, 0.0, 0.0))),
            (E_INVALID, lambda: sm.append_scans(long_cloud, np.array([0, 10, 5], np.int64))),           # decreasing offsets
            (E_INVALID, lambda: sm._check(sm._lib.dpgicp_append_scans(sm._h, long_cloud.ctypes.data, 6,
                                                                      np.array([0, 3], np.int64).ctypes.data, 1))),
            (E_INVALID, lambda: sm._check(sm._lib.dpgicp_append_scans(sm._h, long_cloud.ctypes.data, 8, None, 1))),
            (E_TOOBIG, lambda: sm.append_scans(np.zeros((8193, 2), np.float32), np.array([0, 8193], np.int64))),
            (E_TOOBIG, lambda: sm.append_ranges(np.ones((1, 8193), np.float32), synth.Scanner(n_beams=8193))),
        ]
        for k, (code, call) in enumerate(attempts):
            with pytest.raises(DpgIcpError) as e:
                call()
            assert e.value.code == code, (k, e.value)
            assert sm.scan_count == 50, k
        _assert_rows_equal(_rows(sm, 50), before, "after the failed appends")
        assert sm.submit_pairs(src, tgt, guess, p).tobytes() == want.tobytes()
        # the store still grows normally afterwards
        sm.append_scans(*_csr([long_cloud]))
        assert sm.scan_count == 51 and sm.download_scan(50).tobytes() == long_cloud.tobytes()
        _assert_rows_equal(_rows(sm, 50), before, "after the next append")


def test_refused_store_writes_touch_nothing():
    """every store writer refuses bad arguments before it touches the store, the batches or the slots"""
    wl = synth.config_corridor(n_pairs=600, seed=38)
    sc = wl.scanner
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    half = len(wl.src_idx) // 2
    with ScanMatcher(0) as sm:
        sm.upload_ranges(wl.ranges, sc)
        row = sm.download_scan(7)
        slot = sm.slot()
        sm.set_pairs(wl.src_idx[:half], wl.tgt_idx[:half], wl.guess[:half])
        slot.set_pairs(wl.src_idx[half:], wl.tgt_idx[half:], wl.guess[half:])
        sm.run(p)
        slot.run(p)
        want = sm.fetch_results(), slot.fetch_results()
        lib, h = sm._lib, sm._h
        geo = (sc.angle_min, sc.angle_max, sc.range_max, 0.2, 0.0, 0.0)
        pts, off = np.zeros((4, 2), np.float32), np.array([0, 4], np.int64)
        wide = np.ones((1, 8193), np.float32)
        ids = np.array([0, 1], np.int32)                             # scan 1 of a one-scan array: out of range
        off_wide = np.array([0, 8193], np.int64)
        attempts = [
            ("upload_scans", E_INVALID, lambda: lib.dpgicp_upload_scans(h, pts.ctypes.data, 6, off.ctypes.data, 1)),
            ("upload_ranges", E_TOOBIG, lambda: lib.dpgicp_upload_ranges(h, wide.ctypes.data, 1, 8193, *geo)),
            ("upload_ranges_subset", E_INVALID,
             lambda: lib.dpgicp_upload_ranges_subset(h, wl.ranges.ctypes.data, 1, wl.ranges.shape[1], ids.ctypes.data, 2,
                                                     *geo)),
            ("convert_ranges_device", E_INVALID, lambda: lib.dpgicp_convert_ranges_device(h, None, 1, 1081, *geo)),
            ("append_ranges", E_INVALID, lambda: lib.dpgicp_append_ranges(h, wide.ctypes.data, 1, 1, *geo)),
            ("append_scans", E_TOOBIG, lambda: lib.dpgicp_append_scans(h, wide.ctypes.data, 8, off_wide.ctypes.data, 1)),
        ]
        for name, code, call in attempts:
            assert call() == code, name
            assert sm.scan_count == wl.n_scans, name
            assert sm.download_scan(7).tobytes() == row.tobytes(), name
            sm.run(p)
            slot.run(p)
            assert sm.fetch_results().tobytes() == want[0].tobytes(), name
            assert slot.fetch_results().tobytes() == want[1].tobytes(), name


# ---- 4. an append is stream-ordered behind a run already enqueued ----------------------------------------------------
def test_append_behind_an_enqueued_run():
    wl = synth.config_corridor(n_pairs=3000, seed=35)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    long_cloud = np.random.default_rng(2).uniform(-20, 20, (1500, 2)).astype(np.float32)
    with ScanMatcher(0) as ref, ScanMatcher(0) as sm:
        ref.upload_ranges(wl.ranges, wl.scanner)
        want = ref.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
        sm.upload_ranges(wl.ranges, wl.scanner)                      # capacity = exactly these rows
        sm.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
        sm.run(p)                                                    # asynchronous: no synchronise before the appends
        sm.append_ranges(wl.ranges[:200], wl.scanner)                # grows rows and counts
        sm.append_scans(*_csr([long_cloud] * 3))                     # re-pitches the store
        got = sm.fetch_results()
        assert got.tobytes() == want.tobytes()
        assert sm.scan_count == wl.n_scans + 203
        assert sm.download_scan(wl.n_scans + 5).tobytes() == ref.download_scan(5).tobytes()
        assert sm.download_scan(wl.n_scans + 202).tobytes() == long_cloud.tobytes()
        sm.run(p)                                                    # the same batch on the grown store
        assert sm.fetch_results().tobytes() == want.tobytes()


# ---- 5. the batch and the node table survive an append -------------------------------------------------------------
def test_batch_and_node_table_survive_an_append():
    ranges, sc, est, passes = _corridor(120, 1081, 2, seed=36)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    with ScanMatcher(0) as sm:
        sm.upload_ranges(ranges[:100], sc)
        sm.set_nodes(est[:100], passes[:100])
        for mode in (ENUM_REOPTIMIZE, ENUM_ONLINE):
            total, _ = sm.enumerate_pairs_device(mode, 5.0, 2.0)
            assert total > 0
            pairs = sm.fetch_pairs()
            sm.run(p)
            want = sm.fetch_results()
            sm.append_ranges(ranges[100:110] if mode == ENUM_REOPTIMIZE else ranges[110:], sc)
            sm.append_scans(*_csr([np.full((1200 + 100 * mode, 2), 0.5, np.float32)]))       # re-pitch
            for a, b in zip(sm.fetch_pairs(), pairs):
                assert a.tobytes() == b.tobytes()
            sm.run(p)
            assert sm.fetch_results().tobytes() == want.tobytes()


# ---- 6. the online loop, update by update, against the oracle ------------------------------------------------------
def _replay(sm, ranges, sc, est, passes, p, check=False):
    """The reference's loop on the device (append -> set_nodes -> enumerate -> run); with check=True every update is
    compared with the oracle on the clouds of nodes 0..k.  Returns [(update tag, src, tgt, records)]."""
    out = []
    pts_all, off_all = O.clouds_from_ranges(ranges, sc) if check else (None, None)

    def batch(n_nodes, mode, tag):
        sm.set_nodes(est[:n_nodes], passes[:n_nodes])
        total, _ = sm.enumerate_pairs_device(mode, 5.0, 2.0)
        src, tgt, _ = sm.fetch_pairs()
        sm.run(p)
        got = sm.fetch_results()
        out.append((tag, src, tgt, got))
        if check:
            enum = O.enumerate_online if mode == ENUM_ONLINE else O.enumerate_pairs
            wsrc, wtgt = enum(est[:n_nodes, :2], passes[:n_nodes], 5.0, 2.0)
            assert np.array_equal(src, wsrc) and np.array_equal(tgt, wtgt), tag
            guess = np.stack([O.relative_guess(est[t, :2], est[t, 2], est[s, :2], est[s, 2]) for s, t in zip(src, tgt)])
            off = off_all[:n_nodes + 1]
            ref, _ = O.run_batch(pts_all[:off[-1]], off, src, tgt, guess, p, fast=1, threads=0)
            assert_records_match(got, ref, f"update {tag}")

    for k in range(len(ranges)):
        if k > 0 and passes[k] != passes[k - 1]:
            batch(k, ENUM_REOPTIMIZE, f"reopt@{k}")
        sm.append_ranges(ranges[k:k + 1], sc)
        if check:
            assert sm.download_scan(k).tobytes() == pts_all[off_all[k]:off_all[k + 1]].tobytes()
        if k >= 1:
            batch(k + 1, ENUM_ONLINE, str(k))
    return out


def test_online_replay_equals_the_oracle():
    ranges, sc, est, passes = _corridor(120, 1081, 2, seed=37)
    with ScanMatcher(0) as sm:
        out = _replay(sm, ranges, sc, est, passes, Params.defaults(cov_mode=COV_CENSI_CORR), check=True)
    assert sum(t.startswith("reopt@") for t, *_ in out) == 1
    assert sum(len(s) for _, s, _, _ in out) > len(out)               # loop closures on the second pass


# ---- 7. the C++ runner's --replay ---------------------------------------------------------------------------------
def _read_log(path):
    raw = open(path, "rb").read()
    assert raw[:8] == b"DPGSCAN1"
    n_scans, n_beams = struct.unpack_from("<ii", raw, 8)
    amin, amax, rmax, lx, ly, lt = struct.unpack_from("<6f", raw, 16)
    rec = 16 + 4 * n_beams
    est = np.zeros((n_scans, 3), np.float32)
    passes = np.zeros(n_scans, np.int32)
    ranges = np.zeros((n_scans, n_beams), np.float32)
    for s in range(n_scans):
        o = 40 + s * rec
        est[s] = struct.unpack_from("<3f", raw, o)
        passes[s] = struct.unpack_from("<i", raw, o + 12)[0]
        ranges[s] = np.frombuffer(raw, np.float32, n_beams, o + 16)
    sc = synth.Scanner(n_beams=n_beams, angle_min=amin, angle_max=amax, range_max=rmax, laser_x=lx, laser_y=ly, laser_theta=lt)
    return ranges, sc, est, passes


def test_cpp_runner_replay_writes_the_python_records(tmp_path):
    log, csv1, csv2 = str(tmp_path / "scans.bin"), str(tmp_path / "a.csv"), str(tmp_path / "b.csv")
    r = subprocess.run([RUNNER, "--replay", "--synthetic", "corridor", "--scans", "60", "--passes", "2", "--beams", "256",
                        "--cov-mode", "2", "--write-log", log, "--out", csv1], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    assert summary["mode"] == "replay" and summary["online_updates"] == 59 and summary["reoptimize_batches"] == 1
    for q in ("update_ms_median", "update_ms_p90"):
        assert set(summary[q]) == {"append", "set_nodes", "enumerate_run_fetch", "total"}
    ranges, sc, est, passes = _read_log(log)
    with ScanMatcher(0) as sm:
        out = _replay(sm, ranges, sc, est, passes, Params.defaults(cov_mode=COV_CENSI_CORR))
    want = [(tag, s[k], t[k], rec[k]) for tag, s, t, rec in out for k in range(len(s))]
    lines = open(csv1).read().strip().splitlines()
    assert lines[0].startswith("update,src,tgt,")
    rows = [ln.split(",") for ln in lines[1:]]
    assert len(rows) == len(want) == summary["pairs"]
    for row, (tag, s, t, g) in zip(rows, want):
        assert row[0] == tag and int(row[1]) == s and int(row[2]) == t
        assert np.float32(row[3]) == g["tx"] and np.float32(row[4]) == g["ty"] and np.float32(row[5]) == g["theta"]
        assert np.array_equal(np.array(row[6:15], np.float64), g["cov"])
        assert int(row[15]) == g["iterations"] and int(row[16]) == g["status"]
    r = subprocess.run([RUNNER, "--replay", "--log", log, "--cov-mode", "2", "--out", csv2], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    assert open(csv2).read() == open(csv1).read()
    r = subprocess.run([RUNNER, "--replay", "--gpus", "2", "--log", log], capture_output=True, text=True, timeout=60)
    assert r.returncode != 0 and "--replay" in r.stderr
