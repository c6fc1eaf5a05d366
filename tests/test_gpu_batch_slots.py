"""GPU (B200): batch slots — several pair batches in flight on one context, over its one scan store (dpgicp_slot_*).

A slot's records, factors and result counters are bit-equal to the same list run alone on the default slot, whatever
else runs at the same time and in whatever order the slots are filled, run and fetched.  Store writes behind queued slot
runs (an append that re-pitches the store, a failed append) leave those runs' records unchanged; set_nodes and an
enumeration into one slot while another runs give the default slot's list and records.  Slots die with work in flight
or with their context, and refuse calls once destroyed.  The C++ runner's --inflight K writes the CSV of --inflight 1."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from dpg_slam_b200 import synth
from dpg_slam_b200._abi import COV_CENSI_CORR, ENUM_REOPTIMIZE, METRIC_POINT_TO_LINE, Params
from dpg_slam_b200.scanmatch import DpgIcpError, ScanMatcher

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "dpg_slam_b200", "dpg_batch_runner")
E_INVALID, E_RANGE, E_STATE = -1, -5, -6
# counters of results; the work counters (distance evaluations, box tests) depend on the stage shape each pass ran in,
# which the hand-over timing decides
RESULT_COUNTERS = ("iterations", "correspondences")

P_CORRIDOR = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
P_LOOP = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
P_RAGGED = Params.defaults(downsample_divisor=5, metric=METRIC_POINT_TO_LINE, cov_mode=COV_CENSI_CORR)


@pytest.fixture(scope="module")
def world():
    """One store for three workloads: corridor rows, loop-closure rows, then ragged clouds (appended)."""
    wc = synth.config_corridor(n_pairs=800, n_beams=1081, seed=21)
    wl = synth.config_loop_closure(n_pairs=3000, n_scans=240, n_beams=1081, seed=22)
    ranges = np.concatenate([wc.ranges, wl.ranges])
    rng = np.random.default_rng(23)
    with ScanMatcher(0) as tmp:
        tmp.upload_ranges(wc.ranges[:301], wc.scanner)
        clouds = []
        for k in range(301):
            pts = tmp.download_scan(k)
            clouds.append(np.ascontiguousarray(pts[rng.random(pts.shape[0]) > rng.uniform(0.0, 0.6)]))
    off = np.zeros(len(clouds) + 1, np.int64)
    off[1:] = np.cumsum([c.shape[0] for c in clouds])
    pts = np.concatenate(clouds)
    base_l, base_r = wc.n_scans, wc.n_scans + wl.n_scans
    work = {
        "corridor": (wc.src_idx, wc.tgt_idx, wc.guess, P_CORRIDOR),
        "loop": (wl.src_idx + base_l, wl.tgt_idx + base_l, wl.guess, P_LOOP),
        "ragged": (np.arange(1, 301, dtype=np.int32) + base_r, np.arange(0, 300, dtype=np.int32) + base_r,
                   wc.guess[:300], P_RAGGED),
    }
    return dict(ranges=ranges, scanner=wc.scanner, pts=pts, off=off, work=work, corridor=wc)


def _matcher(world):
    sm = ScanMatcher(0)
    sm.upload_ranges(world["ranges"], world["scanner"])
    sm.append_scans(world["pts"], world["off"])
    return sm


def _counters(c):
    return {k: c[k] for k in RESULT_COUNTERS}


@pytest.fixture(scope="module")
def alone(world):
    """every workload run by itself on the default slot: records, factors, result counters"""
    out = {}
    with _matcher(world) as sm:
        for name, (s, t, g, p) in world["work"].items():
            sm.set_pairs(s, t, g)
            sm.run(p)
            out[name] = (sm.fetch_results(len(s)), sm.fetch_factors(len(s)), _counters(sm.last_run_counters()))
    return out


def _assert_alone(name, rec, alone, fac=None, counters=None):
    want = alone[name]
    assert rec.tobytes() == want[0].tobytes(), f"{name}: records differ from the batch run alone"
    if fac is not None:
        assert fac.tobytes() == want[1].tobytes(), f"{name}: factors differ"
    if counters is not None:
        assert _counters(counters) == want[2], name


# ---- 1. equal to running alone ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("names", [("corridor", "loop"), ("loop", "ragged", "corridor")])
def test_concurrent_slots_equal_running_alone(world, alone, names):
    with _matcher(world) as sm:
        slots = [sm.slot() for _ in names]
        for sl, name in zip(slots, names):
            sl.set_pairs(*world["work"][name][:3])
        for sl, name in zip(slots, names):
            sl.run(world["work"][name][3])
        for sl, name in zip(slots, names):
            n = len(world["work"][name][0])
            _assert_alone(name, sl.fetch_results(n), alone, sl.fetch_factors(n), sl.last_run_counters())


def test_run_range_slices_and_cost_hints_on_a_slot(world, alone):
    s, t, g, p = world["work"]["corridor"]
    n = len(s)
    with _matcher(world) as sm:
        a, b = sm.slot(), sm.slot()
        b.set_pairs(*world["work"]["loop"][:3])
        b.run(P_LOOP)
        a.set_pairs(s, t, g)
        a.set_pair_cost_hints(alone["corridor"][0]["iterations"].astype(np.float32))
        a.run(p)
        _assert_alone("corridor", a.fetch_results(n), alone)
        cuts = [0, 1, 333, n]
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            a.run_range(p, lo, hi - lo)
        b.run(P_LOOP)
        got = np.concatenate([a.fetch_results_range(lo, hi - lo) for lo, hi in zip(cuts[:-1], cuts[1:])])
        _assert_alone("corridor", got, alone)
        _assert_alone("loop", b.fetch_results(), alone)


# ---- 2. interleavings ------------------------------------------------------------------------------------------------
def test_interleavings(world, alone):
    W = world["work"]
    with _matcher(world) as sm:
        a, b = sm.slot(), sm.slot()
        # set_pairs on A while B runs; fetch B before A
        b.set_pairs(*W["loop"][:3])
        b.run(P_LOOP)
        a.set_pairs(*W["corridor"][:3])
        a.run(P_CORRIDOR)
        _assert_alone("loop", b.fetch_results(), alone)
        _assert_alone("corridor", a.fetch_results(), alone)
        # re-run a slot with another list before the other slot's records are fetched
        b.run(P_LOOP)
        a.set_pairs(*W["ragged"][:3])
        a.run(P_RAGGED)
        a.run(P_RAGGED)
        _assert_alone("ragged", a.fetch_results(), alone, a.fetch_factors())
        _assert_alone("loop", b.fetch_results(), alone, b.fetch_factors())
        # query does not block: pending right after a launch in at least one case, done after a synchronise
        seen_pending = False
        for _ in range(5):
            b.run(P_LOOP)
            seen_pending = seen_pending or not b.query()
            b.synchronize()
            assert b.query()
            if seen_pending:
                break
        assert seen_pending
        _assert_alone("loop", b.fetch_results(), alone)


# ---- 3. store and node table under in-flight slots -------------------------------------------------------------------
def test_append_regrowing_the_store_behind_queued_runs(world, alone):
    wc = world["corridor"]
    s, t, g, p = world["work"]["corridor"]
    half = len(s) // 2
    long_cloud = np.random.default_rng(5).uniform(-20, 20, (1500, 2)).astype(np.float32)
    with ScanMatcher(0) as sm:
        sm.upload_ranges(wc.ranges, wc.scanner)              # rows fill the store: any append moves it
        a, b = sm.slot(), sm.slot()
        a.set_pairs(s[:half], t[:half], g[:half])
        b.set_pairs(s[half:], t[half:], g[half:])
        a.run(p)
        b.run(p)
        sm.append_scans(long_cloud, np.array([0, 1500], np.int64))       # grows and re-pitches (1500 > 1082 points)
        assert sm.scan_count == wc.n_scans + 1
        got = np.concatenate([a.fetch_results(), b.fetch_results()])
        _assert_alone("corridor", got, alone)
        # a failed append behind queued runs leaves them as they were
        a.run(p)
        b.run(p)
        bad = long_cloud[:10].copy()
        bad[3, 0] = np.nan
        with pytest.raises(DpgIcpError) as e:
            sm.append_scans(bad, np.array([0, 10], np.int64))
        assert e.value.code == E_RANGE and sm.scan_count == wc.n_scans + 1
        got = np.concatenate([a.fetch_results(), b.fetch_results()])
        _assert_alone("corridor", got, alone)


def test_set_nodes_and_enumeration_into_a_slot_while_another_runs():
    wl = synth.config_corridor_passes(n_scans=400, n_beams=1081, passes=2, seed=24)
    with ScanMatcher(0) as sm:
        sm.upload_ranges(wl.ranges, wl.scanner)
        sm.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
        sm.run(P_CORRIDOR)
        succ = sm.fetch_results(len(wl.src_idx))
        sm.set_nodes(wl.poses_est, wl.passes)
        _, n = sm.enumerate_pairs_device(ENUM_REOPTIMIZE)
        sm.run(P_CORRIDOR)
        want = sm.fetch_results(n)
        want_pairs = sm.fetch_pairs(n)
        a, b = sm.slot(), sm.slot()
        b.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
        b.run(P_CORRIDOR)
        sm.set_nodes(wl.poses_est, wl.passes)
        assert a.enumerate_pairs_device(ENUM_REOPTIMIZE) == (n, n)
        a.run(P_CORRIDOR)
        got_pairs = a.fetch_pairs()
        for x, y in zip(got_pairs, want_pairs):
            assert x.tobytes() == y.tobytes()
        assert a.fetch_results().tobytes() == want.tobytes()
        assert b.fetch_results().tobytes() == succ.tobytes()


# ---- 4. lifetime and errors ------------------------------------------------------------------------------------------
def test_lifetime_and_errors(world, alone):
    lib_p = P_LOOP
    sm = _matcher(world)
    lib = sm._lib
    # destroy a slot with work in flight; the context carries on
    x = sm.slot()
    x.set_pairs(*world["work"]["loop"][:3])
    x.run(lib_p)
    h = x._h
    x.close()
    assert lib.dpgicp_slot_run(h, C.byref(lib_p)) == E_INVALID                  # a destroyed slot
    assert lib.dpgicp_slot_query(h) == E_INVALID and lib.dpgicp_slot_destroy(h) == E_INVALID
    assert lib.dpgicp_slot_run(None, C.byref(lib_p)) == E_INVALID               # a NULL slot
    sm.set_pairs(*world["work"]["loop"][:3])
    sm.run(lib_p)
    _assert_alone("loop", sm.fetch_results(), alone)
    # run before set_pairs; count mismatch on fetch
    y = sm.slot()
    with pytest.raises(DpgIcpError) as e:
        y.run(lib_p)
    assert e.value.code == E_STATE
    s, t, g, _ = world["work"]["corridor"]
    y.set_pairs(s[:10], t[:10], g[:10])
    y.run(P_CORRIDOR)
    for fetch in (y.fetch_results, y.fetch_factors):
        with pytest.raises(DpgIcpError) as e:
            fetch(11)
        assert e.value.code == E_INVALID
    with pytest.raises(ValueError):
        y.set_pairs(s[:10], t[:9], g[:10])
    # dpgicp_destroy with live slots, one of them running
    y.set_pairs(*world["work"]["loop"][:3])
    y.run(lib_p)
    hy = y._h
    sm.close()
    assert lib.dpgicp_slot_run(hy, C.byref(lib_p)) == E_INVALID
    y.close()


# ---- 5. C++ path -------------------------------------------------------------------------------------------------------
def test_runner_inflight_writes_the_csv_of_one_batch(tmp_path):
    base = [RUNNER, "--synthetic", "corridor", "--scans", "400", "--passes", "2", "--divisor", "1", "--cov-mode", "2"]
    outs = {}
    for k, extra in (("1", []), ("2", ["--inflight", "2", "--batch-pairs", "300"]),
                     ("3", ["--inflight", "3", "--batch-pairs", "128"])):
        path = tmp_path / f"inflight{k}.csv"
        r = subprocess.run(base + extra + ["--out", str(path)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        outs[k] = path.read_bytes()
    assert outs["1"].count(b"\n") > 600
    assert outs["2"] == outs["1"] and outs["3"] == outs["1"]
