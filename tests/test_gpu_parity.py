"""GPU (B200): the CUDA path, called through the C ABI, against the CPU oracle on the same seeded
inputs.  Bars (BASELINE.json north_star): correspondence index sets bit-exact at equal iterate;
poses within 1e-5 m / 1e-5 rad; covariances within 1e-4 relative.  Because both sides follow one
arithmetic contract (DESIGN.md), most fields are in fact compared bit for bit; the tolerances are
written where the device's libm (atan2f, cos/sin in the covariance) may differ from glibc's."""
import ctypes as C

import numpy as np
import pytest

from dpg_slam_b200 import _abi, synth
from dpg_slam_b200._abi import (METRIC_POINT_TO_LINE, STOP_DEGENERATE, COV_CENSI_CORR, COV_CENSI_INDEXPAIR, COV_REFERENCE_LIVE, FLAG_CONVERGED,
                                FLAG_COV_SINGULAR, FLAG_EMPTY_INPUT, SEARCH_BRUTE, SEARCH_PRUNED, SEARCH_PROJECTIVE, STOP_ITERATIONS,
                                STOP_MASK, STOP_NO_CORRESPONDENCES, Params)
from dpg_slam_b200.scanmatch import DpgIcpError
from oracle import oracle_py as O

pytestmark = pytest.mark.gpu

POSE_TOL_M = 1e-5        # north_star: final poses agree within 1e-5 m / 1e-5 rad
POSE_TOL_RAD = 1e-5
COV_REL_TOL = 1e-4       # north_star: covariances agree within 1e-4 relative
EXACT_FIELDS = ("tx", "ty", "rot_c", "rot_s", "iterations", "status", "n_correspondences", "mse")


def assert_records_match(got, ref, ctx=""):
    assert len(got) == len(ref)
    for f in EXACT_FIELDS:                      # same arithmetic contract on both sides -> same bits
        bad = np.nonzero(got[f] != ref[f])[0]
        assert bad.size == 0, f"{ctx}: field {f} differs at pairs {bad[:5]}: {got[f][bad[:5]]} vs {ref[f][bad[:5]]}"
    assert np.max(np.abs(got["tx"] - ref["tx"]), initial=0) <= POSE_TOL_M
    assert np.max(np.abs(got["ty"] - ref["ty"]), initial=0) <= POSE_TOL_M
    dth = np.abs(got["theta"] - ref["theta"])
    dth = np.minimum(dth, np.abs(dth - 2 * np.pi))
    assert np.max(dth, initial=0) <= POSE_TOL_RAD, ctx
    scale = np.abs(ref["cov"]).max(axis=1)
    rel = np.abs(got["cov"] - ref["cov"]).max(axis=1) / np.where(scale > 0, scale, 1.0)
    assert np.max(rel, initial=0) <= COV_REL_TOL, f"{ctx}: cov rel err {rel.max():.3e}"


def run_both(sm, wl, p, threads=0):
    sm.upload_ranges(wl.ranges, wl.scanner)
    pts, off = sm.download_store()
    got = sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    ref, _ = O.run_batch(pts, off, wl.src_idx, wl.tgt_idx, wl.guess, p, fast=1, threads=threads)
    return got, ref, pts, off


# ---- scan store ------------------------------------------------------------------------------------------
def test_upload_ranges_matches_oracle_cloud_bit_exact(gpu_matcher):
    wl = synth.config_loop_closure(n_pairs=4, n_scans=24, seed=21)
    wl.ranges[3, ::7] = wl.scanner.range_max            # ragged: extra dropped beams
    wl.ranges[5, :] = wl.scanner.range_max + 1          # an empty scan
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    assert gpu_matcher.scan_count == 24
    for k in range(24):
        want = O.ranges_to_cloud(wl.ranges[k], wl.scanner)
        got = gpu_matcher.download_scan(k)
        assert got.shape == want.shape and got.tobytes() == want.tobytes(), k
    assert gpu_matcher.download_scan(5).shape == (0, 2)


def test_upload_ranges_subset_pinned_and_pageable(gpu_matcher):
    """A per-rank store holds only the scans its pairs touch; page-locked input is read in place by the kernel."""
    import torch
    wl = synth.config_corridor(n_pairs=60, n_beams=721, seed=14)
    ids = np.array([5, 0, 17, 17, 60, 3], np.int32)
    want = [O.ranges_to_cloud(wl.ranges[k], wl.scanner) for k in ids]
    pinned = torch.from_numpy(wl.ranges).pin_memory()
    for src in (wl.ranges, pinned.data_ptr()):
        gpu_matcher.upload_ranges_subset(src, ids, wl.scanner, n_scans_total=wl.n_scans, n_beams=721)
        assert gpu_matcher.scan_count == len(ids)
        for row, w in enumerate(want):
            got = gpu_matcher.download_scan(row)
            assert got.shape == w.shape and got.tobytes() == w.tobytes()
    with pytest.raises(DpgIcpError) as e:
        gpu_matcher.upload_ranges_subset(wl.ranges, np.array([61], np.int32), wl.scanner)
    assert e.value.code == -1
    # aligning through the subset store with remapped indices == aligning through the full store
    from dpg_slam_b200 import sharded
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    full = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    sh = sharded.ShardedScanMatcher(gpu_matcher, 1, 3)
    sh.upload_ranges_for_shard(pinned.data_ptr(), wl.scanner, wl.src_idx, wl.tgt_idx, n_scans_total=wl.n_scans, n_beams=721)
    sh.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
    sh.run(p)
    part = gpu_matcher.fetch_results(sharded.shard_len(60, 1, 3))
    assert part.tobytes() == full[sharded.shard_indices(60, 1, 3)].tobytes()


def test_upload_scans_packed_and_pointxyz_stride_agree(gpu_matcher):
    wl = synth.config_corridor(n_pairs=3, n_beams=361, seed=4)
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_scans(pts, off)
    a = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    xyz = np.zeros((pts.shape[0], 4), np.float32)       # pcl::PointXYZ layout {x, y, z, pad}
    xyz[:, :2] = pts
    xyz[:, 2] = 0.0
    xyz[:, 3] = 1.0
    gpu_matcher.upload_scans(xyz, off)
    b = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    assert a.tobytes() == b.tobytes()
    ref, _ = O.run_batch(pts, off, wl.src_idx, wl.tgt_idx, wl.guess, p, fast=1)
    assert_records_match(a, ref, "stride")


# ---- correspondences: bit-exact index sets at equal iterate ------------------------------------------------
@pytest.mark.parametrize("search", [SEARCH_BRUTE, SEARCH_PRUNED])
@pytest.mark.parametrize("reciprocal", [1, 0])
def test_correspondence_sets_bit_exact_at_every_iterate(gpu_matcher, search, reciprocal):
    wl = synth.config_loop_closure(n_pairs=3, n_scans=16, seed=33)
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    p = Params.defaults(downsample_divisor=1, search=search, use_reciprocal=reciprocal, max_iterations=40)
    for k in range(wl.n_pairs):
        s, t = wl.src_idx[k], wl.tgt_idx[k]
        src, tgt = pts[off[s]:off[s + 1]], pts[off[t]:off[t + 1]]
        _, iterates, n_corr = O.icp(src, tgt, wl.guess[k], p, trace=True)
        # the oracle's iterate k is the accumulated float transform; replaying it from the original cloud is
        # the same iterate for both sides (they are fed the identical T and identical points)
        picks = sorted(set([0, 1, 2, len(iterates) // 2, len(iterates) - 1]))
        for it in picks:
            T = iterates[it]
            cur = O.transform_points(T, src)
            kk, want, want_d2 = O.correspondences(cur, tgt, p)
            got, got_d2 = gpu_matcher.correspondences(src, tgt, T, p)
            assert np.array_equal(got, want), (k, it)
            m = want >= 0
            assert np.array_equal(got_d2[m].view(np.uint32), want_d2[m].view(np.uint32)), (k, it)
            assert int((got >= 0).sum()) == kk


def test_correspondence_ties_pick_lowest_index(gpu_matcher):
    # lattice target: many exact distance ties; source points on cell centres and edges
    gx, gy = np.meshgrid(np.arange(12, dtype=np.float32) * 0.25, np.arange(9, dtype=np.float32) * 0.25)
    tgt = np.stack([gx.ravel(), gy.ravel()], 1).astype(np.float32)
    sx, sy = np.meshgrid(np.arange(23, dtype=np.float32) * 0.125, np.arange(17, dtype=np.float32) * 0.125)
    src = np.stack([sx.ravel(), sy.ravel()], 1).astype(np.float32)
    T = np.array([1, 0, 0, 0], np.float32)
    for search in (SEARCH_BRUTE, SEARCH_PRUNED):
        for rec in (0, 1):
            p = Params.defaults(search=search, use_reciprocal=rec)
            kk, want, want_d2 = O.correspondences(src, tgt, p)
            got, got_d2 = gpu_matcher.correspondences(src, tgt, T, p)
            assert np.array_equal(got, want), (search, rec)


@pytest.mark.parametrize("n", [300, 1500, 4097, 8192])
def test_box_hierarchy_on_large_unordered_clouds(gpu_matcher, n):
    """The two-level candidate rounds of the pruned search (one round over 256-point boxes, then the groups of the
    surviving ones, two upper boxes per round) against the brute-force walk and the oracle on clouds that are NOT in
    beam order — loose boxes, many surviving upper boxes, several rounds — with lattice ties and duplicated points, at
    sizes that leave the last upper box partly filled (300, 1500, 4097) and at the maximum (8192 = 32 upper boxes)."""
    rng = np.random.default_rng(100 + n)
    tgt = rng.uniform(0, 12, (n, 2))
    tgt[: n // 4] = np.round(tgt[: n // 4] * 4) / 4                     # lattice points: exact ties
    tgt[n // 4: n // 3] = tgt[rng.integers(0, n // 4, n // 3 - n // 4)]  # duplicates
    tgt = tgt[rng.permutation(n)].astype(np.float32)
    m = max(n - 37, 1)
    src = (tgt[rng.permutation(n)[:m]] + rng.normal(0, 0.02, (m, 2))).astype(np.float32)
    src[: m // 5] = tgt[rng.integers(0, n, m // 5)]                      # exact hits, zero distance
    T = np.array([np.cos(0.01), np.sin(0.01), 0.02, -0.01], np.float32)
    for rec in (1, 0):
        for gate in (0.6, 0.05):
            want = None
            for search in (SEARCH_BRUTE, SEARCH_PRUNED):
                p = Params.defaults(search=search, use_reciprocal=rec, max_correspondence_distance=gate)
                got, got_d2 = gpu_matcher.correspondences(src, tgt, T, p)
                if want is None:
                    _, want, want_d2 = O.correspondences(O.transform_points(T, src), tgt, p)
                assert np.array_equal(got, want), (n, rec, gate, search)
                ok = want >= 0
                assert np.array_equal(got_d2[ok].view(np.uint32), want_d2[ok].view(np.uint32)), (n, rec, gate, search)


# ---- whole path: BASELINE configs at oracle-sized batches ---------------------------------------------------
def test_config1_room_pair_default_params(gpu_matcher):
    wl = synth.config_room_pair()
    for p in (Params.defaults(), Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)):
        got, ref, _, _ = run_both(gpu_matcher, wl, p)
        assert_records_match(got, ref, "room pair")
        assert got["status"][0] & FLAG_CONVERGED
        assert abs(got["tx"][0] - 0.30) < 0.02 and abs(got["ty"][0] + 0.20) < 0.02 and abs(got["theta"][0] - 0.10) < 0.01


@pytest.mark.parametrize("search", [SEARCH_BRUTE, SEARCH_PRUNED])
@pytest.mark.parametrize("divisor", [1, 5])
@pytest.mark.parametrize("cov_mode", [COV_REFERENCE_LIVE, COV_CENSI_INDEXPAIR, COV_CENSI_CORR])
def test_config2_corridor_batch(gpu_matcher, search, divisor, cov_mode):
    wl = synth.config_corridor(n_pairs=64, seed=2)
    p = Params.defaults(downsample_divisor=divisor, search=search, cov_mode=cov_mode)
    got, ref, _, _ = run_both(gpu_matcher, wl, p)
    assert_records_match(got, ref, f"corridor s{search} d{divisor} c{cov_mode}")
    if cov_mode == COV_REFERENCE_LIVE:          # cov.h:572-575, bit-exact
        want = np.diag([0.5, 0.5, np.float64(np.float32(0.3))]).reshape(9)
        assert np.all(got["cov"] == want)


@pytest.mark.parametrize("cov_cap", [200, 0])
def test_config3_loop_closure_batch(gpu_matcher, cov_cap):
    wl = synth.config_loop_closure(n_pairs=300, n_scans=120, seed=3)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR, cov_cap=cov_cap)
    got, ref, _, _ = run_both(gpu_matcher, wl, p)
    assert_records_match(got, ref, "loop closure")
    assert (got["status"] & FLAG_CONVERGED).mean() > 0.9


def test_dense_4096_beam_scans(gpu_matcher):
    wl = synth.config_loop_closure(n_pairs=12, n_scans=24, n_beams=4096, seed=4)
    for div in (1, 5):
        p = Params.defaults(downsample_divisor=div, cov_mode=COV_CENSI_CORR)
        got, ref, _, _ = run_both(gpu_matcher, wl, p)
        assert_records_match(got, ref, f"dense d{div}")


def test_maximum_size_scans(gpu_matcher):
    wl = synth.config_corridor(n_pairs=2, n_beams=_abi.MAX_POINTS, seed=6)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR, max_iterations=12)
    got, ref, _, _ = run_both(gpu_matcher, wl, p)
    assert_records_match(got, ref, "8192 beams")
    with pytest.raises(DpgIcpError) as e:
        gpu_matcher.upload_ranges(np.ones((1, _abi.MAX_POINTS + 1), np.float32), wl.scanner)
    assert e.value.code == -7


def test_non_reciprocal_and_iteration_limits(gpu_matcher):
    wl = synth.config_corridor(n_pairs=24, seed=8)
    for kw in (dict(use_reciprocal=0), dict(max_iterations=1), dict(max_iterations=7),
               dict(max_correspondence_distance=0.15), dict(transformation_epsilon=1e-6)):
        p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR, **kw)
        got, ref, _, _ = run_both(gpu_matcher, wl, p)
        assert_records_match(got, ref, str(kw))
    assert np.all(got["iterations"] >= 1)


# ---- point-to-line metric (north-star extension; oracle-defined) ----------------------------------------------
@pytest.mark.parametrize("search", [SEARCH_BRUTE, SEARCH_PRUNED])
def test_point_to_line_batches(gpu_matcher, search):
    for wl, div in ((synth.config_corridor(n_pairs=64, seed=2), 1), (synth.config_loop_closure(n_pairs=200, n_scans=80, seed=3), 1),
                    (synth.config_loop_closure(n_pairs=64, n_scans=80, seed=3), 5)):
        p = Params.defaults(downsample_divisor=div, cov_mode=COV_CENSI_CORR, metric=METRIC_POINT_TO_LINE, search=search)
        got, ref, _, _ = run_both(gpu_matcher, wl, p)
        assert_records_match(got, ref, f"p2l {wl.name} d{div} s{search}")
    assert (got["status"] & FLAG_CONVERGED).mean() > 0.9


def test_point_to_line_dense_4096(gpu_matcher):
    """BASELINE config 4 shape: 4096 beams/scan, point-to-line."""
    wl = synth.config_loop_closure(n_pairs=16, n_scans=24, n_beams=4096, seed=4)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR, metric=METRIC_POINT_TO_LINE)
    got, ref, _, _ = run_both(gpu_matcher, wl, p)
    assert_records_match(got, ref, "p2l dense")


def test_point_to_line_degenerate_and_ragged(gpu_matcher):
    x = np.linspace(-3, 3, 200, dtype=np.float32)
    wall = np.stack([x, np.full_like(x, 2.0)], 1)
    p = Params.defaults(downsample_divisor=1, metric=METRIC_POINT_TO_LINE, cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_scans(np.concatenate([wall, wall]), np.array([0, 200, 400]))
    got = gpu_matcher.submit_pairs([1], [0], [[0.0, 0.05, 0.0]], p)
    ref = O.run_pair(wall, wall, [0.0, 0.05, 0.0], p)
    assert got["status"][0] == ref.status and (got["status"][0] & STOP_MASK) == STOP_DEGENERATE
    assert (got["tx"][0], got["ty"][0], got["iterations"][0]) == (ref.tx, ref.ty, ref.iterations)
    wl = synth.config_corridor(n_pairs=8, n_beams=721, seed=12)
    wl.ranges[2, :] = 40.0
    wl.ranges[4, 2:] = 40.0
    wl.ranges[6, ::2] = 40.0
    got, ref, _, _ = run_both(gpu_matcher, wl, p)
    assert_records_match(got, ref, "p2l ragged")


# ---- edge cases ------------------------------------------------------------------------------------------------
def test_empty_ragged_and_degenerate_inputs(gpu_matcher):
    wl = synth.config_corridor(n_pairs=8, n_beams=721, seed=12)
    wl.ranges[2, :] = 40.0                              # scan 2: everything at max range -> empty cloud
    wl.ranges[4, 2:] = 40.0                             # scan 4: two points only (< 3 correspondences)
    wl.ranges[6, ::2] = 40.0                            # scan 6: half the beams dropped
    wl.guess[7] = (60.0, 60.0, 0.0)                     # pair 7: nothing within the 0.6 m gate
    for cov_mode in (COV_CENSI_CORR, COV_CENSI_INDEXPAIR, COV_REFERENCE_LIVE):
        for search in (SEARCH_BRUTE, SEARCH_PRUNED):
            p = Params.defaults(downsample_divisor=1, cov_mode=cov_mode, search=search)
            got, ref, _, _ = run_both(gpu_matcher, wl, p)
            assert_records_match(got, ref, f"edge c{cov_mode} s{search}")
    # pairs touching the empty scan: flagged, not converged, guess returned (record always written)
    touched = (wl.src_idx == 2) | (wl.tgt_idx == 2)
    assert np.all(got["status"][touched] & FLAG_EMPTY_INPUT)
    assert np.all((got["status"][touched] & STOP_MASK) == STOP_NO_CORRESPONDENCES)
    assert np.all((got["status"][touched] & FLAG_CONVERGED) == 0)
    assert (got["status"][7] & STOP_MASK) == STOP_NO_CORRESPONDENCES and got["tx"][7] == 60.0


def test_identical_clouds_identity(gpu_matcher):
    wl = synth.config_room_pair()
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    pts, off = gpu_matcher.download_store()
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    got = gpu_matcher.submit_pairs([0], [0], [[0, 0, 0]], p)
    assert got["iterations"][0] == 1 and got["mse"][0] == 0.0 and got["theta"][0] == 0.0
    assert got["n_correspondences"][0] == off[1] - off[0]


def test_error_codes(gpu_matcher):
    wl = synth.config_room_pair()
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    p = Params.defaults()
    for bad, code in ((dict(src=[5], tgt=[0]), -1), (dict(src=[0], tgt=[-1]), -1)):
        with pytest.raises(DpgIcpError) as e:
            gpu_matcher.submit_pairs(bad["src"], bad["tgt"], [[0, 0, 0]], p)
        assert e.value.code == code
    with pytest.raises(DpgIcpError) as e:
        gpu_matcher.submit_pairs([1], [0], [[np.nan, 0, 0]], p)
    assert e.value.code == -5
    for kw in (dict(max_iterations=0), dict(downsample_divisor=0), dict(max_correspondence_distance=-1.0),
               dict(cov_mode=7), dict(search=9), dict(metric=5)):
        with pytest.raises(DpgIcpError) as e:
            gpu_matcher.submit_pairs([1], [0], [[0, 0, 0]], Params.defaults(**kw))
        assert e.value.code == -1, kw
    pts = np.array([[0, 0], [np.inf, 1]], np.float32)
    with pytest.raises(DpgIcpError) as e:
        gpu_matcher.upload_scans(pts, np.array([0, 2]))
    assert e.value.code == -5
    with pytest.raises(DpgIcpError) as e:
        gpu_matcher.upload_scans(np.array([[2000.0, 0]], np.float32), np.array([0, 1]))
    assert e.value.code == -5
    assert gpu_matcher.submit_pairs([], [], np.zeros((0, 3)), p).shape == (0,)     # empty batch is fine, even with no store
    with pytest.raises(DpgIcpError) as e:                                          # a failed upload leaves no store behind
        gpu_matcher.submit_pairs([0], [0], [[0, 0, 0]], p)
    assert e.value.code == -6


def test_random_small_problems_bit_exact(gpu_matcher):
    """Many tiny random problems: 0..150 points per cloud, duplicated points and lattice ties, random gates, both
    metrics, reciprocal on/off, all covariance modes, divisors 1..4, extreme coordinates (|x| up to 990 m)."""
    rng = np.random.default_rng(2025)
    clouds, offsets, family = [], [0], []
    for base_id in range(40):
        n = int(rng.choice([0, 1, 2, 3, 5, 17, 31, 32, 33, 64, 100, 150]))
        centre = rng.uniform(-950, 950, 2) if base_id % 7 == 0 else rng.uniform(-20, 20, 2)
        kind = base_id % 4
        if kind == 0:      # wall-like polyline
            t = np.sort(rng.uniform(0, 6, n))
            pts = np.stack([t, 0.3 * np.sin(t)], 1)
        elif kind == 1:    # lattice: exact distance ties
            pts = np.stack([rng.integers(0, 8, n) * 0.25, rng.integers(0, 8, n) * 0.25], 1).astype(float)
        elif kind == 2:    # duplicated points
            base = rng.uniform(0, 3, (max(n // 2, 1), 2))
            pts = base[rng.integers(0, len(base), n)] if n else np.zeros((0, 2))
        else:
            pts = rng.uniform(0, 4, (n, 2))
        for variant in range(3):       # the base and two moved, noisy, thinned copies of it
            v = pts.copy()
            if variant:
                th = rng.normal(0, 0.05)
                R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
                v = v @ R.T + rng.normal(0, 0.1, 2)
                if kind != 1:
                    v = v + rng.normal(0, 0.005, v.shape)
                v = v[rng.random(len(v)) < 0.9]
            clouds.append((v + centre).astype(np.float32))
            offsets.append(offsets[-1] + len(v))
            family.append(base_id)
    n_scans = len(clouds)
    pts = np.concatenate(clouds).astype(np.float32)
    off = np.array(offsets, np.int64)
    gpu_matcher.upload_scans(pts, off)
    n_pairs = 400
    src = rng.integers(0, n_scans, n_pairs).astype(np.int32)
    tgt = (3 * (src // 3) + rng.integers(0, 3, n_pairs)).astype(np.int32)          # same family (possibly itself)
    far = rng.random(n_pairs) < 0.1
    tgt[far] = rng.integers(0, n_scans, int(far.sum()))                             # some unrelated pairs
    guess = np.zeros((n_pairs, 3), np.float32)
    guess[:, :2] = rng.normal(0, 0.08, (n_pairs, 2))
    guess[:, 2] = rng.normal(0, 0.04, n_pairs)
    for trial in range(10):
        p = Params.defaults(downsample_divisor=int(rng.integers(1, 5)), cov_mode=int(rng.integers(0, 3)),
                            metric=int(rng.integers(0, 2)), use_reciprocal=int(rng.integers(0, 2)),
                            search=int(rng.integers(0, 2)), max_iterations=int(rng.choice([1, 3, 25, 500])),
                            max_correspondence_distance=float(rng.choice([0.05, 0.6, 2.5])),
                            cov_cap=int(rng.choice([0, 5, 200])))
        got = gpu_matcher.submit_pairs(src, tgt, guess, p)
        ref, _ = O.run_batch(pts, off, src, tgt, guess, p, fast=int(rng.integers(0, 2)), threads=0)
        assert_records_match(got, ref, f"random trial {trial}: div {p.downsample_divisor} cov {p.cov_mode} metric {p.metric} "
                                       f"rec {p.use_reciprocal} search {p.search} it {p.max_iterations} gate {p.max_correspondence_distance}")
    with pytest.raises(DpgIcpError) as e:
        gpu_matcher.submit_pairs(src[:1], tgt[:1], guess[:1], Params.defaults(max_correspondence_distance=31.0))
    assert e.value.code == -1


# ---- projective search (north-star extension): bit-exact against its definition in the oracle ------------------------
@pytest.mark.parametrize("window", [3, 8, 40])
@pytest.mark.parametrize("reciprocal", [1, 0])
def test_projective_correspondence_sets_bit_exact_at_every_iterate(gpu_matcher, window, reciprocal):
    wl = synth.config_loop_closure(n_pairs=3, n_scans=16, seed=33)
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    p = Params.defaults(downsample_divisor=1, search=SEARCH_PROJECTIVE, projective_window=window, use_reciprocal=reciprocal,
                        max_iterations=40)
    for k in range(wl.n_pairs):
        s, t = wl.src_idx[k], wl.tgt_idx[k]
        src, tgt = pts[off[s]:off[s + 1]], pts[off[t]:off[t + 1]]
        _, iterates, n_corr = O.icp(src, tgt, wl.guess[k], p, trace=True)
        for it in sorted(set([0, 1, 2, len(iterates) // 2, len(iterates) - 1])):
            T = iterates[it]
            cur = O.transform_points(T, src)
            kk, want, want_d2 = O.correspondences(cur, tgt, p, src_orig=src, T=T)
            got, got_d2 = gpu_matcher.correspondences(src, tgt, T, p)
            assert np.array_equal(got, want), (k, it)
            m = want >= 0
            assert np.array_equal(got_d2[m].view(np.uint32), want_d2[m].view(np.uint32)), (k, it)
            assert int((got >= 0).sum()) == kk


@pytest.mark.parametrize("divisor", [1, 5])
@pytest.mark.parametrize("metric", [0, METRIC_POINT_TO_LINE])
def test_projective_batches(gpu_matcher, divisor, metric):
    wl = synth.config_corridor(n_pairs=64, seed=2)
    for cov_mode in (COV_CENSI_CORR, COV_CENSI_INDEXPAIR):
        p = Params.defaults(downsample_divisor=divisor, search=SEARCH_PROJECTIVE, cov_mode=cov_mode, metric=metric)
        got, ref, _, _ = run_both(gpu_matcher, wl, p)
        assert_records_match(got, ref, f"projective corridor d{divisor} m{metric} c{cov_mode}")
    wl = synth.config_loop_closure(n_pairs=96, n_scans=40, seed=3)
    p = Params.defaults(downsample_divisor=divisor, search=SEARCH_PROJECTIVE, cov_mode=COV_CENSI_CORR, metric=metric,
                        projective_window=12, use_reciprocal=divisor == 1)
    got, ref, _, _ = run_both(gpu_matcher, wl, p)
    assert_records_match(got, ref, f"projective loop closure d{divisor} m{metric}")


def test_projective_random_small_problems_and_sensor_origins(gpu_matcher):
    """Ragged, empty, duplicated and lattice clouds (keys not sorted, exact ties), random windows and sensor origins."""
    rng = np.random.default_rng(77)
    clouds, offsets = [], [0]
    for base_id in range(30):
        n = int(rng.choice([0, 1, 2, 3, 5, 31, 32, 33, 64, 100, 150]))
        kind = base_id % 3
        if kind == 0:
            t = np.sort(rng.uniform(0, 6, n))
            pts = np.stack([t, 0.3 * np.sin(t)], 1)
        elif kind == 1:
            pts = np.stack([rng.integers(0, 8, n) * 0.25, rng.integers(0, 8, n) * 0.25], 1).astype(float)
        else:
            pts = rng.uniform(-3, 3, (n, 2))
        for variant in range(2):
            v = pts + (rng.normal(0, 0.05, 2) if variant else 0.0)
            clouds.append(v.astype(np.float32))
            offsets.append(offsets[-1] + len(v))
    pts = np.concatenate(clouds).astype(np.float32)
    off = np.array(offsets, np.int64)
    gpu_matcher.upload_scans(pts, off)
    n_pairs = 240
    src = rng.integers(0, len(clouds), n_pairs).astype(np.int32)
    tgt = (2 * (src // 2) + rng.integers(0, 2, n_pairs)).astype(np.int32)
    guess = np.concatenate([rng.normal(0, 0.05, (n_pairs, 2)), rng.normal(0, 0.03, (n_pairs, 1))], 1).astype(np.float32)
    for trial in range(6):
        p = Params.defaults(downsample_divisor=int(rng.integers(1, 4)), cov_mode=int(rng.integers(0, 3)),
                            metric=int(rng.integers(0, 2)), use_reciprocal=int(rng.integers(0, 2)), search=SEARCH_PROJECTIVE,
                            projective_window=int(rng.choice([1, 2, 7, 33, 1024])), sensor_x=float(rng.uniform(-1, 1)),
                            sensor_y=float(rng.uniform(-1, 1)), max_iterations=int(rng.choice([1, 4, 60])),
                            max_correspondence_distance=float(rng.choice([0.05, 0.6, 2.5])))
        got = gpu_matcher.submit_pairs(src, tgt, guess, p)
        ref, _ = O.run_batch(pts, off, src, tgt, guess, p, fast=0, threads=0)
        assert_records_match(got, ref, f"projective random trial {trial}: W {p.projective_window} div {p.downsample_divisor}")
    for bad in (dict(projective_window=0), dict(projective_window=2000), dict(sensor_x=float("nan"))):
        with pytest.raises(DpgIcpError) as e:
            gpu_matcher.submit_pairs(src[:1], tgt[:1], guess[:1], Params.defaults(search=SEARCH_PROJECTIVE, **bad))
        assert e.value.code == -1


def test_projective_staged_chain_equals_single_stage(gpu_matcher, monkeypatch):
    """Suspend/resume recomputes the beam-order keys from the store: any chain gives the single-stage records."""
    from dpg_slam_b200.scanmatch import ScanMatcher
    wl = synth.config_corridor(n_pairs=300, n_beams=721, seed=21)
    p = Params.defaults(downsample_divisor=1, search=SEARCH_PROJECTIVE, cov_mode=COV_CENSI_CORR)
    out = {}
    for chain in ("16", "2,4,16", "1,4,9x4"):
        monkeypatch.setenv("DPGICP_CHAIN", chain)
        with ScanMatcher(0) as sm:
            sm.upload_ranges(wl.ranges, wl.scanner)
            out[chain] = sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p).copy()
    p5 = p.copy(downsample_divisor=5, projective_window=5)
    with ScanMatcher(0) as sm:                      # chain "1,4,9x4": resumed pairs re-gather the down-sampled originals
        sm.upload_ranges(wl.ranges, wl.scanner)
        chained5 = sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p5).copy()
    monkeypatch.setenv("DPGICP_CHAIN", "16")
    with ScanMatcher(0) as sm:
        sm.upload_ranges(wl.ranges, wl.scanner)
        assert sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p5).tobytes() == chained5.tobytes()
    monkeypatch.delenv("DPGICP_CHAIN")
    assert out["16"].tobytes() == out["2,4,16"].tobytes() == out["1,4,9x4"].tobytes()
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    ref, _ = O.run_batch(pts, off, wl.src_idx[:60], wl.tgt_idx[:60], wl.guess[:60], p, fast=0, threads=0)
    assert_records_match(out["16"][:60], ref, "projective chain")


# ---- the two reference call shapes -------------------------------------------------------------------------------
def test_run_icp_call_shape(gpu_matcher):
    wl = synth.config_room_pair()
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    node_1, node_2 = pts[off[0]:off[1]], pts[off[1]:off[2]]
    from dpg_slam_b200.scanmatch import relative_guess
    guess = relative_guess([0, 0, 0], [0.35, -0.15, 0.12])
    converged, ((tx, ty), theta), cov, rec = gpu_matcher.run_icp(node_1, node_2, guess)      # reference defaults
    ref = O.run_pair(node_2, node_1, guess, Params.defaults())
    assert converged == bool(ref.status & FLAG_CONVERGED)
    assert (tx, ty, rec.iterations, rec.status) == (ref.tx, ref.ty, ref.iterations, ref.status)
    assert abs(theta - ref.theta) <= POSE_TOL_RAD
    assert np.array_equal(cov, np.diag([0.5, 0.5, np.float64(np.float32(0.3))]))   # live output, cov.h:572-575


def test_calculate_icp_cov_against_compiled_reference(gpu_matcher, cov_golden):
    """dpgicp_cov vs the golden vectors produced by the reference's own cov_func_point_to_point.h."""
    for c in cov_golden:
        T = c["T_colmajor"].reshape(4, 4).T
        live = Params.defaults(cov_mode=COV_REFERENCE_LIVE, laser_x_variance=c["live_in"][0],
                               laser_y_variance=c["live_in"][1], laser_theta_variance=c["live_in"][2])
        cov, st = gpu_matcher.calculate_icp_cov(c["P"], c["Q"], T, live)
        assert np.array_equal(cov, c["live_cov"]), c["name"]                      # bit-exact live output
        if c["singular"]:
            continue
        cov, st = gpu_matcher.calculate_icp_cov(c["P"], c["Q"], T, live.copy(cov_mode=COV_CENSI_INDEXPAIR))
        rel = np.abs(cov - c["cov3"]).max() / np.abs(c["cov3"]).max()
        assert st == 0 and rel <= COV_REL_TOL, (c["name"], rel)
        assert rel < 1e-7, (c["name"], rel)                                       # in practice: double rounding only (n = 3 is ill-conditioned)


def test_batched_covariance_over_the_store(gpu_matcher):
    """dpgicp_cov_pairs == the oracle's index-paired Censi form per item (and == the single-item call)."""
    wl = synth.config_corridor(n_pairs=50, n_beams=721, seed=27)
    wl.ranges[3, ::3] = 40.0                                        # clouds of different lengths
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    pts, off = gpu_matcher.download_store()
    rng = np.random.default_rng(5)
    th = rng.normal(0, 0.05, 50).astype(np.float32)
    T = np.stack([np.cos(th.astype(np.float64)).astype(np.float32), np.sin(th.astype(np.float64)).astype(np.float32),
                  wl.truth[:, 0].astype(np.float32), wl.truth[:, 1].astype(np.float32)], 1)
    p = Params.defaults(cov_mode=COV_CENSI_INDEXPAIR)
    cov, st, ms = gpu_matcher.calculate_icp_cov_pairs(wl.src_idx, wl.tgt_idx, T, p)
    assert ms > 0 and cov.shape == (50, 3, 3)
    for k in range(50):
        P = pts[off[wl.src_idx[k]]:off[wl.src_idx[k] + 1]]
        Q = pts[off[wl.tgt_idx[k]]:off[wl.tgt_idx[k] + 1]]
        nh = min(len(P), len(Q))
        s_ref, want, _ = O.cov_censi(P, Q, nh, min(nh, 200), T[k])
        assert st[k] == s_ref
        rel = np.abs(cov[k] - want).max() / np.abs(want).max()
        assert rel <= COV_REL_TOL and rel < 1e-7, (k, rel)
    live, st, _ = gpu_matcher.calculate_icp_cov_pairs(wl.src_idx, wl.tgt_idx, T, Params.defaults())
    assert np.all(live == np.diag([0.5, 0.5, np.float64(np.float32(0.3))]))
    with pytest.raises(DpgIcpError):
        gpu_matcher.calculate_icp_cov_pairs([99], [0], T[:1], p)


def test_enumerate_pairs_matches_oracle(gpu_matcher):
    rng = np.random.default_rng(17)
    for n in (0, 1, 2, 3, 200, 1500):
        xy = rng.uniform(0, 30, (n, 2)).astype(np.float32)
        ps = (np.arange(n) // 400).astype(np.int32)
        src, tgt = gpu_matcher.enumerate_pairs(xy, ps, 5.0, 2.0)
        wsrc, wtgt = O.enumerate_pairs(xy, ps, 5.0, 2.0)
        assert np.array_equal(src, wsrc) and np.array_equal(tgt, wtgt), n


def test_factor_handoff_matches_oracle(gpu_matcher):
    """addObservationConstraint hand-off (dpg_slam.cc:331-338): from/to, Pose2, sqrt information R with
    R^T R = cov^-1; bit-exact against the oracle applied to the same records."""
    wl = synth.config_loop_closure(n_pairs=300, n_scans=100, seed=41)
    wl.guess[7] = (70.0, 70.0, 0.0)                                   # a pair with no correspondences
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    for cov_mode in (COV_CENSI_CORR, COV_REFERENCE_LIVE):
        p = Params.defaults(downsample_divisor=1, cov_mode=cov_mode)
        rec = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
        got = gpu_matcher.fetch_factors()
        want = O.factors(rec, wl.src_idx, wl.tgt_idx)
        assert got.tobytes() == want.tobytes()
        assert np.array_equal(got["from_node"], wl.tgt_idx) and np.array_equal(got["to_node"], wl.src_idx)
        ok = (got["status"] & _abi.FLAG_FACTOR_INVALID) == 0
        assert ok.all()
        R = got["sqrt_info"].reshape(-1, 3, 3)
        info = np.einsum("kji,kjl->kil", R, R)
        cov = rec["cov"].reshape(-1, 3, 3)
        eye = np.einsum("kij,kjl->kil", info, cov)
        assert np.abs(eye - np.eye(3)).max() < 1e-6
        assert np.all(np.tril(R, -1) == 0)
    # a covariance that is not positive definite is flagged and zeroed, never passed on
    assert gpu_matcher.fetch_factors(0).shape == (0,)


def test_config5_multisession_gated_pairs(gpu_matcher):
    """BASELINE config 5 shape at oracle size: sessions on a shared, partly changed world; candidate pairs from
    the callers' distance gate (5 m same pass / 2 m across passes) enumerated on the device; guesses from the
    drifted node estimates exactly as runIcp derives them."""
    from dpg_slam_b200.scanmatch import relative_guess
    wl = synth.config_multisession(n_sessions=3, scans_per_session=60, n_beams=541, seed=5, size=30.0, n_boxes=30)
    src, tgt = gpu_matcher.enumerate_pairs(wl.poses_est[:, :2], wl.passes, 5.0, 2.0)
    wsrc, wtgt = O.enumerate_pairs(wl.poses_est[:, :2], wl.passes, 5.0, 2.0)
    assert np.array_equal(src, wsrc) and np.array_equal(tgt, wtgt) and len(src) > 180
    guess = np.stack([relative_guess(wl.poses_est[t], wl.poses_est[s]) for s, t in zip(src, tgt)])
    og = np.stack([O.relative_guess(wl.poses_est[t, :2], float(wl.poses_est[t, 2]), wl.poses_est[s, :2],
                                    float(wl.poses_est[s, 2])) for s, t in zip(src, tgt)])
    assert guess.tobytes() == og.tobytes()
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    pts, off = gpu_matcher.download_store()
    for metric in (0, METRIC_POINT_TO_LINE):
        p = Params.defaults(cov_mode=COV_CENSI_CORR, metric=metric)          # reference defaults: divisor 5
        got = gpu_matcher.submit_pairs(src, tgt, guess, p)
        ref, _ = O.run_batch(pts, off, src, tgt, guess, p, fast=1, threads=0)
        assert_records_match(got, ref, f"multisession m{metric}")


# ---- size-independent properties at full batch sizes ------------------------------------------------------------
def test_full_size_batch_properties(gpu_matcher):
    """BASELINE config 2 at full size (5000 pairs, 1081 beams): the oracle checks a strided sample; the
    whole batch is checked through properties: brute == pruned, batch == one-at-a-time, permutation
    invariance, SPD covariances, truth recovered."""
    wl = synth.config_corridor(n_pairs=5000, seed=2)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    got = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    # (1) oracle on a strided sample
    pts, off = gpu_matcher.download_store()
    idx = np.arange(0, 5000, 97)
    ref, _ = O.run_batch(pts, off, wl.src_idx[idx], wl.tgt_idx[idx], wl.guess[idx], p, fast=1, threads=0)
    assert_records_match(got[idx], ref, "config2 sample")
    # (2) exhaustive search gives the same bits as the pruned search
    brute = gpu_matcher.submit_pairs(wl.src_idx[:600], wl.tgt_idx[:600], wl.guess[:600], p.copy(search=SEARCH_BRUTE))
    assert brute.tobytes() == got[:600].tobytes()
    # (3) permutation invariance / no cross-pair state
    perm = np.random.default_rng(0).permutation(5000)
    shuf = gpu_matcher.submit_pairs(wl.src_idx[perm], wl.tgt_idx[perm], wl.guess[perm], p)
    assert shuf.tobytes() == got[perm].tobytes()
    # (4) one-at-a-time equals the batch
    for k in (0, 1234, 4999):
        one = gpu_matcher.submit_pairs(wl.src_idx[k:k + 1], wl.tgt_idx[k:k + 1], wl.guess[k:k + 1], p)
        assert one.tobytes() == got[k:k + 1].tobytes()
    # (5) covariances symmetric positive definite where not flagged
    ok = (got["status"] & FLAG_COV_SINGULAR) == 0
    covs = got["cov"][ok].reshape(-1, 3, 3)
    assert np.allclose(covs, covs.transpose(0, 2, 1), rtol=1e-9, atol=1e-18)
    assert np.all(np.linalg.eigvalsh(0.5 * (covs + covs.transpose(0, 2, 1))) > 0)
    # (6) rotation and lateral offset recovered (the corridor axis is weakly observable)
    conv = (got["status"] & FLAG_CONVERGED) != 0
    assert conv.mean() > 0.99
    assert np.median(np.abs(got["theta"] - wl.truth[:, 2])) < 5e-3
    assert np.median(np.abs(got["ty"] - wl.truth[:, 1])) < 2e-2


def gpu_matcher_records(gpu_matcher, wl, p):
    """records from the session-wide matcher (default chain, created before any env override)"""
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    return gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)


def test_staged_chain_equals_single_stage(gpu_matcher, monkeypatch):
    """The kernel runs as a chain of stages (narrow CTAs first; pairs still running when a stage's queue
    runs dry are suspended to HBM and resumed by wider CTAs).  Suspension restores state bit for bit,
    so any chain length and any CTA width must give identical records."""
    from dpg_slam_b200.scanmatch import ScanMatcher
    wl = synth.config_corridor(n_pairs=1500, seed=23)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    want = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    for chain in ("4", "2,4", "1,2,16", "8,16,16x4", "16", "3,5,11,32", "4,8,16,32", "1,32", "32",
                  # last stage as thread-block clusters: 2 or 4 CTAs (SMs) per pair, partial sums through DSMEM
                  "4,8,16,9x2", "4,8,9x4", "2,5x2", "4,16x4"):
        monkeypatch.setenv("DPGICP_CHAIN", chain)
        with ScanMatcher(0) as sm:
            sm.upload_ranges(wl.ranges, wl.scanner)
            got = sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
            assert got.tobytes() == want.tobytes(), chain
            c = sm.last_run_counters()
            assert c["iterations"] == int(got["iterations"].sum())
    # the hand-over rule (a stage suspends its pairs once its queue is dry AND few enough are left for the next stage)
    # only moves the moment of suspension
    monkeypatch.delenv("DPGICP_CHAIN")
    for handover in ("0", "0.5,0.5", "1.0,3.0", "4"):
        monkeypatch.setenv("DPGICP_HANDOVER", handover)
        with ScanMatcher(0) as sm:
            sm.upload_ranges(wl.ranges, wl.scanner)
            assert sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p).tobytes() == want.tobytes(), handover
    monkeypatch.delenv("DPGICP_HANDOVER")
    # down-sampled clouds take the gather path when fresh and the contiguous path when resumed
    p5 = p.copy(downsample_divisor=5)
    want5 = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p5)
    monkeypatch.setenv("DPGICP_CHAIN", "2")
    with ScanMatcher(0) as sm:
        sm.upload_ranges(wl.ranges, wl.scanner)
        assert sm.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p5).tobytes() == want5.tobytes()
    # clusters with every covariance mode and metric, ragged and empty scans, small batches (all pairs reach the cluster stage)
    wl2 = synth.config_corridor(n_pairs=40, n_beams=721, seed=12)
    wl2.ranges[2, :] = 40.0
    wl2.ranges[4, 2:] = 40.0
    wl2.ranges[6, ::2] = 40.0
    for chain in ("4,8,9x2", "2,6x4"):
        monkeypatch.setenv("DPGICP_CHAIN", chain)
        with ScanMatcher(0) as sm:
            sm.upload_ranges(wl2.ranges, wl2.scanner)
            for cov_mode in (COV_REFERENCE_LIVE, COV_CENSI_INDEXPAIR, COV_CENSI_CORR):
                for metric, div in ((0, 1), (METRIC_POINT_TO_LINE, 1), (0, 5)):
                    pc = Params.defaults(downsample_divisor=div, cov_mode=cov_mode, metric=metric)
                    got = sm.submit_pairs(wl2.src_idx, wl2.tgt_idx, wl2.guess, pc)
                    ref = gpu_matcher_records(gpu_matcher, wl2, pc)
                    assert got.tobytes() == ref.tobytes(), (chain, cov_mode, metric, div)


def test_cost_hints_change_the_schedule_not_the_results(gpu_matcher):
    wl = synth.config_corridor(n_pairs=1200, seed=29)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    want = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    gpu_matcher.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
    for hints in (want["iterations"].astype(np.float32), -want["iterations"].astype(np.float32),
                  np.random.default_rng(1).random(1200).astype(np.float32)):
        gpu_matcher.set_pair_cost_hints(hints)
        gpu_matcher.run(p)
        assert gpu_matcher.fetch_results().tobytes() == want.tobytes()
    gpu_matcher.set_pair_cost_hints(None)
    with pytest.raises(DpgIcpError):
        gpu_matcher.set_pair_cost_hints(np.zeros(5, np.float32))


def test_rotation_entries_stay_orthonormal(gpu_matcher):
    wl = synth.config_loop_closure(n_pairs=2000, n_scans=400, seed=13)
    p = Params.defaults(downsample_divisor=5)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    got = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    n = got["rot_c"].astype(np.float64) ** 2 + got["rot_s"].astype(np.float64) ** 2
    assert np.max(np.abs(n - 1.0)) < 1e-4                # float composition over <= 500 steps
    assert np.all(np.abs(np.arctan2(got["rot_s"], got["rot_c"]) - got["theta"]) <= POSE_TOL_RAD)


def test_stream_and_resident_api(gpu_matcher):
    import torch
    wl = synth.config_corridor(n_pairs=40, n_beams=541, seed=19)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    want = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
    s = torch.cuda.Stream()
    gpu_matcher.set_stream(s.cuda_stream)
    try:
        gpu_matcher.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        gpu_matcher.run(p)
        e1.record(s)
        got = gpu_matcher.fetch_results()
        assert e0.elapsed_time(e1) > 0
        assert got.tobytes() == want.tobytes()
        c = gpu_matcher.last_run_counters()
        assert c["iterations"] == int(got["iterations"].sum()) and c["distance_evals"] > 0
        ptr, n = gpu_matcher.results_device_ptr()
        assert ptr != 0 and n == 40
    finally:
        gpu_matcher.set_stream(None)


def test_cpp_batch_runner_equals_python_path(gpu_matcher, tmp_path):
    """The C++ host path (dpgicp_shim.hpp + dpg_batch_runner: scan log -> enumerate -> guesses -> one batch -> CSV) gives
    the same records as the Python mirror driving the same C ABI."""
    import os
    import struct
    import subprocess
    from dpg_slam_b200.scanmatch import relative_guess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "dpg_slam_b200", "dpg_batch_runner")
    log, csv_path = str(tmp_path / "scans.bin"), str(tmp_path / "out.csv")
    r = subprocess.run([exe, "--synthetic", "corridor", "--scans", "60", "--passes", "2", "--beams", "541", "--cov-mode", "2",
                        "--write-log", log, "--out", csv_path], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    import json
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    # read the scan log (format documented in dpg_batch_runner.cc)
    raw = open(log, "rb").read()
    assert raw[:8] == b"DPGSCAN1"
    n_scans, n_beams = struct.unpack_from("<ii", raw, 8)
    amin, amax, rmax, lx, ly, lt = struct.unpack_from("<6f", raw, 16)
    rec_bytes = 12 + 4 + 4 * n_beams
    est = np.zeros((n_scans, 3), np.float32); passes = np.zeros(n_scans, np.int32); ranges = np.zeros((n_scans, n_beams), np.float32)
    for s in range(n_scans):
        o = 40 + s * rec_bytes
        est[s] = struct.unpack_from("<3f", raw, o)
        passes[s] = struct.unpack_from("<i", raw, o + 12)[0]
        ranges[s] = np.frombuffer(raw, np.float32, n_beams, o + 16)
    sc = synth.Scanner(n_beams=n_beams, angle_min=amin, angle_max=amax, range_max=rmax, laser_x=lx, laser_y=ly, laser_theta=lt)
    gpu_matcher.upload_ranges(ranges, sc)
    src, tgt = gpu_matcher.enumerate_pairs(est[:, :2], passes, 5.0, 2.0)
    guess = np.stack([relative_guess(est[t], est[s]) for s, t in zip(src, tgt)])
    p = Params.defaults(cov_mode=COV_CENSI_CORR)                                   # runner defaults + --cov-mode 2
    got = gpu_matcher.submit_pairs(src, tgt, guess, p)
    rows = [ln.split(",") for ln in open(csv_path).read().strip().splitlines()[1:]]
    assert len(rows) == len(src) == summary["pairs"]
    for k, row in enumerate(rows):
        assert int(row[0]) == src[k] and int(row[1]) == tgt[k]
        assert np.float32(row[2]) == got["tx"][k] and np.float32(row[3]) == got["ty"][k] and np.float32(row[4]) == got["theta"][k]
        assert np.array_equal(np.array(row[5:14], np.float64), got["cov"][k])
        assert int(row[14]) == got["iterations"][k] and int(row[15]) == got["status"][k]
