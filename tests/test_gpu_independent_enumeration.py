"""GPU (B200): candidate-pair enumeration on the device against the independent reference (``ref_enumeration``), not
the oracle, bit for bit — pair lists of both modes, every guess entry, the host-list form, shards, boundary guesses
beyond any fixed list size, the node table after a host-list call, and one enumerate -> run -> fetch."""
import numpy as np
import pytest

import enum_cases as EC
import ref_enumeration as R
from dpg_slam_b200 import synth
from dpg_slam_b200._abi import COV_CENSI_CORR, ENUM_ONLINE, ENUM_REOPTIMIZE, Params
from dpg_slam_b200.scanmatch import DpgIcpError
from oracle import oracle_py as O
from test_gpu_parity import assert_records_match

pytestmark = pytest.mark.gpu
F32 = np.float32


def _reference(c, online=False, method="auto"):
    xy = c["poses"][:, :2]
    if online:
        return R.enumerate_online(xy, c["passes"], c["r_same"], c["r_other"])
    return R.enumerate_reoptimize(xy, c["passes"], c["r_same"], c["r_other"], method=method)


def _check_device(sm, c, online=False, rank=0, world=1, host_list=True, ref=None):
    """set_nodes + enumerate_pairs_device + fetch_pairs == the reference (indices and every T entry)"""
    ws, wt = ref if ref is not None else _reference(c, online)
    sm.set_nodes(c["poses"], c["passes"])
    total, local = sm.enumerate_pairs_device(ENUM_ONLINE if online else ENUM_REOPTIMIZE, c["r_same"], c["r_other"], rank, world)
    ls, lt = ws[rank::world], wt[rank::world]
    assert total == len(ws) and local == len(ls), (c["name"], total, local, len(ws))
    src, tgt, T = sm.fetch_pairs()
    assert np.array_equal(src, ls) and np.array_equal(tgt, lt), c["name"]
    _, wT = R.guesses(c["poses"], ls, lt)
    if T.tobytes() != wT.tobytes():
        bad = np.nonzero((T.view(np.uint32) != wT.view(np.uint32)).any(1))[0]
        raise AssertionError(f"{c['name']}: {len(bad)} guesses differ, first pair {bad[0]}: {T[bad[0]]} vs {wT[bad[0]]}")
    if host_list and not online and world == 1:
        s2, t2 = sm.enumerate_pairs(c["poses"][:, :2], c["passes"], c["r_same"], c["r_other"])
        assert np.array_equal(s2, ws) and np.array_equal(t2, wt), c["name"]
    return ws, wt, T


_GROUPS = {
    "tie345": EC.tie_345_cases,
    "ties": EC.tie_cases,
    "passes_radii": EC.pass_radius_cases,
    "geometry": EC.geometry_cases,
    "angles": lambda: [EC.angle_case(extra=[0.11056483, -0.31426188, 1.0480543, -1.0480543, 1e4 + 0.31426188])],
}


@pytest.mark.parametrize("group", list(_GROUPS))
def test_device_reoptimize_equals_reference(gpu_matcher, group):
    for c in _GROUPS[group]():
        _check_device(gpu_matcher, c)


@pytest.mark.parametrize("n", EC.SIZES)
def test_device_reoptimize_sizes_equal_reference(gpu_matcher, n):
    """hierarchy level boundaries: 32/33 nodes (one leaf), 1024/1025 (two levels), 32768/32769 (three levels)"""
    _check_device(gpu_matcher, EC.size_case(n), host_list=n <= 1025 or n == 32769)


def test_device_reoptimize_four_levels_equals_reference(gpu_matcher):
    c = EC.four_level_case()
    ref = _reference(c, method="kd")
    assert len(ref[0]) > 3 * len(c["passes"])
    _check_device(gpu_matcher, c, host_list=False, ref=ref)


def test_device_online_equals_reference(gpu_matcher):
    cases = [EC.online_size_case(n) for n in EC.ONLINE_SIZES + [2, 3, 4, 5]]
    cases += EC.tie_cases(online=True) + EC.tie_345_cases() + EC.pass_radius_cases() + EC.geometry_cases()
    cases.append(EC.angle_case(extra=[0.11056483, -0.31426188]))
    for c in cases:
        _check_device(gpu_matcher, c, online=True)


def test_device_shards_partition_the_list(gpu_matcher):
    """world 1..8: each shard is global[rank::world], also for lists shorter than world; an empty shard's batch runs
    and fetches cleanly"""
    wl = synth.config_corridor(n_pairs=4, seed=3)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    p = Params.defaults()
    for c in [EC.size_case(2), EC.size_case(3), EC.size_case(5), EC.pass_radius_cases()[1], EC.angle_case()]:
        ws, wt = _reference(c)
        for world in range(1, 9):
            seen = np.zeros(len(ws), np.int64)
            for rank in range(world):
                _check_device(gpu_matcher, c, rank=rank, world=world, host_list=False, ref=(ws, wt))
                seen[rank::world] += 1
                if len(ws[rank::world]) == 0:
                    gpu_matcher.run(p)
                    assert len(gpu_matcher.fetch_results()) == 0 and len(gpu_matcher.fetch_factors()) == 0
                    assert all(len(a) == 0 for a in gpu_matcher.fetch_pairs())
            assert np.all(seen == 1)


def _boundary_pairs(c, src, tgt):
    g, _ = R.guesses(c["poses"], src, tgt)
    g2 = g[:, 2].astype(np.float64)
    return int((R.near_boundary(np.cos(g2)) | R.near_boundary(np.sin(g2))).sum())


@pytest.mark.parametrize("angle", [0.11056483, 0.31426188, 1.0480543])
def test_device_boundary_guesses_beyond_4096(gpu_matcher, angle):
    """200 nodes within 1 m in one pass, theta alternating 0 and a boundary angle: about 10 000 pairs whose guess cos or
    sin lies next to a binary32 rounding midpoint.  The whole list and one shard of a 2-way split (each > 4096 such
    pairs) enumerate, and every c, s equals the host libm's"""
    c = EC.boundary_heading_case([angle], n=200, name=f"boundary_{angle}")
    ws, wt = _reference(c)
    assert _boundary_pairs(c, ws, wt) > 8192
    assert _boundary_pairs(c, ws[1::2], wt[1::2]) > 4096
    _check_device(gpu_matcher, c)
    _check_device(gpu_matcher, c, rank=1, world=2)
    _check_device(gpu_matcher, c, online=True)


def test_device_boundary_angles_from_the_finder(gpu_matcher):
    """every boundary angle of (0.05, 3.0) and its negative as headings of one cluster"""
    angles = R.boundary_angles(0.05, 3.0)
    assert len(angles) >= 8
    c = EC.boundary_heading_case(np.concatenate([angles, -angles]), n=240, name="finder_headings")
    ws, wt = _reference(c)
    assert _boundary_pairs(c, ws, wt) > 1000
    _check_device(gpu_matcher, c)


def test_host_list_form_leaves_the_node_table_and_batch(gpu_matcher):
    """set_nodes(A), enumerate on the device, run; the host-list enumerate_pairs(B) must leave A's table and the batch
    as they were: the batch fetches and runs unchanged, and a new device enumeration equals the reference on A"""
    wl = synth.config_multisession(n_sessions=2, scans_per_session=40, n_beams=361, seed=8, size=25.0, n_boxes=20)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    A = EC.case("A", wl.poses_est, wl.passes, 5.0, 2.0)
    A["poses"][1::3, 2] = F32(0.11056483)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    ws, wt, T0 = _check_device(gpu_matcher, A, host_list=False)
    gpu_matcher.run(p)
    rec0 = gpu_matcher.fetch_results()
    B = EC.size_case(1025)
    s2, t2 = gpu_matcher.enumerate_pairs(B["poses"][:, :2], B["passes"], 5.0, 2.0)
    wbs, wbt = _reference(B)
    assert np.array_equal(s2, wbs) and np.array_equal(t2, wbt)
    src, tgt, T = gpu_matcher.fetch_pairs()
    assert np.array_equal(src, ws) and np.array_equal(tgt, wt) and T.tobytes() == T0.tobytes()
    gpu_matcher.run(p)
    assert gpu_matcher.fetch_results().tobytes() == rec0.tobytes()
    total, local = gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0)
    assert total == local == len(ws)
    src, tgt, T = gpu_matcher.fetch_pairs()
    assert np.array_equal(src, ws) and np.array_equal(tgt, wt) and T.tobytes() == T0.tobytes()


@pytest.mark.parametrize("r_same,r_other", [(float("nan"), 2.0), (5.0, float("nan")), (-1.0, 2.0), (5.0, -0.5),
                                            (-float("inf"), 1.0)])
def test_invalid_radii_are_refused_in_both_forms(gpu_matcher, r_same, r_other):
    c = EC.size_case(33)
    gpu_matcher.set_nodes(c["poses"], c["passes"])
    for call in (lambda: gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, r_same, r_other),
                 lambda: gpu_matcher.enumerate_pairs(c["poses"][:, :2], c["passes"], r_same, r_other),
                 lambda: gpu_matcher.enumerate_pairs(c["poses"][:1, :2], c["passes"][:1], r_same, r_other)):
        with pytest.raises(DpgIcpError) as e:
            call()
        assert e.value.code == -1


def test_end_to_end_with_boundary_headings(gpu_matcher):
    """a small multisession store whose headings include boundary angles: enumerate -> run -> fetch_results /
    fetch_factors equals the oracle's run_batch on the reference's pair list and guesses"""
    wl = synth.config_multisession(n_sessions=3, scans_per_session=40, n_beams=541, seed=6, size=30.0, n_boxes=30)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    pts, off = gpu_matcher.download_store()
    poses = wl.poses_est.astype(F32).copy()
    poses[:, 2] = F32(0.0)                               # a pair of headings 0 and g has the boundary angle +-g
    poses[::4, 2] = F32(0.11056483)
    poses[2::4, 2] = F32(-1.0480543)
    c = EC.case("e2e", poses, wl.passes, 5.0, 2.0)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    for mode in (ENUM_REOPTIMIZE, ENUM_ONLINE):
        ws, wt, _ = _check_device(gpu_matcher, c, online=mode == ENUM_ONLINE, host_list=False)
        gpu_matcher.run(p)
        got = gpu_matcher.fetch_results()
        fac = gpu_matcher.fetch_factors()
        guess, _ = R.guesses(poses, ws, wt)
        ref, _ = O.run_batch(pts, off, ws, wt, guess, p, fast=1, threads=0)
        assert_records_match(got, ref, f"enumerated with boundary headings, mode {mode}")
        assert np.array_equal(fac["from_node"], wt) and np.array_equal(fac["to_node"], ws)
        if mode == ENUM_REOPTIMIZE:
            assert _boundary_pairs(c, ws, wt) > 0
