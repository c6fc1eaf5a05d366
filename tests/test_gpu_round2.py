"""GPU (B200): ABI v3 features against the CPU oracle, through the C ABI — the sticky tie rule with seeds, the outlier
rejectors, the device-resident caller forms (node table -> pair list + guesses enumerated on the device, reoptimize and
online shapes, sharded), conversion of device-resident ranges, the single-process multi-context gather (two contexts on
one GPU), stage timing."""
import ctypes as C
import os
import subprocess
import time

import numpy as np
import pytest

from dpg_slam_b200 import _abi, synth
from dpg_slam_b200._abi import (COV_CENSI_CORR, COV_CENSI_INDEXPAIR, ENUM_ONLINE, ENUM_REOPTIMIZE, METRIC_POINT_TO_LINE, OUTLIER_MEDIAN,
                                OUTLIER_TRIMMED, SEARCH_BRUTE, SEARCH_PROJECTIVE, SEARCH_PRUNED, Params)
from dpg_slam_b200.scanmatch import DpgIcpError, ScanMatcher, relative_guess
from oracle import oracle_py as O
from test_gpu_parity import assert_records_match

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- tie rule ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("search", [SEARCH_BRUTE, SEARCH_PRUNED])
@pytest.mark.parametrize("reciprocal", [1, 0])
def test_seeded_correspondences_follow_the_sticky_tie_rule(gpu_matcher, search, reciprocal):
    """Lattice clouds (many exact distance ties) with random seeds: previous neighbour among the minimisers wins, else the
    lowest index; the reciprocal test keeps every asker of an exact tie.  Both the accepted set and the neighbours
    handed to the next pass must equal the oracle's."""
    rng = np.random.default_rng(77 + search + 2 * reciprocal)
    T = np.array([1, 0, 0, 0], np.float32)
    for trial in range(12):
        nt, ns = int(rng.integers(1, 400)), int(rng.integers(1, 400))
        tgt = np.stack([rng.integers(0, 12, nt) * 0.25, rng.integers(0, 9, nt) * 0.25], 1).astype(np.float32)
        src = np.stack([rng.integers(0, 23, ns) * 0.125, rng.integers(0, 17, ns) * 0.125], 1).astype(np.float32)
        prev = rng.integers(-1, nt, ns).astype(np.int32)
        p = Params.defaults(search=search, use_reciprocal=reciprocal, max_correspondence_distance=float(rng.choice([0.2, 0.6, 1.5])))
        kk, want, want_d2, want_nn = O.correspondences(src, tgt, p, prev_nn=prev)
        got, got_d2, got_nn = gpu_matcher.correspondences_seeded(src, tgt, T, p, prev)
        assert np.array_equal(got, want), (trial, np.nonzero(got != want)[0][:5])
        assert np.array_equal(got_nn, want_nn), trial
        m = want_nn >= 0
        assert np.array_equal(got_d2[m].view(np.uint32), want_d2[m].view(np.uint32))
    with pytest.raises(DpgIcpError):
        gpu_matcher.correspondences_seeded(src, tgt, T, p, np.full(ns, nt, np.int32))          # seed out of range


def test_sticky_rule_over_whole_runs_with_ties(gpu_matcher):
    """Whole ICP runs on lattice / duplicated clouds: the history-dependent tie rule has to be carried identically by
    both sides through every pass, the suspended-pair state and the covariance pass."""
    rng = np.random.default_rng(123)
    clouds, offsets = [], [0]
    for k in range(30):
        n = int(rng.integers(20, 300))
        base = np.stack([rng.integers(0, 16, n) * 0.125, rng.integers(0, 10, n) * 0.125], 1)
        if k % 3 == 0:
            base = base[rng.integers(0, n, n)]                                           # duplicates
        shift = rng.integers(-2, 3, 2) * 0.125 if k % 2 else rng.normal(0, 0.05, 2)        # lattice-aligned or generic offsets
        clouds.append((base + shift).astype(np.float32))
        offsets.append(offsets[-1] + n)
    pts, off = np.concatenate(clouds), np.array(offsets, np.int64)
    gpu_matcher.upload_scans(pts, off)
    n_pairs = 300
    src = rng.integers(0, 30, n_pairs).astype(np.int32)
    tgt = rng.integers(0, 30, n_pairs).astype(np.int32)
    guess = np.zeros((n_pairs, 3), np.float32)
    guess[:, :2] = rng.integers(-1, 2, (n_pairs, 2)) * 0.125                              # lattice-aligned guesses keep the ties exact
    for search in (SEARCH_BRUTE, SEARCH_PRUNED):
        for cov_mode in (COV_CENSI_CORR, COV_CENSI_INDEXPAIR):
            p = Params.defaults(downsample_divisor=1, search=search, cov_mode=cov_mode, max_iterations=60)
            got = gpu_matcher.submit_pairs(src, tgt, guess, p)
            ref, _ = O.run_batch(pts, off, src, tgt, guess, p, fast=0, threads=0)
            assert_records_match(got, ref, f"ties search {search} cov {cov_mode}")


# ---- outlier rejection ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,param,k_small", [(OUTLIER_TRIMMED, 0.7, None), (OUTLIER_TRIMMED, 1.0, None), (OUTLIER_MEDIAN, 1.5, None),
                                                (OUTLIER_MEDIAN, 0.8, None), (OUTLIER_MEDIAN, 0.5, 1), (OUTLIER_MEDIAN, 0.5, 2)],
                         ids=["1-0.7", "1-1.0", "2-1.5", "2-0.8", "2-0.5-K1", "2-0.5-K2"])
def test_outlier_rejection_correspondences_bit_exact(gpu_matcher, mode, param, k_small):
    if k_small:
        # 3 target points, k_small accepted pairs: MEDIAN 0.5 keeps fewer than all of them (1 of 2, 0 of 1)
        tgt = np.array([[0.0, 0.0], [0.0, 1.5], [0.0, 3.0]], np.float32)
        src = (tgt[:k_small] + np.array([0.1, 0.0], np.float32) * np.arange(1, k_small + 1, dtype=np.float32)[:, None]).astype(np.float32)
        Tm = np.array([1, 0, 0, 0], np.float32)
        for search in (SEARCH_BRUTE, SEARCH_PRUNED, SEARCH_PROJECTIVE):
            p = Params.defaults(downsample_divisor=1, search=search, outlier_mode=mode, outlier_param=param)
            kk, want, _ = O.correspondences(src, tgt, p, src_orig=src, T=Tm)
            got, _ = gpu_matcher.correspondences(src, tgt, Tm, p)
            assert kk == k_small - 1 and np.array_equal(got, want), (search, got, want)
        return
    wl = synth.config_corridor(n_pairs=6, seed=21)
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    for search in (SEARCH_BRUTE, SEARCH_PRUNED, SEARCH_PROJECTIVE):
        p = Params.defaults(downsample_divisor=1, search=search, outlier_mode=mode, outlier_param=param)
        for k in range(wl.n_pairs):
            s, t = wl.src_idx[k], wl.tgt_idx[k]
            S, T_ = pts[off[s]:off[s + 1]], pts[off[t]:off[t + 1]]
            Tm = O.guess_matrix(wl.guess[k])
            cur = O.transform_points(Tm, S)
            kk, want, want_d2 = O.correspondences(cur, T_, p, src_orig=S, T=Tm)
            got, got_d2 = gpu_matcher.correspondences(S, T_, Tm, p)
            assert np.array_equal(got, want), (search, k)
            k0, _, _ = O.correspondences(cur, T_, p.copy(outlier_mode=0), src_orig=S, T=Tm)
            assert 3 <= kk <= k0 and int((got >= 0).sum()) == kk
            if mode == OUTLIER_TRIMMED and param >= 1.0:
                assert kk == k0


@pytest.mark.parametrize("mode,param", [(OUTLIER_TRIMMED, 0.8), (OUTLIER_MEDIAN, 2.0)])
def test_outlier_rejection_batches(gpu_matcher, mode, param):
    """Whole batches with a rejector: every metric / search / covariance mode, both divisors; the stage chain (without
    its cluster stage, which the rejector's block-wide select does not span) must not change results."""
    wl = synth.config_corridor(n_pairs=48, seed=33)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    pts, off = gpu_matcher.download_store()
    for div, metric, search, cov in ((1, 0, SEARCH_PRUNED, COV_CENSI_CORR), (5, 0, SEARCH_BRUTE, COV_CENSI_CORR), (1, METRIC_POINT_TO_LINE, SEARCH_PRUNED, COV_CENSI_CORR),
                                     (1, 0, SEARCH_PROJECTIVE, COV_CENSI_CORR), (3, 0, SEARCH_PRUNED, COV_CENSI_INDEXPAIR)):
        p = Params.defaults(downsample_divisor=div, metric=metric, search=search, cov_mode=cov, outlier_mode=mode, outlier_param=param)
        got = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
        ref, _ = O.run_batch(pts, off, wl.src_idx, wl.tgt_idx, wl.guess, p, fast=1, threads=0)
        assert_records_match(got, ref, f"outlier {mode}/{param}: div {div} metric {metric} search {search} cov {cov}")
    wl2 = synth.config_loop_closure(n_pairs=300, n_scans=60, seed=34)
    gpu_matcher.upload_ranges(wl2.ranges, wl2.scanner)
    pts, off = gpu_matcher.download_store()
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR, outlier_mode=mode, outlier_param=param)
    got = gpu_matcher.submit_pairs(wl2.src_idx, wl2.tgt_idx, wl2.guess, p)
    ref, _ = O.run_batch(pts, off, wl2.src_idx, wl2.tgt_idx, wl2.guess, p, fast=1, threads=0)
    assert_records_match(got, ref, f"outlier {mode}/{param}: loop closure batch (staged chain)")


def test_outlier_param_validation(gpu_matcher):
    wl = synth.config_corridor(n_pairs=2, seed=1)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    for kw in (dict(outlier_mode=3), dict(outlier_mode=OUTLIER_TRIMMED, outlier_param=0.0), dict(outlier_mode=OUTLIER_TRIMMED, outlier_param=1.5),
               dict(outlier_mode=OUTLIER_MEDIAN, outlier_param=-1.0), dict(outlier_mode=OUTLIER_MEDIAN, outlier_param=float("inf"))):
        with pytest.raises(DpgIcpError) as e:
            gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, Params.defaults(**kw))
        assert e.value.code == -1


# ---- device-resident callers ------------------------------------------------------------------------------------------
def _random_walk_nodes(n, rng, size=60.0, passes=3):
    """trajectory-like node estimates (1 m steps, bounded area) in `passes` sessions"""
    pos = np.empty((n, 3), np.float32)
    cur = np.array([size / 2, size / 2, 0.0])
    per = (n + passes - 1) // passes
    for k in range(n):
        if k % per == 0:
            cur = np.array([rng.uniform(5, size - 5), rng.uniform(5, size - 5), rng.uniform(-np.pi, np.pi)])
        pos[k] = cur
        for _ in range(8):
            th = cur[2] + rng.uniform(-0.5, 0.5)
            nx, ny = cur[0] + np.cos(th), cur[1] + np.sin(th)
            if 0 < nx < size and 0 < ny < size:
                cur = np.array([nx, ny, th])
                break
            cur[2] += rng.uniform(1.0, 2.5)
    return pos, (np.arange(n) // per).astype(np.int32)


def _host_guess_T(poses, src, tgt):
    """the host path: dpgicp_relative_guess + the Matrix4f cos/sin of set_pairs (host libm)"""
    g = np.stack([relative_guess(poses[t], poses[s]) for s, t in zip(src, tgt)]) if len(src) else np.zeros((0, 3), np.float32)
    T = np.zeros((len(src), 4), np.float32)
    T[:, 0] = np.cos(g[:, 2].astype(np.float64)).astype(np.float32)
    T[:, 1] = np.sin(g[:, 2].astype(np.float64)).astype(np.float32)
    T[:, 2:] = g[:, :2]
    return g, T


@pytest.mark.parametrize("n", [0, 1, 2, 3, 33, 200, 1500, 21000])
def test_device_enumeration_reoptimize_matches_reference_loop(gpu_matcher, n):
    """dpgicp_enumerate_pairs_device == the reference's reoptimize loop order (oracle), and the device-derived guesses
    == the host path's, bit for bit — also for node indices in NO spatial order (worst case of the box hierarchy)."""
    rng = np.random.default_rng(1000 + n)
    for order in ("trajectory", "shuffled"):
        poses, passes = _random_walk_nodes(n, rng) if n else (np.zeros((0, 3), np.float32), np.zeros(0, np.int32))
        if order == "shuffled":
            if n > 3000:
                continue
            perm = rng.permutation(n)
            poses, passes = poses[perm], passes[perm]
        gpu_matcher.set_nodes(poses, passes)
        total, local = gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0)
        wsrc, wtgt = O.enumerate_pairs(poses[:, :2], passes, 5.0, 2.0)
        assert total == local == len(wsrc), (n, order)
        src, tgt, T = gpu_matcher.fetch_pairs()
        assert np.array_equal(src, wsrc) and np.array_equal(tgt, wtgt), (n, order)
        sel = np.arange(len(src)) if len(src) <= 4000 else rng.choice(len(src), 4000, replace=False)
        _, wT = _host_guess_T(poses, src[sel], tgt[sel])
        assert T[sel].tobytes() == wT.tobytes(), (n, order)
        # the v2 host-array form runs on the same kernels
        s2, t2 = gpu_matcher.enumerate_pairs(poses[:, :2], passes, 5.0, 2.0)
        assert np.array_equal(s2, wsrc) and np.array_equal(t2, wtgt)


def test_device_enumeration_shards_partition_the_list(gpu_matcher):
    rng = np.random.default_rng(4)
    poses, passes = _random_walk_nodes(3000, rng)
    gpu_matcher.set_nodes(poses, passes)
    wsrc, wtgt = O.enumerate_pairs(poses[:, :2], passes, 5.0, 2.0)
    for world in (2, 3, 8):
        seen = np.zeros(len(wsrc), bool)
        for rank in range(world):
            total, local = gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, rank, world)
            assert total == len(wsrc) and local == len(range(rank, total, world))
            src, tgt, _ = gpu_matcher.fetch_pairs()
            assert np.array_equal(src, wsrc[rank::world]) and np.array_equal(tgt, wtgt[rank::world])
            seen[rank::world] = True
        assert seen.all()
    with pytest.raises(DpgIcpError):
        gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, 3, 3)


@pytest.mark.parametrize("n", [2, 3, 4, 5, 40, 700, 5000])
def test_device_enumeration_online_matches_reference_loop(gpu_matcher, n):
    rng = np.random.default_rng(50 + n)
    poses, passes = _random_walk_nodes(n, rng, size=25.0, passes=2)
    gpu_matcher.set_nodes(poses, passes)
    total, local = gpu_matcher.enumerate_pairs_device(ENUM_ONLINE, 5.0, 2.0)
    wsrc, wtgt = O.enumerate_online(poses[:, :2], passes, 5.0, 2.0)
    src, tgt, T = gpu_matcher.fetch_pairs()
    assert total == len(wsrc) and np.array_equal(src, wsrc) and np.array_equal(tgt, wtgt)
    assert src[0] == n - 1 and tgt[0] == n - 2 and np.all(src[1:] == n - 2)               # closures attach to the preceding node
    _, wT = _host_guess_T(poses, src, tgt)
    assert T.tobytes() == wT.tobytes()


def test_device_enumerated_batch_equals_host_pair_list(gpu_matcher):
    """config 5 shape at oracle size through the device-resident caller: enumerate on the device, run, fetch — equal to
    the host-built pair list through set_pairs and to the oracle; factors carry the enumerated node ids."""
    wl = synth.config_multisession(n_sessions=3, scans_per_session=60, n_beams=541, seed=5, size=30.0, n_boxes=30)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    pts, off = gpu_matcher.download_store()
    gpu_matcher.set_nodes(wl.poses_est, wl.passes)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    for mode in (ENUM_REOPTIMIZE, ENUM_ONLINE):
        total, local = gpu_matcher.enumerate_pairs_device(mode, 5.0, 2.0)
        src, tgt, _ = gpu_matcher.fetch_pairs()
        gpu_matcher.run(p)
        got = gpu_matcher.fetch_results()
        fac = gpu_matcher.fetch_factors()
        guess, _ = _host_guess_T(wl.poses_est, src, tgt)
        ref, _ = O.run_batch(pts, off, src, tgt, guess, p, fast=1, threads=0)
        assert_records_match(got, ref, f"device-enumerated batch mode {mode}")
        assert np.array_equal(fac["from_node"], tgt) and np.array_equal(fac["to_node"], src)
        host = gpu_matcher.submit_pairs(src, tgt, guess, p)
        assert host.tobytes() == got.tobytes()
    # nodes without scans are refused at run time
    gpu_matcher.set_nodes(np.concatenate([wl.poses_est, wl.poses_est[:5]]), np.concatenate([wl.passes, wl.passes[:5]]))
    gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0)
    with pytest.raises(DpgIcpError) as e:
        gpu_matcher.run(p)
    assert e.value.code == -6


def test_enumeration_of_400k_nodes_is_fast(gpu_matcher):
    """BASELINE config 5 size: 8 sessions x 50 000 nodes on a 100 m x 100 m world.  Counts + scan + fill with the guesses
    for this context's shard of an 8-way split; the strided sample of the list equals the reference loop."""
    rng = np.random.default_rng(8)
    poses, passes = _random_walk_nodes(400_000, rng, size=100.0, passes=8)
    gpu_matcher.set_nodes(poses, passes)
    gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, 0, 8)                   # warm-up (allocations)
    gpu_matcher.synchronize()
    t0 = time.perf_counter()
    total, local = gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, 0, 8)
    gpu_matcher.synchronize()
    dt = time.perf_counter() - t0
    print(f"\n[enumeration] 400k nodes: {total} pairs, shard 0/8 = {local}, {dt * 1e3:.1f} ms")
    assert total > 10_000_000 and dt < 0.25
    # the pairs of node i involve only nodes j < i, so the list of the first m nodes is a prefix of the whole list:
    # this shard's first pairs are every 8th pair of the reference loop over those nodes
    m = 20_000
    wsrc, wtgt = O.enumerate_pairs(poses[:m, :2], passes[:m], 5.0, 2.0)
    k = len(range(0, len(wsrc), 8))
    src, tgt, T = gpu_matcher.fetch_pairs(k)
    assert np.array_equal(src, wsrc[0::8]) and np.array_equal(tgt, wtgt[0::8])
    sel = rng.choice(k, 2000, replace=False)
    _, wT = _host_guess_T(poses, src[sel], tgt[sel])
    assert T[sel].tobytes() == wT.tobytes()


def test_convert_ranges_already_on_the_device(gpu_matcher):
    import torch
    wl = synth.config_corridor(n_pairs=20, seed=6)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    want_pts, want_off = gpu_matcher.download_store()
    d = torch.from_numpy(wl.ranges).cuda()
    torch.cuda.synchronize()
    gpu_matcher.convert_ranges_device(d.data_ptr(), wl.n_scans, wl.ranges.shape[1], wl.scanner)
    got_pts, got_off = gpu_matcher.download_store()
    assert np.array_equal(got_off, want_off) and got_pts.tobytes() == want_pts.tobytes()


def test_stage_timing(gpu_matcher):
    wl = synth.config_corridor(n_pairs=600, seed=2)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    gpu_matcher.set_pairs(wl.src_idx, wl.tgt_idx, wl.guess)
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    with pytest.raises(DpgIcpError):
        gpu_matcher.last_run_stage_ms()
    gpu_matcher.enable_stage_timing(True)
    gpu_matcher.run(p)
    ms = gpu_matcher.last_run_stage_ms()
    gpu_matcher.enable_stage_timing(False)
    assert 1 <= len(ms) <= 5 and all(m >= 0 for m in ms) and sum(ms) > 0.05


# ---- one process, several contexts: the C/C++ multi-GPU host path ----------------------------------------------------------
def test_two_contexts_one_process_gather_equals_single_context(gpu_matcher):
    """dpgicp_gather_attach_local: two contexts of ONE process (here both on cuda:0, on a multi-GPU box one per device)
    shard the device-enumerated list round-robin and store their records into context 0's buffer from the kernel
    epilogue; the gathered batch equals the single-context run bit for bit."""
    wl = synth.config_multisession(n_sessions=2, scans_per_session=80, n_beams=541, seed=9, size=30.0, n_boxes=30)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
    gpu_matcher.set_nodes(wl.poses_est, wl.passes)
    total, _ = gpu_matcher.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0)
    gpu_matcher.run(p)
    want = gpu_matcher.fetch_results()
    lib = _abi.load_library()
    n_dev = 1
    try:
        import torch
        n_dev = torch.cuda.device_count()
    except Exception:
        pass
    for root_only in (1, 0):
        ms = [ScanMatcher(0), ScanMatcher(1 if n_dev > 1 else 0), ScanMatcher(0)]
        try:
            world = len(ms)
            for r, m in enumerate(ms):
                m.upload_ranges(wl.ranges, wl.scanner)
                m.set_nodes(wl.poses_est, wl.passes)
                t, l = m.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0, r, world)
                assert t == total
            arr = (C.c_void_p * world)(*[m._h for m in ms])
            assert lib.dpgicp_gather_attach_local(arr, world, total, root_only) == 0
            for m in ms:
                m.run(p)
            for m in ms:
                m.synchronize()
            got = ms[0].gather_fetch(total)
            assert got.tobytes() == want.tobytes(), f"root_only={root_only}"
            if not root_only:
                assert ms[2].gather_fetch(total).tobytes() == want.tobytes()
            for m in ms:
                m.gather_detach()
        finally:
            for m in ms:
                m.close()


def test_cpp_runner_multi_context_writes_the_same_csv(tmp_path):
    """dpg_batch_runner --devices a,b (one C++ process, dpgicp_shim::MultiGpuScanMatcher) == --devices a: same CSV."""
    exe = os.path.join(ROOT, "dpg_slam_b200", "dpg_batch_runner")
    n_dev = 1
    try:
        import torch
        n_dev = torch.cuda.device_count()
    except Exception:
        pass
    outs = []
    for devs in ("0", "0,1" if n_dev > 1 else "0,0", "0,0,0"):
        out = tmp_path / f"r_{devs.replace(',', '_')}.csv"
        r = subprocess.run([exe, "--synthetic", "office", "--scans", "140", "--beams", "541", "--passes", "2", "--cov-mode", "2",
                            "--devices", devs, "--out", str(out)], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        outs.append(out.read_text())
    assert outs[0] == outs[1] == outs[2] and outs[0].count("\n") > 200
    for caller in ("online",):
        a = tmp_path / "on1.csv"
        b = tmp_path / "on2.csv"
        for devs, out in (("0", a), ("0,0", b)):
            r = subprocess.run([exe, "--synthetic", "office", "--scans", "140", "--beams", "541", "--caller", caller, "--devices", devs,
                                "--out", str(out)], capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stderr
        assert a.read_text() == b.read_text()


# ---- the CUDA search against a real FLANN kd-tree, first hand ------------------------------------------------------------
@pytest.mark.parametrize("divisor", [1, 5])
def test_cuda_correspondences_equal_a_real_flann_kdtree(gpu_matcher, divisor):
    """dpgicp_correspondences (the exact pruned search) against OpenCV's bundled FLANN KDTreeSingleIndex — the index and the
    exact search pcl::KdTreeFLANN runs — at several iterates of corridor and loop-closure pairs: the same forward neighbours,
    the same binary32 squared distances, and the reciprocal sets PCL's determineReciprocalCorrespondences forms from two
    such trees (north star: "correspondence index sets bit-exact given the same iterate")."""
    pytest.importorskip("cv2")
    import pcl_emulation as E

    def xyz(a):
        out = np.zeros((len(a), 3), np.float32)
        out[:, :2] = a
        return out

    n_q = 0
    for wl in (synth.config_corridor(n_pairs=12, seed=31), synth.config_loop_closure(n_pairs=12, n_scans=30, seed=32)):
        pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
        for k in range(0, wl.n_pairs, 3):
            s, t = int(wl.src_idx[k]), int(wl.tgt_idx[k])
            S, T = pts[off[s]:off[s + 1]][::divisor], pts[off[t]:off[t + 1]][::divisor]
            _, iterates, _ = O.icp(S, T, wl.guess[k], Params.defaults(downsample_divisor=1), trace=True)
            tree_t = E.FlannTree(xyz(T))
            for it in sorted(set([0, len(iterates) // 2, len(iterates) - 1])):
                Tm = iterates[it]
                cur = O.transform_points(Tm, S)
                d2f, jf = tree_t.query(xyz(cur))
                inside = d2f.astype(np.float64) <= 0.36
                got, got_d2 = gpu_matcher.correspondences(S, T, Tm, Params.defaults(use_reciprocal=0))
                assert np.array_equal(got >= 0, inside), (k, it)
                assert np.array_equal(got[inside], jf[inside]), (k, it)
                assert np.array_equal(got_d2[inside].view(np.uint32), d2f[inside].view(np.uint32)), (k, it)
                _, back = E.FlannTree(xyz(cur)).query(xyz(T)[jf])
                want_r = np.where(inside & (back == np.arange(len(cur))), jf, -1)
                got_r, _ = gpu_matcher.correspondences(S, T, Tm, Params.defaults(use_reciprocal=1))
                assert np.array_equal(got_r, want_r), (k, it)
                n_q += int(inside.sum())
    assert n_q > 3000


def test_small_batches_start_at_the_stage_that_keeps_them(gpu_matcher):
    """A single runIcp-shaped call and the online caller's handful of pairs run as ONE launch of the widest fitting shape (no
    stage that would suspend every pair after its first pass), with the records of the staged chain: the same pairs inside a
    batch large enough to start at the narrow stage give identical bits."""
    wl = synth.config_corridor(n_pairs=1200, seed=41)
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    for p in (Params.defaults(), Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)):
        gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
        big = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
        n_big = gpu_matcher.last_run_counters()["kernel_launches"]
        for k in (0, 7, 300):
            s, t = int(wl.src_idx[k]), int(wl.tgt_idx[k])
            before = gpu_matcher.last_run_counters()["kernel_launches"]
            _, _, _, r = gpu_matcher.run_icp(pts[off[t]:off[t + 1]], pts[off[s]:off[s + 1]], wl.guess[k], p)
            assert gpu_matcher.last_run_counters()["kernel_launches"] - before == 1
            assert (r.tx, r.ty, r.iterations, r.status, r.mse) == (big["tx"][k], big["ty"][k], big["iterations"][k], big["status"][k], big["mse"][k])
        gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
        before = gpu_matcher.last_run_counters()["kernel_launches"]
        few = gpu_matcher.submit_pairs(wl.src_idx[:20], wl.tgt_idx[:20], wl.guess[:20], p)
        assert gpu_matcher.last_run_counters()["kernel_launches"] - before == 1
        assert few.tobytes() == big[:20].tobytes()
        assert n_big >= 1


def test_cuda_correspondences_equal_flann_golden_vectors(gpu_matcher):
    """The committed FLANN golden vectors (tests/golden/flann_nn.json, generated by tools/make_flann_golden.py from OpenCV's
    bundled FLANN) against dpgicp_correspondences: forward neighbours, binary32 squared distances and reciprocal sets."""
    import json
    cases = json.load(open(os.path.join(ROOT, "tests", "golden", "flann_nn.json")))["cases"]

    def hexf(h, cols=None):
        a = np.array([int(x, 16) for x in h], np.uint32).view(np.float32)
        return a.reshape(-1, cols) if cols else a

    for c in cases:
        S, T, Tm = hexf(c["source_hex"], 2), hexf(c["target_hex"], 2), hexf(c["T_hex"])
        jf = np.array(c["flann_forward_index"]); d2f = hexf(c["flann_forward_d2_hex"]); back = np.array(c["flann_backward_index"])
        inside = d2f.astype(np.float64) <= 0.36
        got, got_d2 = gpu_matcher.correspondences(S, T, Tm, Params.defaults(use_reciprocal=0))
        assert np.array_equal(got >= 0, inside) and np.array_equal(got[inside], jf[inside]), (c["workload"], c["pair"], c["iterate"])
        assert np.array_equal(got_d2[inside].view(np.uint32), d2f[inside].view(np.uint32))
        got_r, _ = gpu_matcher.correspondences(S, T, Tm, Params.defaults(use_reciprocal=1))
        assert np.array_equal(got_r, np.where(inside & (back == np.arange(len(S))), jf, -1))
