"""Synthetic Hokuyo-like workloads for the batch runner, tests and bench (SURVEY.md §8d).

Host-side input generation only: worlds are wall-segment lists, scans are ray-cast by
``libdpgsynth.so`` (csrc/dpgsynth.c).  Each builder returns a :class:`Workload` holding raw ranges
(what ``DpgSLAM::ObserveLaser`` receives, reference src/dpg_slam/dpg_slam.cc:122-140), node pose
estimates, the scan-pair list in the reference's loop order and the per-pair guess
(dpg_slam.cc:364-378).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _synth():
    global _lib
    if _lib is None:
        path = os.path.join(_HERE, "libdpgsynth.so")
        if not os.path.exists(path):
            raise RuntimeError(f"{path} missing: run __graft_entry__.build()")
        lib = C.CDLL(path)
        lib.dpgsynth_uniform.restype = C.c_double
        lib.dpgsynth_uniform.argtypes = [C.c_uint64] * 3
        lib.dpgsynth_world_room.restype = C.c_int
        lib.dpgsynth_world_room.argtypes = [C.c_double, C.c_double, C.c_void_p, C.c_int]
        lib.dpgsynth_world_corridor.restype = C.c_int
        lib.dpgsynth_world_corridor.argtypes = [C.c_double] * 4 + [C.c_uint64, C.c_void_p, C.c_int]
        lib.dpgsynth_world_office.restype = C.c_int
        lib.dpgsynth_world_office.argtypes = [C.c_double, C.c_int, C.c_uint64, C.c_int, C.c_double,
                                              C.c_void_p, C.c_int]
        lib.dpgsynth_is_free.restype = C.c_int
        lib.dpgsynth_is_free.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double]
        lib.dpgsynth_inside_box.restype = C.c_int
        lib.dpgsynth_inside_box.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double]
        lib.dpgsynth_cast_scans.restype = None
        lib.dpgsynth_cast_scans.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                            C.c_float, C.c_float, C.c_float, C.c_float, C.c_double,
                                            C.c_uint64, C.c_double, C.c_double, C.c_int, C.c_void_p]
        _lib = lib
    return _lib


@dataclass
class Scanner:
    """UTM-30LX-class scanner: 270 deg FOV, 1081 beams, 0.02-30 m (SURVEY.md §8d)."""
    n_beams: int = 1081
    angle_min: float = -0.75 * math.pi
    angle_max: float = 0.75 * math.pi
    range_min: float = 0.02
    range_max: float = 30.0
    noise_sigma: float = 0.01
    # laser pose in base_link, parameters.h:319-339
    laser_x: float = 0.2
    laser_y: float = 0.0
    laser_theta: float = 0.0


@dataclass
class Workload:
    name: str
    scanner: Scanner
    ranges: np.ndarray          # (n_scans, n_beams) float32
    poses_true: np.ndarray      # (n_scans, 3) float64 base_link poses in the world
    poses_est: np.ndarray       # (n_scans, 3) float32 node estimates (truth + drift/noise)
    src_idx: np.ndarray         # (n_pairs,) int32   node_2 (source)
    tgt_idx: np.ndarray         # (n_pairs,) int32   node_1 (target)
    guess: np.ndarray           # (n_pairs, 3) float32 (dx, dy, dtheta) of node_2 in node_1's frame
    truth: np.ndarray           # (n_pairs, 3) float64 true relative pose
    passes: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int32))
    seed: int = 0

    @property
    def n_pairs(self) -> int:
        return int(self.src_idx.shape[0])

    @property
    def n_scans(self) -> int:
        return int(self.ranges.shape[0])


# ---- worlds ---------------------------------------------------------------------------------------
def _segs(fn, *args, cap=1 << 16) -> np.ndarray:
    buf = np.zeros((cap, 4), np.float32)
    n = fn(*args, buf.ctypes.data, cap)
    if n > cap:
        buf = np.zeros((n, 4), np.float32)
        n = fn(*args, buf.ctypes.data, n)
    return np.ascontiguousarray(buf[:n])


def world_room(w=10.0, h=6.0) -> np.ndarray:
    return _segs(_synth().dpgsynth_world_room, w, h)


def world_corridor(x_from, x_to, width=2.5, period=4.0, seed=2) -> np.ndarray:
    return _segs(_synth().dpgsynth_world_corridor, float(x_from), float(x_to), width, period, seed)


def world_office(size=40.0, n_boxes=60, seed=3, variant=0, moved_fraction=0.05) -> np.ndarray:
    return _segs(_synth().dpgsynth_world_office, size, n_boxes, seed, variant, moved_fraction)


def _cast_threads() -> int:
    """Host threads for the ray caster: all cores this process may use, shared between the ranks of a torch.distributed
    launch (which sets OMP_NUM_THREADS=1 — input generation is not the measured path and should not take minutes)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", os.environ.get("WORLD_SIZE", "1"))))
    return max(1, n // world)


def cast_scans(segs: np.ndarray, poses: np.ndarray, scanner: Scanner, seed: int) -> np.ndarray:
    segs = np.ascontiguousarray(segs, np.float32)
    poses = np.ascontiguousarray(poses, np.float64)
    out = np.empty((poses.shape[0], scanner.n_beams), np.float32)
    _synth().dpgsynth_cast_scans(segs.ctypes.data, segs.shape[0], poses.ctypes.data, poses.shape[0],
                                 scanner.n_beams, scanner.angle_min, scanner.angle_max,
                                 scanner.range_min, scanner.range_max, scanner.noise_sigma, seed,
                                 scanner.laser_x, scanner.laser_y, _cast_threads(), out.ctypes.data)
    return out


# ---- pose helpers (float32 restatement of math_utils for building *inputs*) --------------------------
def relative_pose(p1: np.ndarray, p2: np.ndarray) -> np.ndarray:
    """pose of p2 in the frame of p1 (float64, used for ground truth)."""
    p1 = np.asarray(p1, np.float64)
    p2 = np.asarray(p2, np.float64)
    d = p2[..., :2] - p1[..., :2]
    c, s = np.cos(-p1[..., 2]), np.sin(-p1[..., 2])
    out = np.empty(np.broadcast(p1, p2).shape, np.float64)
    out[..., 0] = c * d[..., 0] - s * d[..., 1]
    out[..., 1] = s * d[..., 0] + c * d[..., 1]
    a = p2[..., 2] - p1[..., 2]
    out[..., 2] = a - 2 * np.pi * np.rint(a / (2 * np.pi))
    return out


def _finish(name, scanner, segs, poses_true, poses_est, src, tgt, seed, passes=None) -> Workload:
    ranges = cast_scans(segs, poses_true, scanner, seed)
    src = np.ascontiguousarray(src, np.int32)
    tgt = np.ascontiguousarray(tgt, np.int32)
    est = np.ascontiguousarray(poses_est, np.float32)
    guess = relative_pose(est[tgt].astype(np.float64), est[src].astype(np.float64)).astype(np.float32)
    truth = relative_pose(poses_true[tgt], poses_true[src])
    if passes is None:
        passes = np.zeros(poses_true.shape[0], np.int32)
    return Workload(name, scanner, ranges, np.asarray(poses_true, np.float64), est, src, tgt,
                    np.ascontiguousarray(guess), truth, np.ascontiguousarray(passes, np.int32), seed)


# ---- BASELINE.json configs --------------------------------------------------------------------------
def config_room_pair(n_beams=1081, seed=1) -> Workload:
    """Config 1: one pair in a 10 m x 6 m room, poses (0,0,0) and (0.30,-0.20,0.10);
    guess = truth + (0.05, 0.05, 0.02)."""
    sc = Scanner(n_beams=n_beams)
    poses = np.array([[0.0, 0.0, 0.0], [0.30, -0.20, 0.10]])
    wl = _finish("room_pair", sc, world_room(), poses, poses, [1], [0], seed)
    wl.guess = (wl.truth + np.array([0.05, 0.05, 0.02])).astype(np.float32)
    return wl


def config_corridor(n_pairs=5000, n_beams=1081, seed=2, step=1.0) -> Workload:
    """Config 2: 2.5 m corridor with hashed door recesses every 4 m, n_pairs+1 poses spaced `step`
    with heading jitter U(-0.05,0.05) and lateral jitter; successive pairs; guess = truth + odometry
    noise N(0, 0.05 m; 0.02 rad).  The corridor is as long as the trajectory needs."""
    rng = np.random.default_rng(seed)
    n = n_pairs + 1
    sc = Scanner(n_beams=n_beams)
    x = 5.0 + step * np.arange(n)
    poses = np.stack([x, rng.uniform(-0.3, 0.3, n), rng.uniform(-0.05, 0.05, n)], axis=1)
    segs = world_corridor(0.0, x[-1] + 5.0, seed=seed)
    src = np.arange(1, n)
    tgt = np.arange(0, n - 1)
    wl = _finish("corridor", sc, segs, poses, poses, src, tgt, seed)
    noise = np.stack([rng.normal(0, 0.05, n_pairs), rng.normal(0, 0.05, n_pairs),
                      rng.normal(0, 0.02, n_pairs)], axis=1)
    wl.guess = (wl.truth + noise).astype(np.float32)
    # node estimates consistent with the guesses are not needed by the path; keep truth as estimate
    return wl


def config_corridor_passes(n_scans=1000, n_beams=1081, passes=2, seed=2) -> Workload:
    """The config-2 corridor driven forth and back in `passes` passes, poses 1 m apart (odd passes face back), as an
    online caller meets it node by node: node estimates = truth + noise N(0, 0.05 m; 0.02 rad), pass number per node.
    The pair list is the successive pairs; an online replay enumerates its own."""
    rng = np.random.default_rng(seed)
    per = -(-n_scans // passes)
    poses = np.zeros((n_scans, 3))
    for s in range(n_scans):
        k, back = s % per, (s // per) % 2 == 1
        poses[s] = (5.0 + (per - 1 - k if back else k), rng.uniform(-0.3, 0.3),
                    (math.pi if back else 0.0) + rng.uniform(-0.05, 0.05))
    est = poses + rng.normal(0, [0.05, 0.05, 0.02], (n_scans, 3))
    src = np.arange(1, n_scans)
    return _finish("corridor_passes", Scanner(n_beams=n_beams), world_corridor(0.0, per + 10.0, seed=seed), poses, est,
                   src, src - 1, seed, (np.arange(n_scans) // per).astype(np.int32))


def _free_poses(segs, size, n, rng, margin=0.4):
    lib = _synth()
    out = np.empty((n, 3))
    k = 0
    p = segs.ctypes.data
    while k < n:
        cand = rng.uniform(margin, size - margin, (max(64, n - k), 2))
        for cx, cy in cand:
            if lib.dpgsynth_is_free(p, segs.shape[0], cx, cy, margin) and \
                    not lib.dpgsynth_inside_box(p, segs.shape[0], cx, cy):
                out[k] = (cx, cy, rng.uniform(-np.pi, np.pi))
                k += 1
                if k == n:
                    break
    return out


def config_loop_closure(n_pairs=100_000, n_scans=2000, n_beams=1081, seed=3, size=40.0,
                        n_boxes=60) -> Workload:
    """Config 3: pairs drawn from n_scans scans of an office-like world; true offset <= 2 m;
    initial offsets U(+-0.3 m, +-0.3 m, +-0.15 rad) around truth."""
    rng = np.random.default_rng(seed)
    sc = Scanner(n_beams=n_beams)
    segs = world_office(size, n_boxes, seed)
    # scans come in clusters so that many pairs within 2 m exist
    n_centres = max(1, n_scans // 8)
    centres = _free_poses(segs, size, n_centres, rng)
    poses = np.empty((n_scans, 3))
    lib = _synth()
    for i in range(n_scans):
        c = centres[i % n_centres]
        for _ in range(100):
            cand = c[:2] + rng.uniform(-0.7, 0.7, 2)
            if lib.dpgsynth_is_free(segs.ctypes.data, segs.shape[0], cand[0], cand[1], 0.3) and \
                    not lib.dpgsynth_inside_box(segs.ctypes.data, segs.shape[0], cand[0], cand[1]):
                break
        else:
            cand = c[:2]
        poses[i] = (cand[0], cand[1], c[2] + rng.uniform(-0.4, 0.4))
    a = rng.integers(0, n_scans, n_pairs)
    off = rng.integers(1, 8, n_pairs) * n_centres      # same cluster, different member
    b = (a + off) % n_scans
    same = b == a
    b[same] = (a[same] + n_centres) % n_scans
    wl = _finish("loop_closure", sc, segs, poses, poses, a, b, seed)
    noise = np.stack([rng.uniform(-0.3, 0.3, n_pairs), rng.uniform(-0.3, 0.3, n_pairs),
                      rng.uniform(-0.15, 0.15, n_pairs)], axis=1)
    wl.guess = (wl.truth + noise).astype(np.float32)
    return wl


def config_dense(n_pairs=1_000_000, n_scans=20_000, n_beams=4096, seed=4) -> Workload:
    """Config 4: 4096 beams/scan, offsets as config 3 (point-to-line is selected by the caller)."""
    wl = config_loop_closure(n_pairs, n_scans, n_beams, seed)
    wl.name = "dense"
    return wl


def config_multisession(n_sessions=8, scans_per_session=50_000, n_beams=1081, seed=5, size=100.0,
                        n_boxes=300, same_radius=5.0, other_radius=2.0, max_pairs=None) -> Workload:
    """Config 5: sessions on a shared world with 5 % of the boxes moved per session; trajectories
    are random walks; candidate pairs are produced by the callers' distance gate
    (parameters.h:212,224; dpg_slam.cc:94-98) on the drifted estimates — enumerate them with
    ``ScanMatcher.enumerate_pairs`` and pass them in via ``with_pairs``."""
    rng = np.random.default_rng(seed)
    sc = Scanner(n_beams=n_beams)
    all_poses, all_ranges, passes = [], [], []
    for s in range(n_sessions):
        segs = world_office(size, n_boxes, seed, s, 0.05)
        start = _free_poses(segs, size, 1, rng)[0]
        poses = np.empty((scans_per_session, 3))
        cur = start.copy()
        lib = _synth()
        for i in range(scans_per_session):
            poses[i] = cur
            for _ in range(50):
                th = cur[2] + rng.uniform(-0.5, 0.5)
                nxt = cur[:2] + 1.0 * np.array([math.cos(th), math.sin(th)])
                if 0.5 < nxt[0] < size - 0.5 and 0.5 < nxt[1] < size - 0.5 and \
                        lib.dpgsynth_is_free(segs.ctypes.data, segs.shape[0], nxt[0], nxt[1], 0.35) and \
                        not lib.dpgsynth_inside_box(segs.ctypes.data, segs.shape[0], nxt[0], nxt[1]):
                    cur = np.array([nxt[0], nxt[1], th])
                    break
                cur[2] += rng.uniform(1.0, 2.5)
        all_poses.append(poses)
        all_ranges.append(cast_scans(segs, poses, sc, seed * 1000 + s))
        passes.append(np.full(scans_per_session, s, np.int32))
    poses = np.concatenate(all_poses)
    ranges = np.concatenate(all_ranges)
    passes = np.concatenate(passes)
    drift = np.stack([rng.normal(0, 0.08, len(poses)), rng.normal(0, 0.08, len(poses)),
                      rng.normal(0, 0.03, len(poses))], axis=1)
    est = (poses + drift).astype(np.float32)
    wl = Workload("multisession", sc, ranges, poses, est, np.zeros(0, np.int32), np.zeros(0, np.int32),
                  np.zeros((0, 3), np.float32), np.zeros((0, 3)), passes, seed)
    return wl


def with_pairs(wl: Workload, src: np.ndarray, tgt: np.ndarray) -> Workload:
    """Attach a pair list (e.g. from the distance-gated enumeration) and derive guesses from the
    node estimates exactly as dpg_slam.cc:364-370 does."""
    src = np.ascontiguousarray(src, np.int32)
    tgt = np.ascontiguousarray(tgt, np.int32)
    wl.src_idx, wl.tgt_idx = src, tgt
    wl.guess = relative_pose(wl.poses_est[tgt].astype(np.float64),
                             wl.poses_est[src].astype(np.float64)).astype(np.float32)
    wl.truth = relative_pose(wl.poses_true[tgt], wl.poses_true[src])
    return wl
