"""GPU (B200): the node table changed in place (dpgicp_update_nodes) and its wrappers.  Whatever sequence of updates led
to a table, its enumerated pair lists and guesses (REOPTIMIZE and ONLINE) are bit for bit those of one set_nodes of the
same full arrays: through growth one node at a time across the leaf and level boundaries, scattered moves, boxes that
shrink, pass changes, the edge layouts of enum_cases; records and factors of an online replay with an optimiser that
moves estimates; refusals that leave the table; a slot enumerated before an update; set_nodes in between; sync_nodes
and the runner's --replay --nodes sync."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import enum_cases as EC
import ref_enumeration as R
from dpg_slam_b200 import synth
from dpg_slam_b200._abi import COV_CENSI_CORR, ENUM_ONLINE, ENUM_REOPTIMIZE, Params
from dpg_slam_b200.scanmatch import DpgIcpError, ScanMatcher

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RUNNER = os.path.join(ROOT, "dpg_slam_b200", "dpg_batch_runner")
E_INVALID, E_RANGE = -1, -5
F32 = np.float32


def _lists(sm, r_same=5.0, r_other=2.0):
    """(src, tgt, T) of both enumeration modes over the context's table, as bytes"""
    out = []
    for mode in (ENUM_REOPTIMIZE, ENUM_ONLINE):
        sm.enumerate_pairs_device(mode, r_same, r_other)
        out.append(tuple(a.tobytes() for a in sm.fetch_pairs()))
    return out


def _assert_same_as_set_nodes(sm, ref, poses, passes, what, r_same=5.0, r_other=2.0):
    ref.set_nodes(poses, passes)
    got, want = _lists(sm, r_same, r_other), _lists(ref, r_same, r_other)
    for mode, g, w in zip(("REOPTIMIZE", "ONLINE"), got, want):
        assert g == w, f"{what}: {mode} list or guesses differ from set_nodes"


# ---- 1. growth one node at a time across leaf (32) and level (1 024, 32 768) boundaries --------------------------------
def test_growth_one_node_at_a_time():
    n_max = 33_000
    poses, passes = EC.walk(n_max, seed=51, sessions=4)
    with ScanMatcher(0) as sm, ScanMatcher(0) as ref:
        for n in range(1, n_max + 1):
            sm.update_nodes([n - 1], poses[n - 1:n], passes[n - 1:n])
            if n < 1100 or n % 1999 == 0 or n in (32_767, 32_768, 32_769, n_max):
                _assert_same_as_set_nodes(sm, ref, poses[:n], passes[:n], f"n={n}")


# ---- 2. scattered updates on a multi-pass corridor -----------------------------------------------------------------
def test_scattered_updates_on_a_multi_pass_corridor():
    wl = synth.config_corridor_passes(3000, 32, 3, seed=52)
    poses, passes = wl.poses_est.astype(F32).copy(), wl.passes.copy()
    n = len(poses)
    rng = np.random.default_rng(52)
    with ScanMatcher(0) as sm, ScanMatcher(0) as ref:
        sm.update_nodes(np.arange(n), poses, passes)
        _assert_same_as_set_nodes(sm, ref, poses, passes, "initial")
        for step in range(12):                                            # random subsets, 1 .. 700 nodes
            ids = rng.choice(n, int(rng.integers(1, 700)), replace=False)
            poses[ids] += rng.normal(0, [0.3, 0.3, 0.05], (len(ids), 3)).astype(F32)
            sm.update_nodes(ids, poses[ids], passes[ids])
            _assert_same_as_set_nodes(sm, ref, poses, passes, f"subset {step}")
        # far away, then back: the box grows, then shrinks.  What this can see is a box left too SMALL (pairs of the moved
        # node lost); a box left too large only prunes less, and the gate still decides every pair, so lists and guesses
        # would not show it.  That the refit box equals the rebuilt one rests on node_boxes_refit_kernel and
        # node_boxes_leaf_kernel sharing node_leaf_box, not on this test.
        for i in (0, 31, 32, 1500, n - 1):
            keep = poses[i].copy()
            poses[i] = (1e4, -1e4, 3.0)
            sm.update_nodes([i], poses[i:i + 1], passes[i:i + 1])
            _assert_same_as_set_nodes(sm, ref, poses, passes, f"node {i} away")
            poses[i] = keep
            sm.update_nodes([i], poses[i:i + 1], passes[i:i + 1])
            _assert_same_as_set_nodes(sm, ref, poses, passes, f"node {i} back")
        for ids, new_pass in ((np.arange(64, 96), 7), (np.array([5, 700, 2999]), -3), (np.arange(2000, 2100), 0)):
            passes[ids] = new_pass                                        # pass ranges of leaves and parents change
            sm.update_nodes(ids, poses[ids], passes[ids])
            _assert_same_as_set_nodes(sm, ref, poses, passes, f"pass {new_pass}")
        poses += rng.normal(0, [0.1, 0.1, 0.01], poses.shape).astype(F32)  # every node
        perm = rng.permutation(n)
        sm.update_nodes(perm, poses[perm], passes[perm])
        _assert_same_as_set_nodes(sm, ref, poses, passes, "every node")


# ---- 3. edge layouts reached through a sequence of updates, against the independent reference -----------------------
def _reach(sm, poses, passes, rng):
    """grow the table in chunks with wrong estimates and passes, then correct it in three random subsets"""
    n = len(poses)
    junk = (poses.astype(np.float64) + rng.uniform(-40, 40, poses.shape)).astype(F32)
    jpass = rng.integers(-2, 6, n).astype(np.int32)
    k = 0
    while k < n:
        e = min(n, k + int(rng.integers(1, 50)))
        ids = np.arange(k, e)[::-1].copy()
        sm.update_nodes(ids, junk[ids], jpass[ids], n_nodes=e)
        k = e
    for ids in np.array_split(rng.permutation(n), 3):
        sm.update_nodes(ids, poses[ids], passes[ids])


def _edge_cases():
    return (EC.tie_345_cases() + EC.tie_cases() + EC.pass_radius_cases() + EC.geometry_cases() + [EC.angle_case()] +
            [EC.size_case(n) for n in (31, 32, 33, 1023, 1024, 1025)])


def test_edge_layouts_reached_by_updates_equal_the_reference():
    rng = np.random.default_rng(53)
    for c in _edge_cases():
        if len(c["poses"]) < 2:
            continue
        with ScanMatcher(0) as sm:
            _reach(sm, c["poses"], c["passes"], rng)
            for online in (False, True):
                xy = c["poses"][:, :2]
                ws, wt = (R.enumerate_online(xy, c["passes"], c["r_same"], c["r_other"]) if online else
                          R.enumerate_reoptimize(xy, c["passes"], c["r_same"], c["r_other"]))
                total, _ = sm.enumerate_pairs_device(ENUM_ONLINE if online else ENUM_REOPTIMIZE, c["r_same"], c["r_other"])
                assert total == len(ws), c["name"]
                src, tgt, T = sm.fetch_pairs()
                assert np.array_equal(src, ws) and np.array_equal(tgt, wt), c["name"]
                _, wT = R.guesses(c["poses"], ws, wt)
                assert T.tobytes() == wT.tobytes(), c["name"]


# ---- 4. records and factors of an online replay with an optimiser that moves estimates --------------------------------
def _replay(sm, ranges, sc, est_of, passes, p, nodes):
    """append -> node table -> enumerate -> run -> records + factors, reoptimize at each pass boundary.  est_of(k) is the
    estimate vector after update k.  nodes: "full" (set_nodes), "update" (update_nodes of the changed rows) or "sync"."""
    out, sent = [], None

    def table(est, n):
        nonlocal sent
        if nodes == "full":
            sm.set_nodes(est[:n], passes[:n])
        elif nodes == "sync":
            sm.sync_nodes(est[:n], passes[:n])
        else:
            m = 0 if sent is None else len(sent)
            ids = np.arange(n) if sent is None else np.concatenate(
                [np.flatnonzero((est[:m].view(np.uint32) != sent.view(np.uint32)).any(1)), np.arange(m, n)])
            sm.update_nodes(ids, est[ids], passes[ids], n_nodes=n)
        sent = est[:n].copy()

    def batch(est, n, mode):
        table(est, n)
        sm.enumerate_pairs_device(mode, 5.0, 2.0)
        pairs = sm.fetch_pairs()
        sm.run(p)
        out.append((pairs[0].tobytes(), pairs[1].tobytes(), pairs[2].tobytes(), sm.fetch_results().tobytes(),
                    sm.fetch_factors().tobytes()))

    for k in range(len(ranges)):
        est = est_of(k)
        if k > 0 and passes[k] != passes[k - 1]:
            batch(est, k, ENUM_REOPTIMIZE)
        sm.append_ranges(ranges[k:k + 1], sc)
        if k >= 1:
            batch(est, k + 1, ENUM_ONLINE)
    return out


def _optimised_estimates(est0, seed, last=6, every=17):
    """estimate vector after update k: the last `last` estimates perturbed, and every `every` updates all of them"""
    rng = np.random.default_rng(seed)
    cur, hist = est0.copy(), []
    for k in range(len(est0)):
        lo = 0 if k % every == every - 1 else max(0, k + 1 - last)
        cur[lo:k + 1] += rng.normal(0, [0.02, 0.02, 0.004], (k + 1 - lo, 3)).astype(F32)
        hist.append(cur.copy())
    return hist.__getitem__


def test_online_replay_records_and_factors_equal_set_nodes():
    wl = synth.config_corridor_passes(150, 256, 3, seed=54)
    est_of = _optimised_estimates(wl.poses_est.astype(F32), 54)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    runs = {}
    for nodes in ("full", "update", "sync"):
        with ScanMatcher(0) as sm:
            runs[nodes] = _replay(sm, wl.ranges, wl.scanner, est_of, wl.passes, p, nodes)
    assert sum(len(b[0]) for b in runs["full"]) // 4 > len(runs["full"])          # loop closures on later passes
    assert runs["update"] == runs["full"]
    assert runs["sync"] == runs["full"]


# ---- 5. refusals leave the table as it was ------------------------------------------------------------------------
def test_refusals_leave_the_table():
    poses, passes = EC.walk(200, seed=55)
    with ScanMatcher(0) as sm:
        sm.set_nodes(poses[:150], passes[:150])
        before = _lists(sm)
        lib, h = sm._lib, sm._h
        ids = np.array([3, 7], np.int32)
        two = poses[[3, 7]] + F32(9.0)
        pa = passes[[3, 7]].copy()

        def raw(n_nodes, i, pz, ps, k):
            return lib.dpgicp_update_nodes(h, n_nodes, None if i is None else i.ctypes.data,
                                           None if pz is None else pz.ctypes.data, None if ps is None else ps.ctypes.data, k)

        nan = two.copy(); nan[1, 0] = np.nan
        inf = two.copy(); inf[0, 2] = np.inf
        ninf = two.copy(); ninf[1, 1] = -np.inf
        new = np.array([150, 151], np.int32)
        cases = [
            (E_INVALID, lambda: raw(149, ids, two, pa, 2)),                                   # shrinking
            (E_INVALID, lambda: raw(152, np.array([150, 3], np.int32), two, pa, 2)),          # new id 151 missing
            (E_INVALID, lambda: raw(151, None, None, None, 0)),                               # new id 150 missing
            (E_INVALID, lambda: raw(150, np.array([7, 7], np.int32), two, pa, 2)),            # duplicate
            (E_INVALID, lambda: raw(152, np.array([151, 150, 151], np.int32), np.tile(two[:1], (3, 1)), np.zeros(3, np.int32), 3)),
            (E_INVALID, lambda: raw(150, np.array([-1, 3], np.int32), two, pa, 2)),           # out of range
            (E_INVALID, lambda: raw(150, np.array([3, 150], np.int32), two, pa, 2)),
            (E_INVALID, lambda: raw(150, None, two, pa, 2)),                                  # NULL arrays
            (E_INVALID, lambda: raw(150, ids, None, pa, 2)),
            (E_INVALID, lambda: raw(150, ids, two, None, 2)),
            (E_INVALID, lambda: raw(150, ids, two, pa, -1)),
            (E_RANGE, lambda: raw(150, ids, nan, pa, 2)),                                     # non-finite estimates
            (E_RANGE, lambda: raw(150, ids, inf, pa, 2)),
            (E_RANGE, lambda: raw(152, new, ninf, pa, 2)),                                    # also when growing
        ]
        for k, (code, call) in enumerate(cases):
            assert call() == code, k
            assert _lists(sm) == before, f"refusal {k} changed the table"
        assert raw(150, None, None, None, 0) == 0                                             # n_ids = 0: no-op
        assert _lists(sm) == before
        with pytest.raises(ValueError):
            sm.update_nodes([1, 2], poses[:3], passes[:2])
        with pytest.raises(DpgIcpError):
            sm.update_nodes([1], poses[1:2], passes[1:2], n_nodes=10)
        with pytest.raises(ValueError):                                  # would wrap to id 3 as int32
            sm.update_nodes(np.array([2**32 + 3], np.int64), poses[3:4], passes[3:4])
        with pytest.raises(ValueError):
            sm.update_nodes([3], poses[3:4], np.array([2**31], np.int64))
        assert _lists(sm) == before


# ---- 6. a slot enumerated before an update runs the old table's guesses ----------------------------------------------
def test_slot_keeps_the_guesses_it_was_enumerated_with():
    wl = synth.config_corridor_passes(400, 512, 2, seed=56)
    old = wl.poses_est.astype(F32)
    new = old.copy()
    new[200:] += F32(0.25)
    p = Params.defaults(cov_mode=COV_CENSI_CORR)
    with ScanMatcher(0) as sm, ScanMatcher(0) as ref:
        for m in (sm, ref):
            m.upload_ranges(wl.ranges, wl.scanner)
        ref.set_nodes(old, wl.passes)
        ref.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0)
        ref.run(p)
        want_old = ref.fetch_results().tobytes()
        ref.set_nodes(new, wl.passes)
        want_new = _lists(ref)
        sm.set_nodes(old, wl.passes)
        s = sm.slot()
        s.enumerate_pairs_device(ENUM_REOPTIMIZE, 5.0, 2.0)
        ids = np.arange(200, 400)
        sm.update_nodes(ids, new[ids], wl.passes[ids])
        s.run(p)
        assert s.fetch_results().tobytes() == want_old
        assert _lists(sm) == want_new
        s.close()


# ---- 7. set_nodes and update_nodes mixed; the host-list form is unaffected ---------------------------------------------
def test_set_nodes_interplay_and_host_list():
    poses, passes = EC.walk(2500, seed=57, sessions=3)
    rng = np.random.default_rng(57)
    xy2, pass2 = EC.walk(700, seed=58)
    host_want = R.enumerate_reoptimize(xy2[:, :2], pass2, 5.0, 2.0)

    def host_list(sm):
        s, t = sm.enumerate_pairs(xy2[:, :2], pass2, 5.0, 2.0)
        assert np.array_equal(s, host_want[0]) and np.array_equal(t, host_want[1])

    with ScanMatcher(0) as sm, ScanMatcher(0) as ref:
        cur = poses.copy()
        sm.update_nodes(np.arange(1000), cur[:1000], passes[:1000])
        host_list(sm)
        _assert_same_as_set_nodes(sm, ref, cur[:1000], passes[:1000], "updates")
        sm.set_nodes(cur[:300], passes[:300])                              # set_nodes after updates: smaller table
        host_list(sm)
        _assert_same_as_set_nodes(sm, ref, cur[:300], passes[:300], "set_nodes after updates")
        ids = np.concatenate([rng.choice(300, 40, replace=False), np.arange(300, 2500)])
        cur[ids] += F32(0.125)
        sm.update_nodes(ids, cur[ids], passes[ids])                        # grows past the earlier capacity
        host_list(sm)
        _assert_same_as_set_nodes(sm, ref, cur, passes, "updates after set_nodes")
        sm.set_nodes(cur, passes)
        sm.update_nodes([17], cur[17:18] + F32(1.0), passes[17:18])
        cur[17] += F32(1.0)
        host_list(sm)
        _assert_same_as_set_nodes(sm, ref, cur, passes, "one update after a full set_nodes")


# ---- 8. sync_nodes and the runner's --replay --nodes sync ------------------------------------------------------------
def test_sync_nodes_equals_set_nodes():
    poses, passes = EC.walk(3000, seed=59)
    rng = np.random.default_rng(59)
    with ScanMatcher(0) as sm, ScanMatcher(0) as ref:
        cur = poses[:100].copy()
        for step in range(40):
            n = len(cur)
            if step % 9 == 8:
                cur = cur + F32(0.01)                                      # every node: a full set_nodes
            else:
                ids = rng.choice(n, int(rng.integers(0, 20)), replace=False)
                cur[ids] += F32(0.05)
            grow = int(rng.integers(0, 80))
            cur = np.concatenate([cur, poses[n:n + grow]])
            sm.sync_nodes(cur, passes[:len(cur)])
            _assert_same_as_set_nodes(sm, ref, cur, passes[:len(cur)], f"step {step}")
        with pytest.raises(ValueError):
            sm.sync_nodes(cur[:, :2], passes[:len(cur)])
        sm.sync_nodes(cur[:50], passes[:50])                               # shorter: the whole table again
        _assert_same_as_set_nodes(sm, ref, cur[:50], passes[:50], "shorter")


def test_runner_replay_nodes_sync_writes_the_full_csv(tmp_path):
    csv = {m: str(tmp_path / f"{m}.csv") for m in ("full", "sync")}
    lines = {}
    for m in ("full", "sync"):
        extra = [] if m == "full" else ["--nodes", "sync"]
        r = subprocess.run([RUNNER, "--replay", "--synthetic", "corridor", "--scans", "300", "--passes", "3", "--beams", "256",
                            "--cov-mode", "2", "--out", csv[m]] + extra, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr
        lines[m] = r.stdout.strip().splitlines()[-1]
        assert f'"nodes": "{m}"' in lines[m]
    assert open(csv["full"], "rb").read() == open(csv["sync"], "rb").read()
