"""The CPU oracle against the independent float64 reference (tests/f64_reference.py): correspondences bit for bit, the
outlier rejectors' kept sets at their edges, one ICP pass within the bound derived from the arithmetic contract, and the
int64 headroom of the moment sums at the parameter limits.  A contract error that the oracle and the CUDA path share
would pass every oracle-vs-GPU test; these would catch it.  The case builders here are shared with the GPU leg
(tests/test_gpu_independent_reference.py)."""
import math

import numpy as np
import pytest

import f64_reference as R
from dpg_slam_b200 import synth
from dpg_slam_b200._abi import (METRIC_POINT_TO_LINE, OUTLIER_MEDIAN, OUTLIER_NONE, OUTLIER_TRIMMED, SEARCH_BRUTE,
                                SEARCH_PROJECTIVE, STOP_MASK, STOP_NO_CORRESPONDENCES, Params)
from oracle import oracle_py as O

F32 = np.float32


# ---- case builders ------------------------------------------------------------------------------------------------
def column_case(offsets, spacing=1.5):
    """Targets on the y axis, source i at target i + offsets[i]: every source point's neighbour is its own target and the
    pair is reciprocal, so the accepted d2 multiset is exactly {fl(dx^2) + fl(dy^2)} and K = len(offsets)."""
    off = np.array([o if isinstance(o, tuple) else (o, 0.0) for o in offsets], np.float64).reshape(-1, 2)
    n = len(off)
    y = ((np.arange(n) - n // 2) * spacing).astype(F32)
    tgt = np.stack([np.zeros(n, F32), y], 1)
    src = np.stack([off[:, 0].astype(F32), y + off[:, 1].astype(F32)], 1).astype(F32)
    return src, tgt


def rejector_cases():
    """(name, src, tgt, mode, param) at the rejectors' edges"""
    rng = np.random.default_rng(5)
    c = []
    for k in (1, 2, 3, 4):                                        # fewer accepted pairs than the pass needs
        offs = [0.1, 0.2, 0.3, 0.4][:k]
        for mode, param in ((OUTLIER_MEDIAN, 0.5), (OUTLIER_MEDIAN, 1.0), (OUTLIER_TRIMMED, 0.5), (OUTLIER_TRIMMED, 1.0)):
            c.append((f"K{k}", *column_case(offs), mode, param))
    ties = [0.1] * 5 + [0.2] * 7 + [0.3] * 4                          # many d2 equal to the threshold
    c += [("ties", *column_case(ties), OUTLIER_TRIMMED, 0.4), ("ties", *column_case(ties), OUTLIER_MEDIAN, 1.0),
          ("ties", *column_case(ties), OUTLIER_MEDIAN, 0.999)]
    zeros = [0.0] * 9 + [0.1, 0.2, 0.3, 0.05]                          # median 0 -> tau 0
    c += [("zero", *column_case(zeros), OUTLIER_MEDIAN, 1.5), ("zero", *column_case(zeros), OUTLIER_TRIMMED, 0.5)]
    # median * factor exactly a binary32 value, with pairs exactly there: offset (0.2, 0.2) has d2 = 2 fl(0.2^2)
    exact = [0.1, 0.15, 0.2, 0.2, 0.2, (0.2, 0.2), (0.2, 0.2), 0.3, (0.1, 0.1), 0.35, 0.4]
    c += [("exact", *column_case(exact), OUTLIER_MEDIAN, 2.0), ("exact", *column_case(exact), OUTLIER_MEDIAN, 0.5)]
    # median * factor just below / just above a binary32 value: the largest binary32 <= it drops / keeps the median's ties
    near = [0.05, 0.1, 0.2, 0.2, 0.2, 0.2, 0.3, 0.4, 0.5]
    c += [("near", *column_case(near), OUTLIER_MEDIAN, 1.0 - 2.0 ** -30), ("near", *column_case(near), OUTLIER_MEDIAN, 1.0 + 2.0 ** -30)]
    # TRIMMED where param * K is an exact integer, where it is one in decimal but not in binary64 (0.1 * 30), and the clamp
    c += [("trim32", *column_case(rng.uniform(0.01, 0.5, 32)), OUTLIER_TRIMMED, 0.5),
          ("trim40", *column_case(np.repeat(rng.uniform(0.01, 0.5, 10), 4)), OUTLIER_TRIMMED, 0.75),
          ("trim30", *column_case(rng.uniform(0.01, 0.5, 30)), OUTLIER_TRIMMED, 0.1),
          ("clamp", *column_case(rng.uniform(0.01, 0.5, 20)), OUTLIER_TRIMMED, 0.05),
          ("clamp", *column_case(rng.uniform(0.01, 0.5, 7)), OUTLIER_TRIMMED, 0.2)]
    for k in (31, 32, 33):                                       # tile boundaries
        offs = np.round(rng.uniform(0.01, 0.5, k), 2)             # rounded: ties
        c += [(f"tile{k}", *column_case(offs), OUTLIER_MEDIAN, 1.0), (f"tile{k}", *column_case(offs), OUTLIER_TRIMMED, 0.6)]
    # d2 that differ only in the low byte (0.25 + k ulp: fl(dx^2) 2 ulps apart) among values spread over many exponents,
    # so that every radix round has to decide
    low = list(0.25 + np.arange(120) * 2.0 ** -25) + list(rng.uniform(1e-3, 0.55, 400)) + [0.25] * 5
    perm = rng.permutation(len(low))
    low = [low[i] for i in perm]
    for mode, param in ((OUTLIER_MEDIAN, 1.0), (OUTLIER_TRIMMED, 0.37), (OUTLIER_TRIMMED, 0.6)):
        c.append(("radix", *column_case(low), mode, param))
    # the median itself among the low-byte cluster
    low2 = list(0.25 + np.arange(200) * 2.0 ** -25) + list(rng.uniform(0.3, 0.55, 100)) + list(rng.uniform(0.01, 0.2, 99))
    c.append(("radix2", *column_case(low2), OUTLIER_MEDIAN, 1.0))
    return c


def lattice_case(rng, nt, ns, dup=False):
    """lattice clouds: many exact distance ties"""
    tgt = np.stack([rng.integers(0, 12, nt) * 0.25, rng.integers(0, 9, nt) * 0.25], 1).astype(F32)
    src = np.stack([rng.integers(0, 23, ns) * 0.125, rng.integers(0, 17, ns) * 0.125], 1).astype(F32)
    if dup:
        src = src[rng.integers(0, ns, ns)]
        tgt = tgt[rng.integers(0, nt, nt)]
    return src, tgt


def apply_T(T, xy):
    """x' = ((c x) + ((-s) y)) + tx, binary32, each operation rounded"""
    c, s, tx, ty = (F32(v) for v in T)
    x, y = xy[:, 0], xy[:, 1]
    return np.stack([((c * x) + ((-s) * y)) + tx, ((s * x) + (c * y)) + ty], 1).astype(F32)


def guess_T(g):
    return np.array([np.cos(np.float64(g[2])), np.sin(np.float64(g[2])), g[0], g[1]], np.float64).astype(F32)


def scan_pairs(wl, ks):
    """(source already at the pair's guess, target) of workload pairs ks"""
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    out = []
    for k in ks:
        s, t = int(wl.src_idx[k]), int(wl.tgt_idx[k])
        out.append((apply_T(guess_T(wl.guess[k]), pts[off[s]:off[s + 1]]), pts[off[t]:off[t + 1]].copy()))
    return out


def far_pair(rng, n, centre, noise=0.02, theta=0.01, shift=(0.05, -0.03)):
    """a wall-like cloud of n points near `centre` (|coord| up to ~1000) and a slightly moved copy"""
    u = np.linspace(-4, 4, n)
    tgt = np.stack([centre[0] + u, centre[1] + 0.3 * np.sin(1.7 * u) + 0.5 * (u > 1)], 1)
    c, s = math.cos(theta), math.sin(theta)
    d = tgt - np.array(centre)
    src = np.stack([c * d[:, 0] - s * d[:, 1], s * d[:, 0] + c * d[:, 1]], 1) + np.array(centre) + np.array(shift)
    src = src + rng.normal(0, noise, src.shape)
    return src.astype(F32), tgt.astype(F32)


def small_cases(rng):
    """n in {1, 2, 3, 31, 32, 33}: source and target of that size"""
    out = []
    for n in (1, 2, 3, 31, 32, 33):
        tgt = (rng.uniform(-3, 3, (n, 2))).astype(F32)
        src = (tgt + rng.normal(0, 0.15, (n, 2))).astype(F32)
        out.append((f"n{n}", src, tgt))
    return out


def big_far_case(rng, n=8192):
    """8192-point clouds centred near (+-990, +-990)"""
    cx, cy = rng.choice([-990.0, 990.0], 2)
    tgt = np.stack([cx + rng.uniform(-9, 9, n), cy + rng.uniform(-9, 9, n)], 1).astype(F32)
    src = (tgt + rng.normal(0, 0.12, (n, 2))).astype(F32)
    return "far8192", src[rng.permutation(n)], tgt


def step_cases():
    """(name, src at the pair's guess, tgt) for one pass from a theta = 0 guess"""
    rng = np.random.default_rng(17)
    wl = synth.config_corridor(n_pairs=12, seed=21)
    lc = synth.config_loop_closure(n_pairs=12, n_scans=30, seed=32)
    cases = [("corridor", s, t) for s, t in scan_pairs(wl, range(0, 12, 3))]
    cases += [("loop_closure", s, t) for s, t in scan_pairs(lc, range(0, 12, 4))]
    for centre in ((990.0, -985.0), (-700.0, 995.0)):            # Sum pq - Sum p Sum q / K cancels heavily
        cases.append(("far", *far_pair(rng, 700, centre)))
    tgt3 = np.array([[0.0, 0.0], [1.0, 0.2], [0.3, 1.1]], F32)
    cases.append(("K3", (tgt3 + np.array([[0.05, -0.02], [0.03, 0.04], [-0.06, 0.01]])).astype(F32), tgt3))
    # h = 0: four source points symmetric around one target point, every pair on it (no reciprocity)
    cases.append(("h0", np.array([[5.25, 3.0], [4.75, 3.0], [5.0, 3.25], [5.0, 2.75]], F32), np.array([[5.0, 3.0], [40.0, 40.0]], F32)))
    return cases


def ring_case(n=8192, radius=29.99, cluster=256, duplicates=False, seed=3):
    """the parameter limits: a dense target cluster at about (970, 970) and n source points on a ring around it, all
    within a 30 m gate: Sum d2 2^40 near 0.88 * 2^63.  With ``duplicates`` the target is one point repeated, so that
    point-to-line has no usable segment and every pair contributes the two isolated-point rows."""
    rng = np.random.default_rng(seed)
    c = np.array([970.0, 970.0])
    if duplicates:
        tgt = np.repeat(c[None], 4, 0).astype(F32)
    else:
        tgt = (c + rng.uniform(-0.005, 0.005, (cluster, 2))).astype(F32)
    a = np.sort(rng.uniform(-np.pi, np.pi, n))
    src = (c + radius * np.stack([np.cos(a), np.sin(a)], 1)).astype(F32)
    return src, tgt


def params_for(search=SEARCH_BRUTE, reciprocal=1, r=0.6, mode=OUTLIER_NONE, param=0.0, window=8, **kw):
    return Params.defaults(downsample_divisor=1, search=search, use_reciprocal=reciprocal, max_correspondence_distance=r,
                           outlier_mode=mode, outlier_param=param, projective_window=window, **kw)


def reference_pass(src, tgt, p, prev_nn=None):
    return R.pass_pairs(src, tgt, p.max_correspondence_distance, bool(p.use_reciprocal), p.outlier_mode, p.outlier_param,
                        prev_nn=prev_nn, projective_full=p.search == SEARCH_PROJECTIVE)


def reference_step(src, tgt, p):
    """-> (K, (c, s, tx, ty), mse, bounds) of one pass from the identity, or (K, None, None, None) when K < 3"""
    m = reference_pass(src, tgt, p)
    acc = m.corr >= 0
    K = int(acc.sum())
    if K < 3:
        return K, None, None, None
    P, Q = src[acc], tgt[m.corr[acc]]
    mse = R.mse(m.d2[acc])
    if p.metric == METRIC_POINT_TO_LINE:
        J, r = R.p2l_rows(P, tgt, m.corr[acc], R.gate_threshold(p.max_correspondence_distance))
        st = R.step_p2l(J, r)
        return K, st, mse, R.p2l_bounds(J, r, st, mse)
    st = R.step_p2p(P, Q)
    return K, st, mse, R.p2p_bounds(P, Q, st, mse)


def check_step(rec, K, st, mse, b, ctx):
    """record (c, s, tx, ty, mse) of one pass against the reference; returns the errors as fractions of their bounds"""
    assert int(rec["n_correspondences"]) == K, ctx
    err = dict(cs=max(abs(float(rec["rot_c"]) - st[0]), abs(float(rec["rot_s"]) - st[1])) / b.cs,
               tx=abs(float(rec["tx"]) - st[2]) / b.tx, ty=abs(float(rec["ty"]) - st[3]) / b.ty,
               mse=abs(float(rec["mse"]) - mse) / b.mse)
    assert max(err.values()) <= 1.0, (ctx, err, b)
    return err


# ---- correspondences -----------------------------------------------------------------------------------------------
def corr_cases():
    rng = np.random.default_rng(11)
    wl = synth.config_corridor(n_pairs=8, seed=21)
    cases = [("corridor", s, t, None, 0.6) for s, t in scan_pairs(wl, (0, 3, 6))]
    for k in range(6):
        s, t = lattice_case(rng, int(rng.integers(1, 300)), int(rng.integers(1, 300)), dup=k % 2 == 1)
        cases.append(("lattice", s, t, rng.integers(-1, len(t), len(s)).astype(np.int32), (0.2, 0.6, 1.5)[k % 3]))
    cases += [(n, s, t, None, 0.6) for n, s, t in small_cases(rng)]
    cases.append(big_far_case(rng) + (None, 0.6))
    return cases


@pytest.mark.parametrize("reciprocal", [1, 0])
def test_reference_correspondences_equal_oracle(reciprocal):
    """Exact search (brute force and the grid) and the projective search with a window covering the cloud: the oracle's
    neighbours, accepted sets, seeds handed on and binary32 distances are the reference's."""
    for name, src, tgt, seed, r in corr_cases():
        p = params_for(reciprocal=reciprocal, r=r)
        want = reference_pass(src, tgt, p, prev_nn=seed)
        for fast in (0, 1):
            if seed is None:
                k, corr, d2 = O.correspondences(src, tgt, p, fast=fast)
            else:
                k, corr, d2, nn = O.correspondences(src, tgt, p, fast=fast, prev_nn=seed)
                assert np.array_equal(nn, want.nn), (name, fast)
            assert k == want.k and np.array_equal(corr, want.corr), (name, fast)
            assert np.array_equal(d2[want.fwd].view(np.uint32), want.d2[want.fwd].view(np.uint32)), (name, fast)
        if len(src) <= 1024 and len(tgt) <= 1024:
            pp = p.copy(search=SEARCH_PROJECTIVE, projective_window=1024)
            wp = reference_pass(src, tgt, pp)
            _, corr, _ = O.correspondences(src, tgt, pp, src_orig=src, T=np.array([1, 0, 0, 0], F32))
            assert np.array_equal(corr, wp.corr), (name, "projective")


def test_reference_beam_key_orders_like_atan2():
    """the §5.7 key as the reference states it equals the oracle's bit for bit and is monotone in atan2"""
    rng = np.random.default_rng(2)
    v = rng.normal(0, 5, (4000, 2)).astype(F32)
    v[:8] = [[1, 0], [0, 1], [-1, 0], [0, -1], [1, 1], [-1, 1], [-1, -1], [1, -1]]
    key = R.beam_key(v[:, 0], v[:, 1], 0.0, 0.0)
    want = np.array([O.lib().orc_beam_key(float(x), float(y), 0.0, 0.0) for x, y in v], F32)
    assert np.array_equal(key.view(np.uint32), want.view(np.uint32))
    order = np.argsort(np.arctan2(v[:, 1].astype(np.float64), v[:, 0].astype(np.float64)), kind="stable")
    assert np.all(np.diff(key[order]) >= 0)


# ---- rejectors -----------------------------------------------------------------------------------------------------
def test_reference_rejector_kept_sets_equal_oracle():
    """Every rejector edge: K in {1, 2, 3, 4}, ties at the threshold, d2 = 0, median * factor exactly on / just off a
    binary32 value, param * K an exact integer, the max(3, .) clamp, tile boundaries, low-byte differences.  Threshold
    and kept set of the oracle equal the reference's, for the exact and the projective search, with and without
    reciprocity."""
    for name, src, tgt, mode, param in rejector_cases():
        for search in (SEARCH_BRUTE, SEARCH_PROJECTIVE):
            for rec in (1, 0):
                p = params_for(search=search, reciprocal=rec, mode=mode, param=param, window=1024)
                want = reference_pass(src, tgt, p)
                k, corr, d2 = O.correspondences(src, tgt, p, src_orig=src, T=np.array([1, 0, 0, 0], F32))
                assert k == want.k and np.array_equal(corr, want.corr), (name, mode, param, search, rec)
        acc = reference_pass(src, tgt, params_for()).d2
        assert O.outlier_threshold(acc, params_for(mode=mode, param=param)) == R.reject(acc, mode, param), (name, mode, param)


def test_small_k_median_rejects_as_defined():
    """MEDIAN 0.5 with one or two accepted pairs keeps fewer than all of them (the pass stops on K < 3 either way)"""
    for k, kept in ((1, 0), (2, 1)):
        src, tgt = column_case([0.1, 0.2][:k])
        p = params_for(mode=OUTLIER_MEDIAN, param=0.5)
        assert reference_pass(src, tgt, p).k == kept
        r = O.icp(src, tgt, np.zeros(3, F32), p.copy(max_iterations=1))
        assert r.n_correspondences == kept and (r.status & STOP_MASK) == STOP_NO_CORRESPONDENCES


def test_reference_rejector_with_seeds_equals_oracle():
    """the sticky tie rule and a rejector together, on lattice clouds with random seeds"""
    rng = np.random.default_rng(91)
    for trial in range(10):
        src, tgt = lattice_case(rng, int(rng.integers(3, 300)), int(rng.integers(3, 300)), dup=trial % 2 == 1)
        seed = rng.integers(-1, len(tgt), len(src)).astype(np.int32)
        for mode, param in ((OUTLIER_TRIMMED, 0.6), (OUTLIER_MEDIAN, 1.0), (OUTLIER_MEDIAN, 0.5)):
            p = params_for(mode=mode, param=param, reciprocal=trial % 3 != 0, r=0.6)
            want = reference_pass(src, tgt, p, prev_nn=seed)
            k, corr, _, nn = O.correspondences(src, tgt, p, prev_nn=seed)
            assert np.array_equal(corr, want.corr) and np.array_equal(nn, want.nn), (trial, mode, param)


# ---- one pass --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", [0, METRIC_POINT_TO_LINE])
def test_one_pass_of_the_oracle_within_the_derived_bound(metric):
    """max_iterations = 1 from a theta = 0 guess (c = 1, s = 0 exactly with any libm): the record pose is the step, and
    it lies within the bound derived from the contract (f64_reference docstring) around the float64 reference step.  On
    corridor scans that bound is below 1e-6 m, else the check would have no teeth."""
    worst = {}
    for name, src, tgt in step_cases():
        rec_p = params_for(reciprocal=0 if name == "h0" else 1, metric=metric, max_iterations=1)
        K, st, mse, b = reference_step(src, tgt, rec_p)
        if st is None or (metric and name == "h0"):
            continue
        r = O.icp(src, tgt, np.zeros(3, F32), rec_p)
        rec = dict(rot_c=r.rot_c, rot_s=r.rot_s, tx=r.tx, ty=r.ty, mse=r.mse, n_correspondences=r.n_correspondences)
        err = check_step(rec, K, st, mse, b, (name, metric))
        if name == "corridor":
            assert b.pose < 1e-6, f"pose bound {b.pose:.2e} m on a corridor pair: no teeth"
        if name == "h0":
            assert (r.rot_c, r.rot_s) == (1.0, 0.0)
        w = worst.setdefault(name, [0.0, 0.0, 0.0])
        w[0] = max(w[0], b.pose)
        w[1] = max(w[1], abs(r.tx - st[2]), abs(r.ty - st[3]))
        w[2] = max(w[2], err["mse"])
    print("\n[one pass, oracle] metric", metric, {k: f"bound {v[0]:.2e} m, max |dt| {v[1]:.2e} m, mse err/bound {v[2]:.2f}" for k, v in worst.items()})


@pytest.mark.parametrize("metric", [0, METRIC_POINT_TO_LINE])
def test_oracle_moment_sums_fit_at_the_parameter_limits(metric):
    """8192 pairs at d2 ~ 899 under a 30 m gate near (970, 970): Sum d2 2^40 ~ 0.88 * 2^63 must not wrap (mse within
    the bound of fsum), and the pass stays within the derived bound."""
    src, tgt = ring_case(duplicates=metric == METRIC_POINT_TO_LINE)
    p = params_for(reciprocal=0, r=30.0, metric=metric, max_iterations=1)
    K, st, mse, b = reference_step(src, tgt, p)
    assert K == 8192
    d2 = reference_pass(src, tgt, p).d2
    frac = sum(int(np.rint(float(v) * 2.0 ** 40)) for v in d2) / 2.0 ** 63
    print(f"\n[contract limit] metric {metric}: Sum d2 2^40 = {frac:.4f} of 2^63")
    assert 0.85 < frac < 1.0
    r = O.icp(src, tgt, np.zeros(3, F32), p)
    rec = dict(rot_c=r.rot_c, rot_s=r.rot_s, tx=r.tx, ty=r.ty, mse=r.mse, n_correspondences=r.n_correspondences)
    check_step(rec, K, st, mse, b, ("limit", metric))
