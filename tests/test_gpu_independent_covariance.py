"""GPU (B200): the CUDA covariance and factor hand-off against the independent float64 reference
(tests/f64_covariance.py), not the oracle.  The standalone kernels (dpgicp_cov at both point strides, dpgicp_cov_pairs at
every DPGICP_COV_WARPS width) at the odd/even tails of every width's stride, the cap edges, unequal and empty clouds, far
clouds, theta = +-pi and the singular cases; the covariance of whole-run and one-pass records (INDEXPAIR and CORR,
divisor 1 and 5, each rejector, both metrics) under forced stage chains, with caps that end inside a tile, on a tile
edge and across a CTA edge of the cluster stage; and dpgicp_fetch_factors, including FLAG_FACTOR_INVALID."""
import numpy as np
import pytest

import f64_covariance as FC
import f64_reference as R
from dpg_slam_b200._abi import COV_CENSI_CORR, COV_CENSI_INDEXPAIR, FLAG_FACTOR_INVALID, Params
from dpg_slam_b200.scanmatch import ScanMatcher
from test_independent_covariance import (Worst, check_cov, check_factor, check_theta, cov_cases, family,
                                         invalid_factor_params, record_cases, record_pairs, run_params, tie_cases)

pytestmark = pytest.mark.gpu
F32 = np.float32
CUDA_ATAN2F_ULPS = 3              # the record's theta is the device's atan2f
CHAINS = (None, "1", "32", "4,8,16,9x2", "2,5x2", "4,16x4")


def store_of(clouds):
    off = np.zeros(len(clouds) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in clouds])
    pts = np.concatenate([np.asarray(c, F32).reshape(-1, 2) for c in clouds]) if clouds else np.zeros((0, 2), F32)
    return pts.astype(F32), off


def T4(T):
    c, s, tx, ty = (float(v) for v in T)
    return np.array([[c, -s, 0, tx], [s, c, 0, ty], [0, 0, 1, 0], [0, 0, 0, 1]], F32)


def kernel_cases():
    """cov_cases plus odd and even n around every width's stride, unequal clouds both ways and an empty scan"""
    rng = np.random.default_rng(50)
    T = np.array([np.cos(0.2), np.sin(0.2), -0.3, 0.45], F32)
    out = list(cov_cases())
    for n in (63, 64, 65, 255, 256, 257, 8191):
        P = rng.uniform(-8, 8, (n, 2)).astype(F32)
        out.append((f"n{n}", P, (P + rng.normal(0, 0.05, P.shape)).astype(F32), 200, T))
    P = rng.uniform(-8, 8, (301, 2)).astype(F32)
    Q = (P + rng.normal(0, 0.05, P.shape)).astype(F32)
    out += [("unequal", P, Q[:250], 0, T), ("unequal", P[:257], Q, 256, T), ("unequal", P[:33], Q, 32, T),
            ("empty", np.zeros((0, 2), F32), Q, 200, T), ("empty", P, np.zeros((0, 2), F32), 200, T)]
    return out


def reference_of(P, Q, cap, T):
    n_h = min(len(P), len(Q))
    return FC.censi_T(P, Q, n_h, FC.cap_of(n_h, cap), T)


def test_dpgicp_cov_both_strides_within_the_derived_bound(gpu_matcher):
    """dpgicp_cov, packed xy (stride 8) and PointXYZ layout (stride 16): status word equal, covariance within the bound"""
    worst = Worst("dpgicp_cov, relative to max |cov|")
    for name, P, Q, cap, T in kernel_cases():
        ref = reference_of(P, Q, cap, T)
        p = Params.defaults(cov_mode=COV_CENSI_INDEXPAIR, cov_cap=cap)
        for stride in (8, 16):
            a, b = P, Q
            if stride == 16:
                a = np.concatenate([P, np.zeros((len(P), 2), F32)], 1)
                b = np.concatenate([Q, np.zeros((len(Q), 2), F32)], 1)
            if len(a) == 0 or len(b) == 0:
                a = a if len(a) else np.zeros((0, stride // 4), F32)
                b = b if len(b) else np.zeros((0, stride // 4), F32)
            cov, st = gpu_matcher.calculate_icp_cov(a, b, T4(T), p)
            worst.add(family(name), check_cov(cov, st, ref, (name, stride)), ref.rel_bound)
    worst.show()


@pytest.mark.parametrize("warps", [1, 2, 4, 8])
def test_dpgicp_cov_pairs_every_width_within_the_derived_bound(gpu_matcher, monkeypatch, warps):
    """dpgicp_cov_pairs over the scan store at DPGICP_COV_WARPS = 1, 2, 4, 8: one call per cap, status words equal"""
    monkeypatch.setenv("DPGICP_COV_WARPS", str(warps))
    cases = kernel_cases()
    pts, off = store_of([c for _, P, Q, _, _ in cases for c in (P, Q)])
    gpu_matcher.upload_scans(pts, off)
    worst = Worst(f"dpgicp_cov_pairs warps {warps}, relative to max |cov|")
    for cap in sorted({c[3] for c in cases}):
        ks = [k for k, c in enumerate(cases) if c[3] == cap]
        T = np.array([cases[k][4] for k in ks], F32)
        cov, st, _ = gpu_matcher.calculate_icp_cov_pairs([2 * k for k in ks], [2 * k + 1 for k in ks], T,
                                                         Params.defaults(cov_mode=COV_CENSI_INDEXPAIR, cov_cap=cap))
        for j, k in enumerate(ks):
            name, P, Q, _, Tk = cases[k]
            ref = reference_of(P, Q, cap, Tk)
            worst.add(family(name), check_cov(cov[j], st[j], ref, (name, cap, warps)), ref.rel_bound)
    worst.show()


# ---- records -----------------------------------------------------------------------------------------------------------
def edge_caps(keep_src, warps=(1, 2, 4, 5, 8, 9, 16)):
    """caps whose first `cap` ranks end on a tile edge (32 source points), one pair inside / past it, and on the edges of
    the CTAs of cluster stages (tile t belongs to CTA (t / warps) % cluster)"""
    keep_src = np.asarray(keep_src)
    tiles = sorted({t for w in warps for t in (w, 2 * w, 3 * w)} | {1, 2, 3})
    caps = set()
    for t in tiles:
        c = int((keep_src < 32 * t).sum())
        if 0 < c < len(keep_src):
            caps |= {c - 1, c, c + 1}
    return sorted(c for c in caps if c > 0) + [len(keep_src) - 1, len(keep_src), len(keep_src) + 1]


class RefCache:
    def __init__(self):
        self.d = {}

    def cov(self, k, case, rec, p, seeded):
        key = (k, tuple(float(rec[f]) for f in ("tx", "ty", "rot_c", "rot_s", "theta")), bytes(p), seeded)
        if key not in self.d:
            name, s, t, g = case
            pairs = record_pairs(rec, s, t, g, p, seeded)
            if pairs is None:
                self.d[key] = None
            else:
                P, Q, n_h, n_d = pairs
                live = (p.laser_x_variance, p.laser_y_variance, p.laser_theta_variance)
                self.d[key] = FC.censi(P, Q, n_h, n_d, float(rec["tx"]), float(rec["ty"]), float(rec["theta"]),
                                       p.cov_sensor_variance, live)
        return self.d[key]


def check_batch(recs, cases, p, seeded, cache, worst, ctx):
    n = 0
    for k, (case, rec) in enumerate(zip(cases, recs)):
        check_theta(rec, CUDA_ATAN2F_ULPS, (ctx, case[0]))
        ref = cache.cov(k, case, rec, p, seeded)
        if ref is None:
            continue
        err = check_cov(rec["cov"], rec["status"], ref, (ctx, case[0], p.cov_mode, p.downsample_divisor, p.outlier_mode,
                                                       p.metric, p.cov_cap))
        worst.add(family(case[0]), err, ref.rel_bound)
        n += 1
    return n


def test_record_covariance_under_forced_chains(monkeypatch):
    """submit_pairs records (whole runs, and lattice ties through max_iterations = 1) against the reference at the
    record's pose, under the default shape, 1-warp and 32-warp CTAs and cluster chains; CORR caps at tile and CTA edges"""
    cases, ties = record_cases(), tie_cases()
    pts, off = store_of([c for _, s, t, _ in cases + ties for c in (s, t)])
    n, m = len(cases), len(ties)
    idx = np.arange(0, 2 * (n + m), 2)
    guess = np.array([g for *_, g in cases + ties], F32)
    base = run_params()
    edge = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR, max_iterations=60)
    cache, worst, checked, skipped = RefCache(), Worst("records, relative to max |cov|"), 0, 0
    caps = None
    for chain in CHAINS:
        if chain is None:
            monkeypatch.delenv("DPGICP_CHAIN", raising=False)
        else:
            monkeypatch.setenv("DPGICP_CHAIN", chain)
        ctx = f"chain {chain}"
        with ScanMatcher(0) as sm:
            sm.upload_scans(pts, off)
            if caps is None:                               # the corridor pair's kept pairs at its final pose
                rec = sm.submit_pairs(idx[:1], idx[:1] + 1, guess[:1], edge)[0]
                _, s, t, _ = cases[0]
                m0 = R.pass_pairs(FC.apply_T((rec["rot_c"], rec["rot_s"], rec["tx"], rec["ty"]), s), t, 0.6, True)
                caps = edge_caps(np.nonzero(m0.corr >= 0)[0])
            for p in base:
                recs = sm.submit_pairs(idx[:n], idx[:n] + 1, guess[:n], p)
                k = check_batch(recs, cases, p, False, cache, worst, ctx)
                checked, skipped = checked + k, skipped + n - k
                q = p.copy(max_iterations=1)
                recs = sm.submit_pairs(idx[n:], idx[n:] + 1, guess[n:], q)
                check_batch(recs, ties, q, True, cache, worst, ctx + " ties")
            for cap in caps:                               # corridor and loop-closure pairs
                p = edge.copy(cov_cap=cap)
                recs = sm.submit_pairs(idx[:4], idx[:4] + 1, guess[:4], p)
                checked += check_batch(recs, cases[:4], p, False, cache, worst, ctx + " cap edges")
    worst.show()
    print(f"[whole runs] {checked} checked, {skipped} skipped for an exact tie at the final pose; caps {caps}")
    assert skipped <= checked // 10
    for fam in ("corridor", "loop_closure"):
        assert worst.bound(fam) < 1e-9, f"{fam}: bound {worst.bound(fam):.1e}: no teeth"


def test_fetch_factors_against_the_reference_factor(gpu_matcher):
    """dpgicp_fetch_factors of whole runs: the reference factor within its bound for valid covariances; under laser
    variances that are zero or negative (LIVE) and a zero sensor variance (CENSI), FLAG_FACTOR_INVALID with sqrt_info
    zeroed; from/to, pose and status bits exact"""
    cases = record_cases()[:6]
    pts, off = store_of([c for _, s, t, _ in cases for c in (s, t)])
    gpu_matcher.upload_scans(pts, off)
    n = len(cases)
    src, tgt = np.arange(0, 2 * n, 2), np.arange(1, 2 * n, 2)
    guess = np.array([g for *_, g in cases], F32)
    worst = Worst("fetch_factors, relative to max |R|")
    for p in invalid_factor_params() + [Params.defaults(cov_mode=COV_CENSI_CORR, downsample_divisor=1),
                                        Params.defaults(cov_mode=COV_CENSI_INDEXPAIR)]:
        recs = gpu_matcher.submit_pairs(src, tgt, guess, p)
        f = gpu_matcher.fetch_factors(n)
        for k in range(n):
            err = check_factor(f[k], recs[k], src[k], tgt[k], (cases[k][0], p.cov_mode))
            worst.add(f"cov_mode {p.cov_mode}", err, FC.factor(recs[k]["cov"]).rel_bound)
        invalid = (f["status"] & FLAG_FACTOR_INVALID) != 0
        assert invalid.all() == (p.cov_sensor_variance == 0 or min(p.laser_x_variance, p.laser_theta_variance) <= 0)
    worst.show()
