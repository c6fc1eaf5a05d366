"""The CPU oracle's covariance and factor against the independent float64 reference (tests/f64_covariance.py).  The
oracle and the CUDA path share one closed form and one pair selection, so a mistake made in both (the cap off by one,
the rejector skipped at the final pose, the D-term over the wrong pairs, INDEXPAIR on the down-sampled clouds) passes
every oracle-vs-GPU test; these would catch it.  The reference is itself pinned first, against the compiled reference's
golden vectors and SURVEY KAT-1.  The case builders here are shared with the GPU leg
(tests/test_gpu_independent_covariance.py)."""
import ctypes
import math

import numpy as np
import pytest

import f64_covariance as FC
import f64_reference as R
from dpg_slam_b200 import synth
from dpg_slam_b200._abi import (COV_CENSI_CORR, COV_CENSI_INDEXPAIR, COV_REFERENCE_LIVE, FLAG_COV_SINGULAR,
                                FLAG_FACTOR_INVALID, METRIC_POINT_TO_LINE, OUTLIER_MEDIAN, OUTLIER_NONE, OUTLIER_TRIMMED,
                                RESULT_DTYPE, SEARCH_BRUTE, SEARCH_PRUNED, Params)
from oracle import oracle_py as O
from test_independent_reference import far_pair, lattice_case

F32 = np.float32
HOST_ATAN2F_ULPS = 1            # glibc atan2f (x86_64), the oracle's record theta
LIBM = ctypes.CDLL("libm.so.6")
LIBM.atan2f.restype, LIBM.atan2f.argtypes = ctypes.c_float, [ctypes.c_float, ctypes.c_float]
REJECTORS = ((OUTLIER_NONE, 0.0), (OUTLIER_TRIMMED, 0.8), (OUTLIER_MEDIAN, 1.5))


def T_from_colmajor(Tc):
    return np.array([Tc[0], Tc[1], Tc[12], Tc[13]], F32)


# ---- case builders -----------------------------------------------------------------------------------------------------
def moved(rng, P, theta, t, noise):
    c, s = math.cos(theta), math.sin(theta)
    P = np.asarray(P, np.float64)
    Q = np.stack([c * P[:, 0] - s * P[:, 1], s * P[:, 0] + c * P[:, 1]], 1) + np.asarray(t) + rng.normal(0, noise, P.shape)
    return Q.astype(F32)


def cov_cases():
    """(name, P, Q, cap, T) for the closed form called directly (n_h = min(len P, len Q)): sizes, caps, far clouds,
    theta at +-pi and 0, exactly singular and near-singular Hessians"""
    rng = np.random.default_rng(40)
    T0 = np.array([math.cos(0.3), math.sin(0.3), 0.4, -0.25], F32)
    out = []
    for n in (0, 1, 2, 3, 31, 32, 33, 8192):
        P = rng.uniform(-8, 8, (n, 2)).astype(F32)
        Q = moved(rng, P, 0.3, (0.4, -0.25), 0.03)
        out.append((f"n{n}", P, Q, 200, T0))
    for n in (199, 201):
        P = rng.uniform(-8, 8, (n, 2)).astype(F32)
        Q = moved(rng, P, 0.3, (0.4, -0.25), 0.03)
        for cap in sorted({0, 1, n - 1, n, n + 1, 200}):
            out.append((f"n{n}_cap{cap}", P, Q, cap, T0))
    for cx, cy in ((990.0, 990.0), (-990.0, 985.0), (987.0, -990.0), (-990.0, -990.0)):
        P = (np.array([cx, cy]) + rng.uniform(-6, 6, (700, 2))).astype(F32)
        T = np.array([math.cos(0.01), math.sin(0.01), 0.05, -0.03], F32)
        Q = (P + rng.normal(0, 0.02, P.shape) + np.array([0.05, -0.03])).astype(F32)     # |coord| stays <= 1000
        out.append((f"far({cx:+.0f},{cy:+.0f})", P, Q, 200, T))
    P = rng.uniform(-8, 8, (300, 2)).astype(F32)
    tiny = float(np.nextafter(F32(0), F32(1)))
    for s in (0.0, -0.0, tiny, -tiny, 2.0 ** -23, -(2.0 ** -23)):         # theta at +-pi
        T = np.array([-1.0, s, 0.2, 0.1], F32)
        out.append((f"pi(s={s:+.3g})", P, moved(rng, P, math.pi, (0.2, 0.1), 0.03), 200, T))
    out.append(("theta0", P, moved(rng, P, 0.0, (0.2, 0.1), 0.03), 200, np.array([1, 0, 0.2, 0.1], F32)))
    out.append(("origin", np.zeros((50, 2), F32), rng.uniform(-2, 2, (50, 2)).astype(F32), 0, T0))   # exactly singular
    near = (rng.uniform(-1e-6, 1e-6, (60, 2))).astype(F32)
    out.append(("near_singular", near, rng.uniform(-2, 2, (60, 2)).astype(F32), 0, T0))
    return out


def scan_clouds(wl):
    pts, off = O.clouds_from_ranges(wl.ranges, wl.scanner)
    return [pts[off[k]:off[k + 1]] for k in range(len(off) - 1)]


def record_cases():
    """(name, src_full, tgt_full, guess) for whole runs: corridor and loop-closure scans, clouds of different sizes both
    ways, far from the origin, and K in {0, 1, 2, 3} at the final pose (plus an empty source)"""
    rng = np.random.default_rng(41)
    wl = synth.config_corridor(n_pairs=8, seed=21)
    cc = scan_clouds(wl)
    lc = synth.config_loop_closure(n_pairs=8, n_scans=30, seed=32)
    lcc = scan_clouds(lc)
    out = [("corridor", cc[wl.src_idx[k]], cc[wl.tgt_idx[k]], wl.guess[k]) for k in (0, 4)]
    out += [("loop_closure", lcc[lc.src_idx[k]], lcc[lc.tgt_idx[k]], lc.guess[k]) for k in (1, 5)]
    s, t, g = cc[wl.src_idx[2]], cc[wl.tgt_idx[2]], wl.guess[2]
    out += [("short_src", s[:-37], t, g), ("short_tgt", s, t[:-51], g)]
    for centre in ((990.0, -985.0), (-985.0, 990.0)):
        out.append(("far", *far_pair(rng, 700, centre), np.zeros(3, F32)))
    tgt3 = np.array([[0.0, 0.0], [1.0, 0.2], [0.3, 1.1], [3.0, 3.0]], F32)
    for k in (0, 1, 2, 3):
        src = (tgt3[:k] + np.array([[0.05, -0.02], [0.03, 0.04], [-0.06, 0.01]])[:k]).astype(F32)
        out.append((f"K{k}", np.concatenate([src, [[9.0, -9.0]]]).astype(F32), tgt3, np.zeros(3, F32)))
    out.append(("empty", np.zeros((0, 2), F32), tgt3, np.zeros(3, F32)))
    return out


def tie_cases():
    """(name, src_full, tgt_full, guess) on lattice clouds with exact ties, for max_iterations = 1 (theta = 0 guesses on
    the lattice, so the guess matrix is exact and the reference can produce the seeds of the covariance pass)"""
    rng = np.random.default_rng(42)
    out = []
    for k in range(8):
        s, t = lattice_case(rng, int(rng.integers(40, 300)), int(rng.integers(40, 300)), dup=k % 3 == 0)
        g = np.array([rng.integers(-1, 2) * 0.125, rng.integers(-1, 2) * 0.125, 0.0], F32)
        out.append((f"lattice{k}", s, t, g))
    return out


def run_params():
    """record parameter sets: INDEXPAIR and CORR, divisor 1 and 5, each rejector (CORR), both metrics, cap 200 / 0 / 7"""
    ps = []
    for div in (1, 5):
        ps.append(Params.defaults(downsample_divisor=div, cov_mode=COV_CENSI_INDEXPAIR, max_iterations=60))
        ps.append(Params.defaults(downsample_divisor=div, cov_mode=COV_CENSI_INDEXPAIR, max_iterations=60, cov_cap=0))
        for mode, q in REJECTORS:
            for metric in (0, METRIC_POINT_TO_LINE):
                ps.append(Params.defaults(downsample_divisor=div, cov_mode=COV_CENSI_CORR, max_iterations=60, metric=metric,
                                          outlier_mode=mode, outlier_param=q, cov_cap=(200, 0, 7)[(mode + metric) % 3]))
    return ps


# ---- the reference at a record ---------------------------------------------------------------------------------------
def record_pairs(rec, src_full, tgt_full, guess, p, seeded):
    """(P, Q, n_h, n_d) of a record, or None when the final pose has an exact forward tie and the seeds are unknown.
    ``seeded``: max_iterations = 1 from a theta = 0 guess, so the last pass's neighbours are pass 1's at the guess."""
    if p.cov_mode == COV_CENSI_INDEXPAIR:
        return FC.indexpair_pairs(src_full, tgt_full, p.cov_cap)
    div = max(1, p.downsample_divisor)
    s, t = FC.downsample(src_full, div), FC.downsample(tgt_full, div)
    T = (rec["rot_c"], rec["rot_s"], rec["tx"], rec["ty"])
    r, recip = p.max_correspondence_distance, bool(p.use_reciprocal)
    prev = None
    if seeded:
        assert guess[2] == 0
        prev = R.correspondences(FC.apply_T((1.0, 0.0, guess[0], guess[1]), s), t, r, recip).nn
    elif FC.forward_ties(FC.apply_T(T, s), t, r):
        return None
    return FC.corr_pairs(s, t, T, r, recip, p.outlier_mode, p.outlier_param, p.cov_cap, prev)


def reference_cov(rec, src_full, tgt_full, guess, p, seeded=False):
    pairs = record_pairs(rec, src_full, tgt_full, guess, p, seeded)
    if pairs is None:
        return None
    P, Q, n_h, n_d = pairs
    live = (p.laser_x_variance, p.laser_y_variance, p.laser_theta_variance)
    return FC.censi(P, Q, n_h, n_d, float(rec["tx"]), float(rec["ty"]), float(rec["theta"]), p.cov_sensor_variance, live)


def check_theta(rec, ulps, ctx):
    want = math.atan2(float(rec["rot_s"]), float(rec["rot_c"]))
    assert abs(float(rec["theta"]) - want) <= (ulps + 0.01) * R.ulp32(want), (ctx, float(rec["theta"]), want)


def check_cov(cov, status, ref, ctx):
    """status bit and covariance of one result against the reference; returns the relative error (None if ambiguous)"""
    cov = np.asarray(cov, np.float64).reshape(3, 3)
    if ref.ambiguous:
        return None
    assert (int(status) & FLAG_COV_SINGULAR) == ref.status, (ctx, hex(int(status)), ref.sigma_min, ref.h_err)
    if ref.status:
        assert np.array_equal(cov, ref.cov), ctx
        return 0.0
    bad = np.abs(cov - ref.cov) > ref.bound
    assert not bad.any(), (ctx, ref.rel_err(cov), ref.rel_bound, np.abs(cov - ref.cov)[bad], ref.bound[bad])
    return ref.rel_err(cov)


class Worst:
    """largest observed error next to the derived bound, per case family (printed with -s)"""

    def __init__(self, what):
        self.what, self.d = what, {}

    def add(self, family, err, bound):
        if err is None:
            return
        e, b = self.d.get(family, (0.0, 0.0))
        self.d[family] = (max(e, err), max(b, bound))

    def bound(self, family):
        return self.d[family][1]

    def show(self):
        print(f"\n[{self.what}] " + "; ".join(f"{k}: bound {b:.1e}, max err {e:.1e}" for k, (e, b) in sorted(self.d.items())))


def family(name):
    return name.rstrip("0123456789").split("(")[0].split("_cap")[0]


# ---- the reference itself ---------------------------------------------------------------------------------------------------
def test_reference_equals_compiled_reference_and_kat1(cov_golden):
    """H3 and cov3 of the compiled cov_func_point_to_point.h (every non-singular golden case, kat2_cap200 included) and
    SURVEY KAT-1, from the cost by automatic differentiation"""
    for c in cov_golden:
        n_h = c["P"].shape[0]
        T = T_from_colmajor(c["T_colmajor"])
        th = LIBM.atan2f(T[1], T[0])                       # the host's atan2f, as the compiled reference used
        ref = FC.censi_T(c["P"], c["Q"][:n_h], n_h, c["n_d_used"], T, c["sensor_var"], c["live_in"], theta=th)
        assert np.allclose(ref.H, c["H3"], rtol=1e-12, atol=1e-9), c["name"]
        if c["singular"]:
            continue
        assert ref.status == 0 and ref.rel_err(c["cov3"]) < 1e-9, (c["name"], ref.rel_err(c["cov3"]))
    assert any(c["name"] == "kat2_cap200" and not c["singular"] for c in cov_golden)
    P = np.array([(1.0, 0.5), (2.0, -1.0), (3.5, 0.25), (0.5, 2.0), (-1.0, 1.5)], F32)
    Q = np.array([(1.2550874948501587, 0.3773355185985565), (2.3748416900634766, -0.9903373122215271),
                  (3.7775561809539795, 0.4081680178642273), (0.5928352475166321, 1.8299250602722168),
                  (-0.8447542786598206, 1.2076728343963623)], F32)
    th = np.float32(0.1)
    ref = FC.censi_T(P, Q, 5, 5, np.array([np.cos(np.float64(th)), np.sin(np.float64(th)), 0.3, -0.2], F32))
    assert np.abs(ref.cov - [[0.004699660395, -0.001029669124, 0.000912736075],
                             [-0.001029669124, 0.005515331835, -0.001343246184],
                             [0.000912736075, -0.001343246184, 0.001190702161]]).max() < 1e-12


# ---- the oracle's closed form ------------------------------------------------------------------------------------------------
def test_oracle_cov_censi_within_the_derived_bound():
    """orc_cov_censi called directly: n_h in {0, 1, 2, 3, 31, 32, 33, 8192}, every cap edge around n = 200, clouds near
    (+-990, +-990), theta at +-pi (rot_s = +-0, +-1 ulp) and 0, an exactly singular and a near-singular Hessian"""
    worst, band = Worst("oracle cov_censi, relative to max |cov|"), []
    for name, P, Q, cap, T in cov_cases():
        n_h = min(len(P), len(Q))
        n_d = FC.cap_of(n_h, cap)
        ref = FC.censi_T(P, Q, n_h, n_d, T)
        st, cov, _ = O.cov_censi(P, Q, n_h, n_d, T)
        if ref.ambiguous:
            band.append((name, ref.sigma_min, ref.h_err, st))
        worst.add(family(name), check_cov(cov, st, ref, name), ref.rel_bound)
    worst.show()
    print("[singular band]", band)
    assert worst.d["origin"] == (0.0, 0.0) and worst.d["n"][0] >= 0            # the singular cases were asserted
    assert worst.bound("theta") < 1e-6, "no teeth"


def check_records(recs, cases, p, seeded, ulps, worst, ctx, cov_of=None):
    """every record of ``cases`` against the reference; returns how many were checked"""
    n = 0
    for (name, s, t, g), rec in zip(cases, recs):
        check_theta(rec, ulps, (ctx, name))
        ref = reference_cov(rec, s, t, g, p, seeded)
        if ref is None:
            continue
        err = check_cov(rec["cov"], rec["status"], ref, (ctx, name, p.cov_mode, p.downsample_divisor, p.outlier_mode,
                                                       p.metric, p.cov_cap))
        worst.add(family(name), err, ref.rel_bound)
        n += 1
    return n


def oracle_records(cases, p, fast):
    out = np.zeros(len(cases), RESULT_DTYPE)
    for k, (_, s, t, g) in enumerate(cases):
        r = O.run_pair(s, t, g, p, fast=fast)
        out[k] = np.frombuffer(bytes(r), RESULT_DTYPE)[0]
    return out


def test_oracle_records_within_the_derived_bound():
    """orc_run_pair (fast 0 and 1), INDEXPAIR and CORR, divisor 1 and 5, each rejector, both metrics: whole runs where
    the final pose has no exact forward tie, and lattice clouds with exact ties through max_iterations = 1"""
    worst = Worst("oracle records, relative to max |cov|")
    cases, ties = record_cases(), tie_cases()
    checked = skipped = 0
    for p in run_params():
        for fast in (0, 1):
            recs = oracle_records(cases, p, fast)
            k = check_records(recs, cases, p, False, HOST_ATAN2F_ULPS, worst, f"whole fast{fast}")
            checked, skipped = checked + k, skipped + len(cases) - k
            q = p.copy(max_iterations=1)
            check_records(oracle_records(ties, q, fast), ties, q, True, HOST_ATAN2F_ULPS, worst, f"ties fast{fast}")
    worst.show()
    print(f"[whole runs] {checked} checked, {skipped} skipped for an exact tie at the final pose")
    assert skipped <= checked // 10
    for fam in ("corridor", "loop_closure"):
        assert worst.bound(fam) < 1e-9, f"{fam}: bound {worst.bound(fam):.1e}: no teeth"


# ---- factor ----------------------------------------------------------------------------------------------------------------
def factor_cases():
    """(name, record) inputs of the factor: well-conditioned and corridor-like badly conditioned covariances, and the
    invalid ones the parameters can produce (zero / negative laser variances, cov_sensor_variance = 0) or a diagonal with
    det > 0 that is not positive definite"""
    def rec(cov, status=0, tx=0.5, ty=-0.25, theta=0.125):
        r = np.zeros(1, RESULT_DTYPE)
        r["cov"][0] = np.asarray(cov, np.float64).reshape(9)
        r["status"], r["tx"], r["ty"], r["theta"] = status, tx, ty, theta
        return r[0]
    rng = np.random.default_rng(43)
    out = [("kat1", rec([[0.004699660395, -0.001029669124, 0.000912736075], [-0.001029669124, 0.005515331835, -0.001343246184],
                         [0.000912736075, -0.001343246184, 0.001190702161]]))]
    Qm, _ = np.linalg.qr(rng.normal(size=(3, 3)))
    out.append(("weak_axis", rec(Qm @ np.diag([3e-5, 1e-5, 3e-10]) @ Qm.T, status=0x102)))  # a weak axis, kappa 1e5
    out.append(("live", rec(np.diag([0.5, 0.5, np.float64(F32(0.3))]))))
    for name, d in (("zero_var", (0.0, 0.5, 0.3)), ("neg_var", (0.5, -0.5, 0.3)), ("neg_pair", (-0.5, -0.5, 0.3))):
        out.append((name, rec(np.diag(d))))
    out.append(("zero_sensor", rec(np.zeros((3, 3)), status=0x101)))
    out.append(("indefinite", rec([[1, 2, 0], [2, 1, 0], [0, 0, 1]])))
    return out


def check_factor(f, rec, src, tgt, ctx):
    ref = FC.factor(rec["cov"])
    assert (int(f["from_node"]), int(f["to_node"])) == (tgt, src), ctx
    assert (f["tx"], f["ty"], f["theta"]) == (rec["tx"], rec["ty"], rec["theta"]), ctx
    if ref.ambiguous:
        return None
    want = int(rec["status"]) | (0 if ref.valid else FLAG_FACTOR_INVALID)
    assert int(f["status"]) == want, (ctx, hex(int(f["status"])), hex(want))
    R_got = np.asarray(f["sqrt_info"], np.float64).reshape(3, 3)
    if not ref.valid:
        assert np.array_equal(R_got, np.zeros((3, 3))) and not np.signbit(R_got).any(), ctx
        return 0.0
    assert np.all(np.tril(R_got, -1) == 0), ctx
    err = np.abs(R_got - ref.R).max()
    assert err <= ref.bound, (ctx, err, ref.bound)
    return err / np.abs(ref.R).max()


def test_oracle_factor_against_the_reference_factor():
    """orc_factor: R = chol(cov^-1)^T within the Cholesky bound scaled by kappa(cov); the invalid covariances are
    flagged, zeroed and still carry from/to, the pose and the record's status bits"""
    worst = Worst("oracle factor, relative to max |R|")
    cases = factor_cases()
    recs = np.array([r for _, r in cases], RESULT_DTYPE)
    src, tgt = np.arange(1, len(cases) + 1), np.arange(0, len(cases))
    f = O.factors(recs, src, tgt)
    for k, (name, r) in enumerate(cases):
        worst.add(name, check_factor(f[k], r, src[k], tgt[k], name), FC.factor(r["cov"]).rel_bound)
    worst.show()
    assert worst.bound("kat1") < 1e-12 and worst.bound("weak_axis") < 1e-3
    assert all(int(f["status"][k]) & FLAG_FACTOR_INVALID for k, (n, _) in enumerate(cases)
               if n in ("zero_var", "neg_var", "neg_pair", "zero_sensor", "indefinite"))


def invalid_factor_params():
    """parameters that check_params accepts and that make a record's covariance non positive definite"""
    return [Params.defaults(cov_mode=COV_REFERENCE_LIVE, laser_x_variance=0.0),
            Params.defaults(cov_mode=COV_REFERENCE_LIVE, laser_theta_variance=-0.3),
            Params.defaults(cov_mode=COV_REFERENCE_LIVE, laser_x_variance=-0.5, laser_y_variance=-0.5),
            Params.defaults(cov_mode=COV_CENSI_CORR, downsample_divisor=1, cov_sensor_variance=0.0),
            Params.defaults(cov_mode=COV_CENSI_INDEXPAIR, cov_sensor_variance=0.0)]


def test_oracle_factors_of_records_with_invalid_parameters():
    """records of whole runs under variances that are not validated (zero / negative laser variances, a zero sensor
    variance) give FLAG_FACTOR_INVALID and a zeroed sqrt_info; valid runs give the reference factor"""
    cases = record_cases()[:4]
    for p in invalid_factor_params() + [Params.defaults(cov_mode=COV_CENSI_CORR, downsample_divisor=1)]:
        recs = oracle_records(cases, p, 1)
        src, tgt = np.arange(10, 10 + len(cases)), np.arange(20, 20 + len(cases))
        f = O.factors(recs, src, tgt)
        for k in range(len(cases)):
            check_factor(f[k], recs[k], src[k], tgt[k], (cases[k][0], p.cov_mode))
        invalid = (f["status"] & FLAG_FACTOR_INVALID) != 0
        assert invalid.all() == (p.cov_sensor_variance == 0 or min(p.laser_x_variance, p.laser_theta_variance) <= 0)
