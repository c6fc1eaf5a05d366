"""GPU (B200): the CUDA path against the independent float64 reference (tests/f64_reference.py), not the oracle.  The
correspondence hook for every search, the outlier rejectors at their edges (hook and records), one pass of the stock
and general kernels within the bound derived from the arithmetic contract, and the int64 moment sums at the parameter
limits.  Plus two oracle-backed checks the reference cannot make (whole runs with a rejector under forced stage chains)
and one with no oracle at all (TRIMMED 1.0 keeps every pair, so its records equal the rejector-off records)."""
import numpy as np
import pytest

from dpg_slam_b200 import synth
from dpg_slam_b200._abi import (COV_CENSI_CORR, METRIC_POINT_TO_LINE, OUTLIER_MEDIAN, OUTLIER_TRIMMED, SEARCH_BRUTE,
                                SEARCH_PROJECTIVE, SEARCH_PRUNED, STOP_MASK, STOP_NO_CORRESPONDENCES, Params)
from dpg_slam_b200.scanmatch import ScanMatcher
from oracle import oracle_py as O
from test_gpu_parity import assert_records_match
from test_independent_reference import (F32, check_step, corr_cases, lattice_case, params_for, reference_pass,
                                        reference_step, rejector_cases, ring_case, step_cases)

pytestmark = pytest.mark.gpu
IDENT = np.array([1, 0, 0, 0], F32)
SEARCHES = [SEARCH_BRUTE, SEARCH_PRUNED, SEARCH_PROJECTIVE]
MAX_WINDOW = 1024          # the largest projective window: W >= n needs clouds of at most 1024 points


def store_of(clouds):
    off = np.zeros(len(clouds) + 1, np.int64)
    off[1:] = np.cumsum([len(c) for c in clouds])
    return np.concatenate(clouds).astype(F32), off


def one_pass_records(sm, cases, p):
    """records of one pass per (src, tgt) case from the identity guess, through submit_pairs"""
    pts, off = store_of([c for s, t in cases for c in (s, t)])
    sm.upload_scans(pts, off)
    n = len(cases)
    return sm.submit_pairs(np.arange(0, 2 * n, 2), np.arange(1, 2 * n, 2), np.zeros((n, 3), F32), p), pts, off


# ---- correspondences -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("reciprocal", [1, 0])
@pytest.mark.parametrize("search", SEARCHES)
def test_hook_correspondences_equal_reference(gpu_matcher, search, reciprocal):
    """corridor scans, 8192-point clouds near (+-990, +-990) (exact searches only: W >= n needs n <= 1024), lattice
    clouds with ties and seeds (exact searches; the projective search has no seeds), n in {1, 2, 3, 31, 32, 33}"""
    for name, src, tgt, seed, r in corr_cases():
        p = params_for(search=search, reciprocal=reciprocal, r=r, window=MAX_WINDOW)
        if search == SEARCH_PROJECTIVE:
            if len(src) > 4 * MAX_WINDOW:
                continue
            src, tgt, seed = src[:MAX_WINDOW], tgt[:MAX_WINDOW], None
        want = reference_pass(src, tgt, p, prev_nn=seed)
        if seed is None:
            got, d2 = gpu_matcher.correspondences(src, tgt, IDENT, p)
        else:
            got, d2, nn = gpu_matcher.correspondences_seeded(src, tgt, IDENT, p, seed)
            assert np.array_equal(nn, want.nn), name
        assert np.array_equal(got, want.corr), (name, np.nonzero(got != want.corr)[0][:5])
        assert np.array_equal(d2[want.fwd].view(np.uint32), want.d2[want.fwd].view(np.uint32)), name


# ---- rejectors -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("search", SEARCHES)
def test_rejector_edges_equal_reference(gpu_matcher, search):
    """Every rejector edge (K in {1, 2, 3, 4}, ties at the threshold, d2 = 0, median * factor on / just off a binary32
    value, param * K an exact integer, the max(3, .) clamp, tiles of 31 / 32 / 33, low-byte differences): the hook's kept
    set, and the n_correspondences of a one-pass record (the kept K; the pass stops on K < 3), equal the reference's."""
    cases = rejector_cases()
    for rec in (1, 0):
        for name, src, tgt, mode, param in cases:
            p = params_for(search=search, reciprocal=rec, mode=mode, param=param, window=MAX_WINDOW)
            want = reference_pass(src, tgt, p)
            got, _ = gpu_matcher.correspondences(src, tgt, IDENT, p)
            assert np.array_equal(got, want.corr), (name, mode, param, rec)
        for mode, param in sorted({(c[3], c[4]) for c in cases}):
            group = [c for c in cases if (c[3], c[4]) == (mode, param)]
            p = params_for(search=search, reciprocal=rec, mode=mode, param=param, window=MAX_WINDOW, max_iterations=1)
            recs, _, _ = one_pass_records(gpu_matcher, [(c[1], c[2]) for c in group], p)
            for (name, src, tgt, _, _), r in zip(group, recs):
                k = reference_pass(src, tgt, p).k
                assert int(r["n_correspondences"]) == k, (name, mode, param, rec, int(r["n_correspondences"]), k)
                assert (int(r["status"]) & STOP_MASK == STOP_NO_CORRESPONDENCES) == (k < 3), name


def test_rejector_whole_runs_under_forced_chains_equal_oracle(gpu_matcher, monkeypatch):
    """A rejector with the sticky tie rule over whole runs (lattice / duplicate clouds, lattice-aligned guesses) and on
    corridor pairs, under forced stage chains: 1-warp and 32-warp CTAs, and chains that ask for a cluster stage, which
    the host drops because the rejector's select is block-wide.  Every record equals the oracle's."""
    rng = np.random.default_rng(321)
    clouds = []
    for k in range(24):
        s, _ = lattice_case(rng, 8, int(rng.integers(20, 300)), dup=k % 3 == 0)
        clouds.append((s + (rng.integers(-2, 3, 2) * 0.125 if k % 2 else rng.normal(0, 0.05, 2))).astype(F32))
    n_lat = len(clouds)
    wl = synth.config_corridor(n_pairs=16, seed=44)
    cpts, coff = O.clouds_from_ranges(wl.ranges, wl.scanner)
    clouds += [cpts[coff[k]:coff[k + 1]] for k in range(wl.n_scans)]
    pts, off = store_of(clouds)
    src = np.concatenate([rng.integers(0, n_lat, 120), wl.src_idx + n_lat]).astype(np.int32)
    tgt = np.concatenate([rng.integers(0, n_lat, 120), wl.tgt_idx + n_lat]).astype(np.int32)
    guess = np.zeros((len(src), 3), F32)
    guess[:120, :2] = rng.integers(-1, 2, (120, 2)) * 0.125
    guess[120:] = wl.guess
    runs = [Params.defaults(downsample_divisor=1, search=SEARCH_PRUNED, cov_mode=COV_CENSI_CORR, max_iterations=60,
                            outlier_mode=m, outlier_param=q) for m, q in ((OUTLIER_TRIMMED, 0.8), (OUTLIER_MEDIAN, 0.5), (OUTLIER_MEDIAN, 1.5))]
    refs = [O.run_batch(pts, off, src, tgt, guess, p, fast=1, threads=0)[0] for p in runs]
    for stages, warps, chain in ((1, 1, None), (1, 32, None), (2, 0, "1,32"), (4, 0, "4,8,16,9x4"), (2, 0, "2,5x2")):
        monkeypatch.setenv("DPGICP_STAGES", str(stages))
        monkeypatch.setenv("DPGICP_WARPS", str(warps))
        if chain:
            monkeypatch.setenv("DPGICP_CHAIN", chain)
        else:
            monkeypatch.delenv("DPGICP_CHAIN", raising=False)
        with ScanMatcher(0) as sm:
            sm.upload_scans(pts, off)
            for p, ref in zip(runs, refs):
                got = sm.submit_pairs(src, tgt, guess, p)
                assert_records_match(got, ref, f"chain {stages}/{warps}/{chain} outlier {p.outlier_mode}/{p.outlier_param}")


# ---- one pass against the float64 step -----------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", [0, METRIC_POINT_TO_LINE])
def test_one_pass_within_the_derived_bound_of_the_float64_step(gpu_matcher, metric):
    """max_iterations = 1 from a theta = 0 guess: the record pose is the step.  PRUNED point-to-point with no rejector runs
    the stock instantiations, so this pins them against a reference that is not the oracle; point-to-line runs the
    general ones.  Corridor and loop-closure scans, far-from-origin clouds, K = 3, and (point-to-point) the symmetric
    h = 0 case, where the step must be the pure translation."""
    worst = {}
    for reciprocal in (1, 0):
        cases = [c for c in step_cases() if (c[0] == "h0") == (reciprocal == 0) and not (metric and c[0] == "h0")]
        if not cases:
            continue
        p = params_for(search=SEARCH_PRUNED, reciprocal=reciprocal, metric=metric, max_iterations=1)
        recs, pts, off = one_pass_records(gpu_matcher, [(s, t) for _, s, t in cases], p)
        n = len(cases)
        ref, _ = O.run_batch(pts, off, np.arange(0, 2 * n, 2), np.arange(1, 2 * n, 2), np.zeros((n, 3), F32), p, fast=0)
        assert_records_match(recs, ref, f"one pass metric {metric}")
        for (name, src, tgt), r in zip(cases, recs):
            K, st, mse, b = reference_step(src, tgt, p)
            err = check_step(r, K, st, mse, b, (name, metric))
            if name == "corridor":
                assert b.pose < 1e-6, f"pose bound {b.pose:.2e} m on a corridor pair: no teeth"
            if name == "h0":
                assert (float(r["rot_c"]), float(r["rot_s"])) == (1.0, 0.0)
            w = worst.setdefault(name, [0.0, 0.0, 0.0])
            w[0] = max(w[0], b.pose)
            w[1] = max(w[1], abs(float(r["tx"]) - st[2]), abs(float(r["ty"]) - st[3]))
            w[2] = max(w[2], err["mse"])
    print("\n[one pass, GPU] metric", metric, {k: f"bound {v[0]:.2e} m, max |dt| {v[1]:.2e} m, mse err/bound {v[2]:.2f}" for k, v in worst.items()})


@pytest.mark.parametrize("metric", [0, METRIC_POINT_TO_LINE])
def test_moment_sums_fit_at_the_parameter_limits(gpu_matcher, metric):
    """8192 source points on a 29.99 m ring around a target cluster at (970, 970), no reciprocity, 30 m gate: all 8192
    pairs accepted at d2 ~ 899, Sum d2 2^40 ~ 0.88 * 2^63 (point-to-line: one repeated target point, so every pair gives
    the isolated-point rows and Sum (px^2 + py^2) 2^28 ~ 4.4e18).  One pass within the derived bound, mse within the bound
    of fsum; one pass and a longer run equal to the oracle."""
    src, tgt = ring_case(duplicates=metric == METRIC_POINT_TO_LINE)
    for search in (SEARCH_BRUTE, SEARCH_PRUNED):
        p = params_for(search=search, reciprocal=0, r=30.0, metric=metric, max_iterations=1)
        K, st, mse, b = reference_step(src, tgt, p)
        assert K == 8192
        recs, pts, off = one_pass_records(gpu_matcher, [(src, tgt)], p)
        check_step(recs[0], K, st, mse, b, ("limit", metric, search))
        for q in (p, p.copy(max_iterations=8, cov_mode=COV_CENSI_CORR)):
            got = gpu_matcher.submit_pairs([0], [1], np.zeros((1, 3), F32), q)
            ref, _ = O.run_batch(pts, off, [0], [1], np.zeros((1, 3), F32), q, fast=0)
            assert_records_match(got, ref, f"limit metric {metric} search {search} iterations {q.max_iterations}")


# ---- stock against general, no oracle ------------------------------------------------------------------------------------
def test_trimmed_one_equals_rejector_off_on_bench_batches(gpu_matcher):
    """TRIMMED 1.0 keeps every pair for every K, and forces the general instantiation with no cluster stage; the
    rejector-off batch runs the stock kernels and the cluster stage.  The records must be the same bits: on the bench's
    corridor batch (5000 pairs x 1081 beams) and on a 2000-pair loop-closure batch."""
    p = Params.defaults(downsample_divisor=1, cov_mode=COV_CENSI_CORR)
    for wl in (synth.config_corridor(n_pairs=5000, n_beams=1081, seed=2), synth.config_loop_closure(n_pairs=2000, n_scans=200, seed=3)):
        gpu_matcher.upload_ranges(wl.ranges, wl.scanner)
        off = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p)
        on = gpu_matcher.submit_pairs(wl.src_idx, wl.tgt_idx, wl.guess, p.copy(outlier_mode=OUTLIER_TRIMMED, outlier_param=1.0))
        bad = [f for f in on.dtype.names if on[f].tobytes() != off[f].tobytes()]
        assert not bad, (wl.name, bad)
