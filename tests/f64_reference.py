"""An independent float64 reference for one ICP pass: correspondences, outlier rejectors, rigid step, mse.

The CPU oracle (``oracle/dpg_oracle.c``) and the CUDA path implement one arithmetic contract (DESIGN.md §3) and are
compared with each other bit for bit.  That cannot show that both are right: a moment sum that wraps, or a rejector rule
implemented wrongly on both sides, still matches.  This module states the same operations from their definitions with
numpy only, without the contract's implementation choices (no fixed-point sums, no closed-form Procrustes, no radix
select), and never imports the oracle.

Correspondences (brute force, chunked so that 8192 x 8192 fits in memory)
    d2 = (dx*dx) + (dy*dy) in numpy float32: every operation is rounded on its own (numpy never fuses a multiply-add),
    which is the distance of §3.  Gate: d2 <= the largest binary32 <= r^2, r^2 in binary64.  Forward neighbour: the
    lowest index among the minimisers, or the seed (``prev_nn``) when it is one of them.  Reciprocity (§3): (i, j) is
    kept iff no source point is STRICTLY closer to target j than d2(i, j).  The projective search (§5.7) is restated only
    by its bearing key and by the fact that a window W >= n covers the whole cloud: its neighbour is then the
    (d2, index)-lexicographic minimum, forward and back, so its reciprocal test keeps only the lowest-index asker of an
    exact tie (where the exact search's emptiness rule keeps every asker).

Rejectors (§5.8), over a sorted copy of the K accepted d2
    TRIMMED keeps the max(3, floor(param*K)) smallest (clamped to K) and every value tied with the last of them;
    MEDIAN keeps d2 <= the largest binary32 <= sorted[K // 2] * param (product in binary64).

Rigid step
    point-to-point: textbook Umeyama on float64 pairs (centre, 2x2 cross-covariance, ``np.linalg.svd``, reflection
    guard).  When the cross-covariance is exactly zero every rotation is optimal; the contract then takes theta = 0.
    point-to-line: the rows of §5.5 stacked and solved with ``np.linalg.lstsq`` in float64, rotation by the Cayley map
    of dtheta / 2.  mse = math.fsum(d2) / K.

Tolerance of the step (derived per case; ``p2p_bounds`` / ``p2l_bounds`` compute it)
    The contract forms a = Sum(p.q) - (Sp.Sq)/K and b = Sum(p x q) - (Sp x Sq)/K from int64 sums, then theta = atan2(b, a)
    with c = a/h, s = b/h, h = |(a, b)|.  Its error in (a, b) has three sources:
      * fixed-point quantisation: each product term is rounded to 2^-28 (error <= 2^-29; the binary64 product of two
        binary32 values is exact), each coordinate term to 2^-32 (<= 2^-33, and exactly 0 when |coord| >= 2^-9, where
        coord * 2^32 is already an integer).  Over K pairs the two product sums in a (and in b) are off by <= 2 K 2^-29;
        a coordinate sum by <= n_small 2^-33 (n_small = terms with |coord| < 2^-9), which enters (Sp.Sq)/K at most as
        (|mean p| + |mean q|) n_small 2^-33;
      * the binary64 rounding of (double)red[k] and of the closed form: <= 2^-53 per operation, relative to the
        magnitude of its operand; bounded by 8 * 2^-53 * (Sum |p||q| + K |mean p||mean q|), which is what makes far-
        from-origin clouds (where Sum p.q - Sp.Sq/K cancels heavily) the hard case.
    With eps_ab the sum of these bounds for |da| + |db|, the angle moves by dtheta <= asin(eps_ab / h) (<= eps_ab / h to
    first order).  Then, with the final rounding to binary32 and the binary64 evaluation of t = mean q - R mean p:
        |dc|, |ds| <= 2^-24 + dtheta
        |dt|       <= ulp32(t) + (|mean p| + 1) dtheta + 8 * 2^-53 (|mean p| + |mean q|)
        |dmse|     <= 2^-41 + 4 * 2^-53 * mse            (2^40 quantisation of d2, then two binary64 roundings)
    The reference's own float64 error (centred data, one SVD) is far below these and is covered by a 2^-46 slack on
    dtheta.  For point-to-line the nine normal-equation sums carry the same quantisation (K 2^-29 each, plus the binary64
    rounding of each term); the solution delta = A^-1 b moves by
        |d delta| <= ||A^-1|| (||dA|| |delta| + ||db||) / (1 - ||A^-1|| ||dA||)
    with ||dA|| including the backward error of a 3x3 Cholesky in binary64 (<= 30 * 2^-53 ||A||); the Cayley map has
    slope <= 1, so |dc|, |ds| <= 2^-24 + |d delta| and |dt| <= ulp32(t) + |d delta|.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

F32 = np.float32
U53 = 2.0 ** -53
_CHUNK_ELEMS = 1 << 22          # distance-matrix elements per chunk (16 MB of float32)


def f32_floor(x: float) -> np.float32:
    """largest binary32 <= x (x a binary64 value)"""
    f = F32(x)
    if float(f) > x:
        f = np.nextafter(f, F32(-np.inf))
    return F32(f)


def gate_threshold(r: float) -> np.float32:
    return f32_floor(float(r) * float(r))


def ulp32(x) -> float:
    x = abs(float(x))
    return float(np.spacing(F32(x))) if x > 0 else float(np.spacing(F32(0)))


def beam_key(px, py, ox, oy) -> np.ndarray:
    """§5.7 bearing key of p seen from (ox, oy): monotone in atan2 on (-pi, pi], binary32, no libm"""
    vx = np.asarray(px, F32) - F32(ox)
    vy = np.asarray(py, F32) - F32(oy)
    a = np.abs(vx) + np.abs(vy)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = np.where(a > 0, vy / np.where(a > 0, a, F32(1)), F32(0)).astype(F32)
    return np.where(vx >= 0, t, np.where(vy >= 0, F32(2) - t, F32(-2) - t)).astype(F32)


def _dist2(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """(len(a), len(b)) binary32 squared distances, each operation rounded (no FMA)"""
    dx = a[:, None, 0] - b[None, :, 0]
    dy = a[:, None, 1] - b[None, :, 1]
    return (dx * dx) + (dy * dy)


@dataclass
class Matches:
    corr: np.ndarray      # int32 target index per source point, -1 = not accepted
    d2: np.ndarray        # binary32 forward minimum distance per source point (+inf for an empty target)
    fwd: np.ndarray       # bool: the forward neighbour passed the gate
    nn: np.ndarray        # int32 gated forward neighbour per source point (the next pass's seed), -1 = none

    @property
    def k(self) -> int:
        return int((self.corr >= 0).sum())


def correspondences(src, tgt, r: float, reciprocal: bool, prev_nn=None, projective_full: bool = False) -> Matches:
    """One correspondence pass, brute force.  ``projective_full`` is the projective search with a window covering the
    whole cloud (lowest-index neighbour both ways, no seeds)."""
    src = np.ascontiguousarray(src, F32).reshape(-1, 2)
    tgt = np.ascontiguousarray(tgt, F32).reshape(-1, 2)
    ns, nt = len(src), len(tgt)
    corr = np.full(ns, -1, np.int32)
    nn = np.full(ns, -1, np.int32)
    if ns == 0 or nt == 0:
        return Matches(corr, np.full(ns, np.inf, F32), np.zeros(ns, bool), nn)
    thr = gate_threshold(r)
    dmin = np.empty(ns, F32)
    jmin = np.empty(ns, np.int64)
    colmin = np.full(nt, np.inf, F32)
    colarg = np.zeros(nt, np.int64)
    seed = None if prev_nn is None else np.asarray(prev_nn, np.int64)
    step = max(1, _CHUNK_ELEMS // nt)
    for lo in range(0, ns, step):
        hi = min(ns, lo + step)
        dd = _dist2(src[lo:hi], tgt)
        j = dd.argmin(axis=1)                                   # first minimiser = lowest index
        dmin[lo:hi] = dd[np.arange(hi - lo), j]
        if seed is not None:
            s = seed[lo:hi]
            ok = (s >= 0) & (s < nt)
            ds = np.full(hi - lo, np.inf, F32)
            ds[ok] = dd[np.nonzero(ok)[0], s[ok]]
            j = np.where(ok & (ds == dmin[lo:hi]), s, j)
        jmin[lo:hi] = j
        cm, ca = dd.min(axis=0), dd.argmin(axis=0) + lo
        better = cm < colmin                                    # strict: an earlier chunk keeps the lower index
        colarg[better] = ca[better]
        colmin = np.minimum(colmin, cm)
    fwd = dmin <= thr
    nn[fwd] = jmin[fwd]
    keep = fwd.copy()
    if reciprocal:
        if projective_full:
            keep &= colarg[jmin] == np.arange(ns)
        else:
            keep &= ~(colmin[jmin] < dmin)
    corr[keep] = jmin[keep]
    return Matches(corr, dmin, fwd, nn)


def reject(d2_accepted, mode: int, param: float) -> float:
    """Threshold tau of a rejector over the accepted d2 (mode 1 = TRIMMED, 2 = MEDIAN; +inf for none / K = 0)."""
    v = np.sort(np.asarray(d2_accepted, F32))
    K = len(v)
    if mode == 0 or K == 0:
        return float("inf")
    if mode == 1:
        keep = min(K, max(3, math.floor(float(param) * K)))
        return float(v[keep - 1])
    return float(f32_floor(float(v[K // 2]) * float(param)))


def apply_rejector(m: Matches, mode: int, param: float) -> Matches:
    acc = m.corr >= 0
    tau = reject(m.d2[acc], mode, param)
    corr = np.where(acc & (m.d2.astype(np.float64) <= tau), m.corr, -1).astype(np.int32)
    return Matches(corr, m.d2, m.fwd, m.nn)


def pass_pairs(src, tgt, r, reciprocal, mode=0, param=0.0, prev_nn=None, projective_full=False) -> Matches:
    return apply_rejector(correspondences(src, tgt, r, reciprocal, prev_nn, projective_full), mode, param)


# ---- rigid step ------------------------------------------------------------------------------------------------
def step_p2p(p, q):
    """Umeyama on float64 pairs -> (c, s, tx, ty) in float64"""
    p = np.asarray(p, np.float64)
    q = np.asarray(q, np.float64)
    mp, mq = p.mean(axis=0), q.mean(axis=0)
    H = (q - mq).T @ (p - mp)                    # Sum q_c p_c^T: R = argmax tr(R^T H)
    if not H.any():
        R = np.eye(2)
    else:
        U, _, Vt = np.linalg.svd(H)
        R = U @ np.diag([1.0, np.sign(np.linalg.det(U @ Vt))]) @ Vt
    t = mq - R @ mp
    return float(R[0, 0]), float(R[1, 0]), float(t[0]), float(t[1])


def p2l_rows(p, tgt, j, gate):
    """§5.5 rows of the accepted pairs: p (K,2) current source points, j (K,) target indices -> J (M,3), r (M,)"""
    tgt = np.asarray(tgt, F32)
    nt = len(tgt)
    J, R = [], []
    for (pxf, pyf), jj in zip(np.asarray(p, F32), np.asarray(j)):
        q = tgt[jj]
        cand = [c for c in (jj - 1, jj + 1) if 0 <= c < nt]
        j2 = -1
        if cand:
            d = [(_dist2(np.array([[pxf, pyf]], F32), tgt[c:c + 1])[0, 0], c) for c in cand]
            j2 = d[0][1] if len(d) == 1 or not d[1][0] < d[0][0] else d[1][1]
        px, py = float(pxf), float(pyf)
        ex, ey = px - float(q[0]), py - float(q[1])
        seg = _dist2(tgt[j2:j2 + 1], q[None])[0, 0] if j2 >= 0 else F32(0)
        if j2 >= 0 and F32(0) < seg <= F32(gate):
            tx, ty = float(tgt[j2, 0]) - float(q[0]), float(tgt[j2, 1]) - float(q[1])
            ln = math.hypot(tx, ty)
            nx, ny = -ty / ln, tx / ln
            J.append((nx, ny, ny * px - nx * py))
            R.append(nx * ex + ny * ey)
        else:
            J += [(1.0, 0.0, -py), (0.0, 1.0, px)]
            R += [ex, ey]
    return np.array(J, np.float64).reshape(-1, 3), np.array(R, np.float64)


def step_p2l(J, r):
    delta = np.linalg.lstsq(J, -r, rcond=None)[0]
    u = 0.5 * delta[2]
    den = 1.0 + u * u
    return (1.0 - u * u) / den, 2.0 * u / den, float(delta[0]), float(delta[1])


def mse(d2_kept) -> float:
    d = np.asarray(d2_kept, F32).astype(np.float64)
    return math.fsum(d) / len(d)


# ---- tolerances --------------------------------------------------------------------------------------------------
@dataclass
class Bounds:
    cs: float      # |dc|, |ds|
    tx: float
    ty: float
    mse: float
    dtheta: float

    @property
    def pose(self) -> float:
        return max(self.tx, self.ty)


def mse_bound(m: float) -> float:
    return 2.0 ** -41 + 4 * U53 * m


def p2p_bounds(p, q, step, m: float) -> Bounds:
    p = np.asarray(p, np.float64)
    q = np.asarray(q, np.float64)
    K = len(p)
    mp, mq = p.mean(axis=0), q.mean(axis=0)
    pc, qc = p - mp, q - mq
    a = float((pc * qc).sum())
    b = float((pc[:, 0] * qc[:, 1] - pc[:, 1] * qc[:, 0]).sum())
    h = math.hypot(a, b)
    sum_pq = float((np.abs(p).sum(axis=1) * np.abs(q).sum(axis=1)).sum())
    nmp, nmq = float(np.abs(mp).sum()), float(np.abs(mq).sum())
    n_small = int((np.abs(p) < 2.0 ** -9).sum() + (np.abs(q) < 2.0 ** -9).sum())
    quant = 2 * (2 * K * 2.0 ** -29) + 2 * (nmp + nmq) * n_small * 2.0 ** -33
    rnd = 2 * 8 * U53 * (sum_pq + K * nmp * nmq)
    eps_ab = quant + rnd
    # h = 0: every rotation is optimal and both sides take theta = 0 (the caller checks c = 1, s = 0 exactly)
    dth = (math.asin(min(1.0, eps_ab / h)) if h > 0 else 0.0) + 2.0 ** -46
    base = (nmp + 1.0) * dth + 8 * U53 * (nmp + nmq)
    return Bounds(2.0 ** -24 + dth, ulp32(step[2]) + base, ulp32(step[3]) + base, mse_bound(m), dth)


def p2l_bounds(J, r, step, m: float) -> Bounds:
    K = len(r)                                            # rows >= pairs: a safe count of terms per sum
    A = J.T @ J
    b = -(J.T @ r)
    terms_A = np.abs(J).T @ np.abs(J)
    terms_b = np.abs(J).T @ np.abs(r)
    dA = np.sqrt(((K * 2.0 ** -29 + 4 * U53 * terms_A) ** 2).sum()) + 30 * U53 * np.linalg.norm(A)
    db = np.sqrt(((K * 2.0 ** -29 + 4 * U53 * terms_b) ** 2).sum())
    inv = np.linalg.norm(np.linalg.inv(A), 2)
    delta = np.linalg.solve(A, b)
    den = 1.0 - inv * dA
    dd = (inv * (dA * np.linalg.norm(delta) + db) / den if den > 0 else np.inf) + 2.0 ** -46
    return Bounds(2.0 ** -24 + dd, ulp32(step[2]) + dd, ulp32(step[3]) + dd, mse_bound(m), dd)
