"""An independent float64 reference for the covariance of a record and the factor built from it.

The CPU oracle (``orc_cov_censi``, ``orc_factor``) and the CUDA path (``finish_cov`` + ``cov_terms``, ``factors_kernel``)
share one hand-derived closed form and one way of choosing the pairs that go into it, so comparing them with each other
cannot show that either is right.  This module restates both from their definitions.  It uses torch (automatic
differentiation) and ``f64_reference``, and never imports the oracle.

Censi covariance (DESIGN.md §3; the reference's cov_func_point_to_point.h restricted to (x, y, yaw) at z = 0)
    J(x; z) = Sum_k |R(theta) p_k + t - q_k|^2,  x = (tx, ty, theta),  z_k = (p_kx, p_ky, q_kx, q_ky).
    H = d2J_h/dx2 over the first n_h pairs and D = d2J_d/dx dz over the first n_d pairs, both by ``torch.func`` on one
    pair's cost (J is a sum, so the per-pair derivatives add up; they are summed with ``math.fsum``).
    cov = sigma^2 H^-1 D D^T H^-1 with ``np.linalg.inv`` in float64.  x and y are the record's binary32 entries widened;
    theta is a binary32 angle: the record's own ``theta`` (the same atan2f of the same (rot_s, rot_c) that the
    covariance pass used), or the binary32 rounding of the float64 atan2 for the standalone kernels.
    When n_h = 0 or H is singular the result is diag(laser variances) with FLAG_COV_SINGULAR.  "Singular" is decided
    by the smallest singular value of H against the bound on the contract's error in H (below): sigma_min = 0 is
    singular, sigma_min > that bound is not, and a case in between is ambiguous (``Cov.ambiguous``).

Pair sets (``indexpair_pairs``, ``corr_pairs``)
    CENSI_INDEXPAIR: the full (not down-sampled) clouds paired by index, n_h = min(n_src, n_tgt), n_d = min(n_h, cap)
    (cap 0: no cap).  CENSI_CORR: the down-sampled source moved by the record's (rot_c, rot_s, tx, ty) in binary32,
    one correspondence pass of ``f64_reference.pass_pairs`` at that pose (gate, reciprocity, rejector, seeded with the
    last pass's forward neighbours), the kept pairs in source order with p the UNtransformed down-sampled source point;
    the Hessian runs over all K of them and D over the first min(K, cap).

Bound on the contract's error (``Cov.bound``, per entry; first order, every constant rounded up)
    u = 2^-53, g_n = n u / (1 - n u).
    (a) angle: |dcov/dtheta| dtheta, dcov/dtheta by autodiff of the whole reference.  dtheta = 0 for records; for the
        standalone kernels dtheta = (3 + 1) ulp32(theta): the CUDA 12.9 Math API documentation bounds atan2f by 3 ulp,
        the glibc manual's table of known maximum errors bounds the host's atan2f by 1 ulp (x86_64).
    (b) the sums.  Every term of the 11 sums of the kernel (and of the oracle's H / D D^T accumulation) is a product of
        at most four factors built from p, q, t and cos/sin(theta); with m_k = |px| + |py| (>= |A|, |B|) and
        e_k = |x - qx| + |y - qy| (>= |dx|, |dy|) the terms of each H and M = D D^T entry are bounded by
            H02, H12: 2 m_k       H22: 2 m_k e_k       M00, M11: 12      M02, M12: 4 (2 e_k + m_k)
            M22: 4 (e_k^2 + 2 m_k^2)
        and their sum of magnitudes ("mag") by the sum of these.  n summands with at most 10 roundings each, in any
        summation order, are off by <= g_{n+10} mag.  cos and sin in binary64 are within 2 ulp (CUDA) and 1 ulp (host)
        of the truth, i.e. |dc|, |ds| <= 3 * 2^-52; A, B, D move by <= that times their magnitude.  Together:
            |dH|, |dM| <= (g_{n+10} + 4 * 6 u) mag.
    (c) the cofactor inverse.  First order in dH: |Hi| |dH| |Hi|.  Rounding: each cofactor (two products and a
        difference) is off by g_3 (|p1| + |p2|); det by g_3 (|a c00| + |b c01| + |c c02|) plus the cofactor errors; the
        quotient by u.  This is the kappa(H) scaling: (|a c00| + ...) / |det| is about kappa(H).
    (d) the two 3x3 products: Tm = Hi M off by |dHi| |M| + |Hi| |dM| + g_3 |Hi| |M|; cov = sigma^2 Tm Hi off by
        sigma^2 (|dTm| |Hi| + |Tm| |dHi| + g_4 |Tm| |Hi|).
    The reference's own float64 evaluation (autodiff terms, fsum, LU inverse, products) obeys the same model with
    smaller constants; (b) to (d) are doubled to cover it.  When |Hi| |dH| is not small (>= 1/4 in norm) the first-order
    bound is not valid and ``bound`` is +inf.

Factor (``factor``): R = cholesky(inv(cov)).T, upper, positive diagonal.  It is invalid when cov is not positive
    definite: eigvalsh(cov) has a value <= 0 that is exactly 0 or below -margin, margin = 16 u ||cov||_2 (ambiguous when
    0 < |lambda_min| <= margin).  Bound: the cofactor inverse as in (c) with an exact input, then the Cholesky backward
    error |dI| <= g_4 |R^T| |R|; the factor of I + dI moves by ||dR|| <= ||R||_2 kappa_2(cov) ||dI||_F / ||I||_2 to
    first order (Sun's perturbation bound without its 1/sqrt 2), doubled for the reference's own factorisation.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch
from torch.func import hessian, jacrev, vmap

import f64_reference as R

F32 = np.float32
U = 2.0 ** -53
FLAG_COV_SINGULAR = 0x200
CS_ERR = 6 * U                     # |d cos|, |d sin|: 2 ulp (CUDA binary64 cos/sin) + 1 ulp (host), ulp <= 2^-52
ATAN2F_ULPS = 3 + 1                # CUDA atan2f (3 ulp) + glibc atan2f (1 ulp)


def gamma(n: int) -> float:
    return n * U / (1.0 - n * U)


# ---- the planar cost and its derivatives ----------------------------------------------------------------------------
def _pair_cost(x, z):
    c, s = torch.cos(x[2]), torch.sin(x[2])
    rx = c * z[0] - s * z[1] + x[0] - z[2]
    ry = s * z[0] + c * z[1] + x[1] - z[3]
    return rx * rx + ry * ry


_HESS = vmap(hessian(_pair_cost, argnums=0), in_dims=(None, 0))                        # (n, 3, 3)
_MIXED = vmap(jacrev(jacrev(_pair_cost, argnums=0), argnums=1), in_dims=(None, 0))      # (n, 3, 4)


def _fsum_rows(t: np.ndarray) -> np.ndarray:
    """correctly rounded sum over axis 0 of an (n, 3, 3) array"""
    out = np.zeros((3, 3))
    if len(t):
        for i in range(3):
            for j in range(3):
                out[i, j] = math.fsum(t[:, i, j])
    return out


def _H_M(P, Q, n_h, n_d, x, y, theta):
    z = torch.from_numpy(np.concatenate([np.asarray(P, np.float64).reshape(-1, 2), np.asarray(Q, np.float64).reshape(-1, 2)], 1))
    xt = torch.tensor([x, y, theta], dtype=torch.float64)
    H = _fsum_rows(_HESS(xt, z[:n_h]).numpy()) if n_h else np.zeros((3, 3))
    if n_d:
        Dk = _MIXED(xt, z[:n_d])
        M = _fsum_rows((Dk @ Dk.transpose(1, 2)).numpy())
    else:
        M = np.zeros((3, 3))
    return H, M


def _cov_of_theta(P, Q, n_h, n_d, x, y, sensor_var):
    """cov as a differentiable function of theta (for term (a))"""
    z = torch.from_numpy(np.concatenate([np.asarray(P, np.float64).reshape(-1, 2), np.asarray(Q, np.float64).reshape(-1, 2)], 1))

    def f(th):
        xt = torch.stack([torch.tensor(x, dtype=torch.float64), torch.tensor(y, dtype=torch.float64), th])
        H = _HESS(xt, z[:n_h]).sum(0)
        Dk = _MIXED(xt, z[:n_d])
        M = (Dk @ Dk.transpose(1, 2)).sum(0)
        Hi = torch.linalg.inv(H)
        return sensor_var * Hi @ M @ Hi
    return f


# ---- error model ------------------------------------------------------------------------------------------------------
def _magnitudes(P, Q, n_h, n_d, x, y):
    P = np.asarray(P, np.float64).reshape(-1, 2)
    Q = np.asarray(Q, np.float64).reshape(-1, 2)
    m = np.abs(P).sum(1)
    e = np.abs(x - Q[:, 0]) + np.abs(y - Q[:, 1])
    mh, eh, md, ed = m[:n_h], e[:n_h], m[:n_d], e[:n_d]
    magH = np.zeros((3, 3))
    magH[0, 0] = magH[1, 1] = 2.0 * n_h
    magH[0, 2] = magH[2, 0] = magH[1, 2] = magH[2, 1] = 2.0 * mh.sum()
    magH[2, 2] = 2.0 * (mh * eh).sum()
    magM = np.zeros((3, 3))
    magM[0, 0] = magM[1, 1] = 12.0 * n_d
    magM[0, 2] = magM[2, 0] = magM[1, 2] = magM[2, 1] = 4.0 * (2 * ed + md).sum()
    magM[2, 2] = 4.0 * (ed * ed + 2 * md * md).sum()
    return magH, magM


def _cofactor_inverse_error(A):
    """rounding error of the contract's cofactor inverse of symmetric A (exact input): entrywise bound"""
    a, b, c, d, e, f = A[0, 0], A[0, 1], A[0, 2], A[1, 1], A[1, 2], A[2, 2]
    cof = np.array([[d * f - e * e, c * e - b * f, b * e - c * d],
                    [c * e - b * f, a * f - c * c, b * c - a * e],
                    [b * e - c * d, b * c - a * e, a * d - b * b]])
    cabs = np.array([[abs(d * f) + e * e, abs(c * e) + abs(b * f), abs(b * e) + abs(c * d)],
                     [abs(c * e) + abs(b * f), abs(a * f) + c * c, abs(b * c) + abs(a * e)],
                     [abs(b * e) + abs(c * d), abs(b * c) + abs(a * e), abs(a * d) + b * b]])
    dcof = gamma(3) * cabs
    det = a * cof[0, 0] + b * cof[0, 1] + c * cof[0, 2]
    ddet = (gamma(3) * (abs(a * cof[0, 0]) + abs(b * cof[0, 1]) + abs(c * cof[0, 2]))
            + abs(a) * dcof[0, 0] + abs(b) * dcof[0, 1] + abs(c) * dcof[0, 2])
    if det == 0:
        return np.full((3, 3), np.inf)
    return np.abs(cof) * ddet / det ** 2 + dcof / abs(det) + U * np.abs(cof / det)


@dataclass
class Cov:
    status: int              # 0 or FLAG_COV_SINGULAR
    cov: np.ndarray          # (3, 3)
    bound: np.ndarray        # (3, 3) per-entry bound on |contract - reference| (0 on a singular result: exact)
    H: np.ndarray
    sigma_min: float         # smallest singular value of H
    h_err: float             # Frobenius bound on the contract's error in H
    ambiguous: bool          # 0 < sigma_min <= h_err: the flag is not asserted
    kappa: float

    @property
    def rel_bound(self) -> float:
        s = np.abs(self.cov).max()
        return float(self.bound.max() / s) if s > 0 else 0.0

    def rel_err(self, got) -> float:
        s = np.abs(self.cov).max()
        return float(np.abs(np.asarray(got).reshape(3, 3) - self.cov).max() / (s if s > 0 else 1.0))


def censi(P, Q, n_h, n_d, x, y, theta, sensor_var=0.01, live=(0.5, 0.5, 0.3), dtheta=0.0) -> Cov:
    """Censi covariance of the first n_h / n_d pairs at pose (x, y, theta) with its bound (module docstring)"""
    live = np.diag(np.asarray(live, F32).astype(np.float64))
    n = max(n_h, n_d)
    P, Q = np.asarray(P, F32).reshape(-1, 2)[:n], np.asarray(Q, F32).reshape(-1, 2)[:n]
    H, M = _H_M(P, Q, n_h, n_d, x, y, theta)
    magH, magM = _magnitudes(P, Q, n_h, n_d, x, y)
    g = gamma(n + 10) + 4 * CS_ERR
    dH, dM = 2 * g * magH, 2 * g * magM
    sv = np.linalg.svd(H, compute_uv=False) if n_h else np.zeros(3)
    smin, h_err = float(sv[-1]), float(np.linalg.norm(dH))
    singular = n_h == 0 or smin == 0.0
    ambiguous = (not singular) and smin <= h_err
    if singular or ambiguous:
        return Cov(FLAG_COV_SINGULAR, live, np.zeros((3, 3)), H, smin, h_err, ambiguous, np.inf)
    Hi = np.linalg.inv(H)
    cov = sensor_var * Hi @ M @ Hi
    aHi = np.abs(Hi)
    if np.linalg.norm(aHi @ dH, 2) >= 0.25:
        bound = np.full((3, 3), np.inf)
    else:
        dHi = aHi @ dH @ aHi + 2 * _cofactor_inverse_error(H)
        Tm = Hi @ M
        dTm = dHi @ np.abs(M) + aHi @ dM + 2 * gamma(3) * aHi @ np.abs(M)
        bound = abs(sensor_var) * (dTm @ aHi + np.abs(Tm) @ dHi + 2 * gamma(4) * np.abs(Tm) @ aHi)
        bound = bound * (1 + 1e-3)                           # second-order terms (|Hi dH| < 1/4)
        if dtheta:
            th = torch.tensor(theta, dtype=torch.float64)
            dcov = torch.func.jacfwd(_cov_of_theta(P, Q, n_h, n_d, x, y, sensor_var))(th).numpy()
            bound = bound + np.abs(dcov) * dtheta
    return Cov(0, cov, bound, H, smin, h_err, False, float(sv[0] / smin))


def theta_of(T) -> float:
    """the binary32 angle of (c, s, tx, ty) from the float64 atan2 (the standalone kernels' pose, up to atan2f's error)"""
    return float(F32(math.atan2(float(F32(T[1])), float(F32(T[0])))))


def atan2f_bound(theta: float) -> float:
    return ATAN2F_ULPS * R.ulp32(theta)


def censi_T(P, Q, n_h, n_d, T, sensor_var=0.01, live=(0.5, 0.5, 0.3), theta=None) -> Cov:
    """the standalone call shape: pose (c, s, tx, ty), angle by atan2 (term (a) with the atan2f bounds), or the given
    binary32 ``theta`` (term (a) = 0)"""
    th = theta_of(T) if theta is None else float(F32(theta))
    return censi(P, Q, n_h, n_d, float(F32(T[2])), float(F32(T[3])), th, sensor_var, live,
                 dtheta=atan2f_bound(th) if theta is None else 0.0)


# ---- pair sets ----------------------------------------------------------------------------------------------------------
def downsample(xy, divisor: int) -> np.ndarray:
    """every divisor-th point, from index 0"""
    return np.ascontiguousarray(np.asarray(xy, F32).reshape(-1, 2)[::max(1, int(divisor))])


def apply_T(T, xy) -> np.ndarray:
    """x' = ((c x) + ((-s) y)) + tx in binary32, each operation rounded"""
    c, s, tx, ty = (F32(v) for v in T)
    xy = np.asarray(xy, F32).reshape(-1, 2)
    x, y = xy[:, 0], xy[:, 1]
    return np.stack([((c * x) + ((-s) * y)) + tx, ((s * x) + (c * y)) + ty], 1).astype(F32)


def cap_of(n: int, cap: int) -> int:
    return min(n, cap) if cap > 0 else n


def indexpair_pairs(src_full, tgt_full, cap):
    """-> (P, Q, n_h, n_d): the full clouds paired by index"""
    s = np.asarray(src_full, F32).reshape(-1, 2)
    t = np.asarray(tgt_full, F32).reshape(-1, 2)
    n_h = min(len(s), len(t))
    return s[:n_h], t[:n_h], n_h, cap_of(n_h, cap)


def corr_pairs(src_ds, tgt_ds, T, r, reciprocal, mode=0, param=0.0, cap=0, prev_nn=None):
    """-> (P, Q, n_h, n_d): the correspondences at pose T in source order, P untransformed"""
    src_ds = np.asarray(src_ds, F32).reshape(-1, 2)
    tgt_ds = np.asarray(tgt_ds, F32).reshape(-1, 2)
    m = R.pass_pairs(apply_T(T, src_ds), tgt_ds, r, reciprocal, mode, param, prev_nn=prev_nn)
    keep = np.nonzero(m.corr >= 0)[0]
    K = len(keep)
    return src_ds[keep], tgt_ds[m.corr[keep]], K, cap_of(K, cap)


def forward_ties(src_t, tgt, r) -> int:
    """number of gated source points with more than one nearest target (where the seeds could matter)"""
    src_t = np.asarray(src_t, F32).reshape(-1, 2)
    tgt = np.asarray(tgt, F32).reshape(-1, 2)
    if len(src_t) == 0 or len(tgt) == 0:
        return 0
    thr = R.gate_threshold(r)
    n = 0
    step = max(1, (1 << 22) // len(tgt))
    for lo in range(0, len(src_t), step):
        dd = R._dist2(src_t[lo:lo + step], tgt)
        mn = dd.min(axis=1)
        n += int(((dd == mn[:, None]).sum(axis=1) > 1)[mn <= thr].sum())
    return n


# ---- factor ---------------------------------------------------------------------------------------------------------------
@dataclass
class Factor:
    valid: bool
    ambiguous: bool
    R: np.ndarray             # (3, 3) upper; zeros when invalid
    bound: float              # max-entry bound on |R_contract - R|

    @property
    def rel_bound(self) -> float:
        s = np.abs(self.R).max()
        return self.bound / s if s > 0 else 0.0


def factor(cov) -> Factor:
    C = np.asarray(cov, np.float64).reshape(3, 3)
    if not np.all(np.isfinite(C)):
        return Factor(False, False, np.zeros((3, 3)), 0.0)
    C = 0.5 * (C + C.T)
    lam = np.linalg.eigvalsh(C)
    margin = 16 * U * np.abs(lam).max()
    if lam[0] == 0.0 or lam[0] < -margin:
        return Factor(False, False, np.zeros((3, 3)), 0.0)
    if lam[0] <= margin:
        return Factor(False, True, np.zeros((3, 3)), np.inf)
    I = np.linalg.inv(C)
    Rm = np.linalg.cholesky(I).T
    dI = _cofactor_inverse_error(C) + gamma(4) * np.abs(Rm.T) @ np.abs(Rm)
    kappa = lam[-1] / lam[0]
    bound = 2 * np.linalg.norm(Rm, 2) * kappa * np.linalg.norm(dI) / np.linalg.norm(I, 2)
    return Factor(True, False, Rm, float(bound))
