"""Independent reference of candidate-pair enumeration and of the pair guesses.

numpy, scipy and the C library only: this module imports neither ``oracle/`` nor ``dpg_slam_b200/``.  It is written
from the reference's loops as ``include/dpgicp.h`` and DESIGN §5.4 state them.

Reoptimize (dpg_slam.cc:79-107): for i = 1 .. n-1, first (i, i-1), then every j < i-1 in ascending order that passes
the gate.  Online (dpg_slam.cc:255-300): (n-1, n-2), then every j <= n-4 in ascending order gated against node n-2,
emitted as (n-2, j).  Pairs are (src, tgt); shard `rank` of `world` is ``global[rank::world]``.

Gate: binary32 throughout, every operation rounded: dx = x_j - x_i, dy = y_j - y_i, dist = sqrt(dx*dx + dy*dy) and
``dist <= (pass_j == pass_i ? r_same : r_other)``.  numpy float32 arrays evaluate exactly that (no fusion; float32
``np.sqrt`` is correctly rounded).  For large n the candidates come from ``cKDTree.query_pairs`` at a widened radius
(see ``_kd_radius``) and the exact gate is applied to them; brute force covers small n and checks the prefilter.

Guess of pair (src, tgt), math_utils.cc:20-34 with node_1 = tgt, node_2 = src: t = p2 - p1 in binary32,
(tx, ty) = Rotation2Df(-theta_1) t with cosf / sinf from libm (through ctypes: numpy's float32 cos is not glibc's
cosf), each product and sum rounded.  Angle: AngleMod in binary64, g = d - 2 pi rint(d / 2 pi) with
d = (double)(float)(theta_2 - theta_1), rounded to binary32.  The matrix entries are c = (float)cos(g),
s = (float)sin(g) in binary64 libm (``math.cos`` / ``math.sin``).

Boundary predicate: a binary64 value whose low 29 bits are within +-32 of 2^28 sits next to the midpoint of two
adjacent binary32 values; two libm implementations with sub-ulp errors may round it to different binary32 values.
``boundary_angles`` finds binary32 angles whose libm cos or sin meets it.
"""
import ctypes
import math

import numpy as np
from scipy.spatial import cKDTree

F32 = np.float32
TWO_PI = 6.283185307179586                     # M_PI * 2.0 in binary64

_libm = ctypes.CDLL("libm.so.6")
_libm.cosf.argtypes = [ctypes.c_float]
_libm.cosf.restype = ctypes.c_float
_libm.sinf.argtypes = [ctypes.c_float]
_libm.sinf.restype = ctypes.c_float


def cosf(x):
    return F32(_libm.cosf(float(x)))


def sinf(x):
    return F32(_libm.sinf(float(x)))


# ---- gate ---------------------------------------------------------------------------------------------------------
def gate(xj, yj, pj, xi, yi, pi, r_same, r_other):
    """the reference's float gate, elementwise over numpy arrays (all broadcast)"""
    dx = np.subtract(np.asarray(xj, F32), np.asarray(xi, F32), dtype=F32)
    dy = np.subtract(np.asarray(yj, F32), np.asarray(yi, F32), dtype=F32)
    with np.errstate(over="ignore"):
        d2 = np.add(np.multiply(dx, dx, dtype=F32), np.multiply(dy, dy, dtype=F32), dtype=F32)
    dist = np.sqrt(d2, dtype=F32)
    thr = np.where(np.asarray(pj) == np.asarray(pi), F32(r_same), F32(r_other)).astype(F32)
    return dist <= thr


def gate_distance(a, b):
    """binary32 distance of the gate between two points (x, y)"""
    dx, dy = F32(F32(b[0]) - F32(a[0])), F32(F32(b[1]) - F32(a[1]))
    with np.errstate(over="ignore"):
        return F32(np.sqrt(F32(F32(dx * dx) + F32(dy * dy))))


def _kd_radius(r):
    """A radius that holds every pair the binary32 gate can pass at radius r.  In the normal range the gate's distance
    is the real one times (1 + e), |e| <= 3 * 2^-24 (two roundings inside the square, one sum, one root); underflow of
    dx*dx or dy*dy shrinks it by at most sqrt(2 * 2^-149) < 1e-22 absolute; overflow only makes it larger.  The KD-tree
    works in binary64 on the exact binary32 coordinates.  2^-16 relative + 1e-20 absolute covers all of it."""
    return float(r) * (1.0 + 2.0 ** -16) + 1e-20


def _gated_pairs_brute(xy, passes, r_same, r_other, query, jmax_of):
    """(i, j) with j < jmax_of(i) passing the gate against node i, for every i in `query`; row-blocked brute force"""
    x, y = xy[:, 0], xy[:, 1]
    out_i, out_j = [], []
    query = np.asarray(query, np.int64)
    block = max(1, (1 << 22) // max(len(xy), 1))
    for b0 in range(0, len(query), block):
        qi = query[b0:b0 + block]
        jm = jmax_of(qi)
        w = int(jm.max()) if len(jm) else 0
        if w <= 0:
            continue
        j = np.arange(w)
        ok = gate(x[None, :w], y[None, :w], passes[None, :w], x[qi, None], y[qi, None], passes[qi, None], r_same, r_other)
        ok &= j[None, :] < jm[:, None]
        r, c = np.nonzero(ok)
        out_i.append(qi[r])
        out_j.append(c.astype(np.int64))
    if not out_i:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    return np.concatenate(out_i), np.concatenate(out_j)


def _gated_pairs_kd(xy, passes, r_same, r_other):
    """(i, j), j < i - 1, passing the gate: cKDTree candidates at the widened radius, then the exact gate"""
    r = max(float(r_same), float(r_other))
    tree = cKDTree(xy.astype(np.float64))
    pr = tree.query_pairs(_kd_radius(r), output_type="ndarray").astype(np.int64)
    i, j = np.maximum(pr[:, 0], pr[:, 1]), np.minimum(pr[:, 0], pr[:, 1])
    keep = j < i - 1
    i, j = i[keep], j[keep]
    ok = gate(xy[j, 0], xy[j, 1], passes[j], xy[i, 0], xy[i, 1], passes[i], r_same, r_other)
    return i[ok], j[ok]


def enumerate_reoptimize(node_xy, node_pass, r_same, r_other, method="auto"):
    """-> (src, tgt) int32: the pair list of one reoptimize() in the reference's loop order.  method: 'brute', 'kd' or
    'auto' (the KD-tree prefilter for n > 4096 at finite radii)."""
    xy = np.ascontiguousarray(node_xy, F32).reshape(-1, 2)
    ps = np.ascontiguousarray(node_pass, np.int32)
    n = xy.shape[0]
    if n < 2:
        return np.zeros(0, np.int32), np.zeros(0, np.int32)
    finite = math.isfinite(max(float(r_same), float(r_other)))
    if method == "kd" or (method == "auto" and n > 4096 and finite):
        if not finite:
            raise ValueError("the KD-tree prefilter needs finite radii")
        gi, gj = _gated_pairs_kd(xy, ps, r_same, r_other)
    else:
        gi, gj = _gated_pairs_brute(xy, ps, r_same, r_other, np.arange(n), lambda q: q - 1)
    si = np.arange(1, n, dtype=np.int64)
    i = np.concatenate([si, gi])
    j = np.concatenate([si - 1, gj])
    key = np.where(j == i - 1, -1, j)                  # the successive pair comes first, then ascending j
    order = np.lexsort((key, i))
    return i[order].astype(np.int32), j[order].astype(np.int32)


def enumerate_online(node_xy, node_pass, r_same, r_other):
    """-> (src, tgt) int32: the pair list of one updatePoseGraphObsConstraints() for the newest node n-1"""
    xy = np.ascontiguousarray(node_xy, F32).reshape(-1, 2)
    ps = np.ascontiguousarray(node_pass, np.int32)
    n = xy.shape[0]
    if n < 2:
        return np.zeros(0, np.int32), np.zeros(0, np.int32)
    pre = n - 2
    j = np.arange(max(n - 3, 0))
    ok = gate(xy[j, 0], xy[j, 1], ps[j], xy[pre, 0], xy[pre, 1], ps[pre], r_same, r_other)
    j = j[ok]
    src = np.concatenate([[n - 1], np.full(len(j), pre)]).astype(np.int32)
    tgt = np.concatenate([[pre], j]).astype(np.int32)
    return src, tgt


def shard(src, tgt, rank, world):
    return src[rank::world], tgt[rank::world]


# ---- guesses ------------------------------------------------------------------------------------------------------
def _map_unique(v, fn, dtype):
    u, inv = np.unique(v, return_inverse=True)
    return np.array([fn(a) for a in u], dtype)[inv].reshape(np.shape(v))


def angle_mod(d):
    """AngleMod in binary64 of binary32 angles, rounded to binary32"""
    d = np.asarray(d, F32).astype(np.float64)
    return (d - TWO_PI * np.rint(d / TWO_PI)).astype(F32)


def guesses(poses, src, tgt):
    """-> (guess (k, 3) = (tx, ty, angle), T (k, 4) = (c, s, tx, ty)) float32 of pairs (src = node_2, tgt = node_1)"""
    P = np.ascontiguousarray(poses, F32).reshape(-1, 3)
    s, t = np.asarray(src, np.int64), np.asarray(tgt, np.int64)
    tx = np.subtract(P[s, 0], P[t, 0], dtype=F32)
    ty = np.subtract(P[s, 1], P[t, 1], dtype=F32)
    ang = np.negative(P[t, 2])
    c1 = _map_unique(ang, lambda a: _libm.cosf(float(a)), F32)
    s1 = _map_unique(ang, lambda a: _libm.sinf(float(a)), F32)
    gx = np.add(np.multiply(c1, tx, dtype=F32), np.multiply(np.negative(s1), ty, dtype=F32), dtype=F32)
    gy = np.add(np.multiply(s1, tx, dtype=F32), np.multiply(c1, ty, dtype=F32), dtype=F32)
    g2 = angle_mod(np.subtract(P[s, 2], P[t, 2], dtype=F32))
    c = _map_unique(g2, lambda a: math.cos(float(a)), np.float64).astype(F32)
    sn = _map_unique(g2, lambda a: math.sin(float(a)), np.float64).astype(F32)
    return np.stack([gx, gy, g2], 1).reshape(-1, 3), np.stack([c, sn, gx, gy], 1).reshape(-1, 4)


# ---- boundary angles ----------------------------------------------------------------------------------------------
def near_boundary(v):
    """binary64 values within 32 binary64 ulps of the midpoint of two adjacent binary32 values"""
    low = np.asarray(v, np.float64).view(np.int64) & 0x1FFFFFFF
    return np.abs(low - 0x10000000) <= 32


def is_boundary_angle(g):
    g = float(F32(g))
    return bool(near_boundary(math.cos(g)) or near_boundary(math.sin(g)))


def boundary_angles(lo, hi):
    """every binary32 g in [lo, hi) (0 < lo < hi) whose libm cos or sin meets the boundary predicate: a vectorised
    search over the binary32 values with numpy's binary64 cos / sin, each hit confirmed with math.cos / math.sin"""
    a = int(np.array(lo, F32).view(np.uint32))
    b = int(np.array(hi, F32).view(np.uint32))
    out = []
    step = 1 << 22
    for k in range(a, b, step):
        g = np.arange(k, min(k + step, b), dtype=np.uint32).view(F32).astype(np.float64)
        # numpy's cos / sin may differ from libm by an ulp or two: search a slightly wider window, then confirm
        low_c = np.abs((np.cos(g).view(np.int64) & 0x1FFFFFFF) - 0x10000000)
        low_s = np.abs((np.sin(g).view(np.int64) & 0x1FFFFFFF) - 0x10000000)
        for x in g[(low_c <= 40) | (low_s <= 40)]:
            if is_boundary_angle(x):
                out.append(F32(x))
    return np.array(out, F32)
