"""Node tables at the edges of candidate-pair enumeration, shared by the CPU tier (oracle against ``ref_enumeration``)
and the GPU tier (CUDA path against ``ref_enumeration``).  Every case is a dict: name, poses (n, 3) float32 =
(x, y, theta), passes (n,) int32, r_same, r_other.  Nothing here computes an expected pair list."""
from fractions import Fraction

import numpy as np

from ref_enumeration import F32, gate_distance

I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
INF = float("inf")
PI32 = F32(np.pi)                                 # float32(pi) = 3.14159274, just above pi


def case(name, poses, passes, r_same, r_other):
    return dict(name=name, poses=np.ascontiguousarray(poses, F32).reshape(-1, 3),
                passes=np.ascontiguousarray(passes, np.int32), r_same=F32(r_same), r_other=F32(r_other))


def walk(n, seed, size=None, sessions=3, step=1.0):
    """trajectory-like nodes: 1 m steps with a drifting heading, folded into a square; `sessions` contiguous passes,
    each starting somewhere else.  theta = heading."""
    rng = np.random.default_rng(seed)
    size = size if size is not None else max(20.0, 2.0 * np.sqrt(max(n, 1)))
    head = np.cumsum(rng.uniform(-0.5, 0.5, n))
    pos = np.cumsum(np.stack([np.cos(head), np.sin(head)], 1) * step, 0)
    per = max(1, -(-n // sessions))
    sess = np.arange(n) // per
    pos += rng.uniform(0, 2 * size, (sessions + 1, 2))[sess]
    pos = size - np.abs(size - np.mod(pos, 2 * size))           # fold (reflect) into [0, size]^2
    poses = np.concatenate([pos, np.angle(np.exp(1j * head))[:, None]], 1)
    return poses.astype(F32), sess.astype(np.int32)


def reorder(poses, passes, order, seed=0):
    n = len(passes)
    if order == "trajectory":
        perm = np.arange(n)
    elif order == "reversed":
        perm = np.arange(n)[::-1]
    elif order == "shuffled":
        perm = np.random.default_rng(seed).permutation(n)
    elif order == "interleaved":                                # round robin over the sessions
        keys = np.zeros(n, np.int64)
        for p in np.unique(passes):
            idx = np.nonzero(passes == p)[0]
            keys[idx] = np.arange(len(idx))
        perm = np.lexsort((passes, keys))
    else:
        raise ValueError(order)
    return poses[perm], passes[perm]


# ---- gate ties --------------------------------------------------------------------------------------------------
def _f32_seq(x0, k):
    """binary32 values x0 + k ulps (x0 > 0)"""
    b = np.array(x0, F32).view(np.int32)
    return (b + np.asarray(k, np.int32)).view(F32)


def tie_point(q, r, which):
    """A point near q + (0.6 r, 0.8 r) whose gate distance from q is exactly r ('tie': the largest such x, so that the
    real distance is above r where the grid allows it), the next binary32 above r ('over') or the one below ('under')."""
    qx, qy = F32(q[0]), F32(q[1])
    y = F32(qy + F32(0.8 * r))
    xs = _f32_seq(F32(qx + F32(0.6 * r)), np.arange(-4096, 4097))
    dx, dy = np.subtract(xs, qx, dtype=F32), np.subtract(y, qy, dtype=F32)
    d = np.sqrt(np.add(np.multiply(dx, dx, dtype=F32), np.multiply(dy, dy, dtype=F32), dtype=F32), dtype=F32)
    assert gate_distance((qx, qy), (xs[0], y)) == d[0]
    r = F32(r)
    want = {"tie": r, "over": np.nextafter(r, F32(INF)), "under": np.nextafter(r, F32(0))}[which]
    hit = np.nonzero(d == want)[0]
    assert len(hit), (q, r, which)
    k = hit[-1] if which == "tie" else hit[0]
    return F32(xs[k]), y


def real_distance_exceeds(q, p, r):
    """exact: |p - q| > r for the binary32 coordinates"""
    dx = Fraction(float(p[0])) - Fraction(float(q[0]))
    dy = Fraction(float(p[1])) - Fraction(float(q[1]))
    return dx * dx + dy * dy > Fraction(float(r)) ** 2


# pass configurations of the tie layout: (name, tied node's pass, box mates' passes, query pass, r_same, r_other)
TIE_CONFIGS = [
    ("same_gt", 0, (0,), 0, 5.0, 2.0),            # same pass, r_same > r_other
    ("same_lt", 0, (1,), 0, 2.0, 5.0),            # same pass, r_same < r_other, mates of the other pass
    ("other_mixed", 1, (0,), 0, 2.0, 5.0),        # mixed-pass box whose only passing member is of the other pass
    ("other_pure", 1, (1,), 0, 5.0, 2.0),         # box without the query's pass
    ("inside_range", 0, (0, 2), 1, 2.0, 5.0),     # query pass inside the box's pass range, equal to none of its members
    ("equal", 1, (0,), 0, 3.0, 3.0),              # r_same == r_other
    ("extreme_min", I32_MIN, (I32_MAX,), I32_MAX, 2.0, 5.0),
    ("extreme_max", I32_MAX, (-7,), I32_MIN, 5.0, 2.0),
]


def tie_layout(config, pos, which="tie", online=False, leaf=13):
    """1026 nodes (two hierarchy levels).  The query node Q is node n-1 (reoptimize) or n-2 (online, with one newest
    node behind it).  One node at gate distance r from Q (see tie_point) sits at position `pos` of leaf `leaf` of the
    first level-2 box; every other node of that box lies further out on the same ray, 6 m apart, so the tied node is
    the only member of its leaf and of its level-2 box that can pass, and it is the lower corner of both boxes: a
    pruning error drops its pair instead of hiding behind a neighbour."""
    name, p_tie, p_mates, p_q, r_same, r_other = config
    r = r_same if p_tie == p_q else r_other
    q = (F32(0.375), F32(-1.25))
    tx, ty = tie_point(q, r, which)
    n = 1026
    k = np.arange(1024, dtype=np.float64)
    far = 2.0 * max(r_same, r_other) + 6.0 * k
    poses = np.zeros((n, 3), F32)
    poses[:1024, 0] = F32(q[0]) + F32(0.6) * far
    poses[:1024, 1] = F32(q[1]) + F32(0.8) * far
    passes = np.array(p_mates, np.int64)[np.arange(n) % len(p_mates)]
    t = 32 * leaf + pos
    poses[t, :2] = (tx, ty)
    passes[t] = p_tie
    qi = n - 2 if online else n - 1
    poses[qi, :2] = q
    passes[qi] = p_q
    other = n - 1 if online else n - 2                         # the node outside the gated range
    poses[other, :2] = (F32(-500.0), F32(-500.0))
    passes[other] = p_q
    poses[:, 2] = F32(0.25) * (np.arange(n) % 7)
    return case(f"tie_{name}_{which}_pos{pos}{'_online' if online else ''}", poses, passes.astype(np.int32), r_same, r_other)


def tie_cases(online=False):
    out = []
    for cfg in TIE_CONFIGS:
        positions = range(32) if cfg[0] in ("same_gt", "other_mixed") else (0, 17, 31)
        for pos in positions:
            out.append(tie_layout(cfg, pos, "tie", online))
        for which in ("over", "under"):
            for pos in (0, 31):
                out.append(tie_layout(cfg, pos, which, online))
    return out


def tie_345_cases():
    """3-4-5 layouts: the gate's distance is exactly 5.0f; radius 5 keeps them, the binary32 below 5 drops them"""
    pts = np.array([[0, 0], [3, 4], [-3, 4], [6, 8], [3, -4], [-4, -3], [0, 5], [5, 0], [100, 100], [103, 104],
                    [97, 96], [100, 105]], np.float64)
    poses = np.concatenate([pts, np.zeros((len(pts), 1))], 1).astype(F32)
    passes = np.zeros(len(pts), np.int32)
    below5 = float(np.nextafter(F32(5), F32(0)))
    return [case("tie345_r5", poses, passes, 5.0, 5.0), case("tie345_below5", poses, passes, below5, below5),
            case("tie345_rev", poses[::-1], passes, 5.0, 2.0)]


# ---- passes, radii, geometry ------------------------------------------------------------------------------------
def cluster(n, seed, spread, pass_values, theta=None):
    rng = np.random.default_rng(seed)
    poses = np.zeros((n, 3), F32)
    poses[:, :2] = rng.uniform(0, spread, (n, 2))
    poses[:, 2] = rng.uniform(-np.pi, np.pi, n) if theta is None else theta
    return poses, np.asarray(pass_values, np.int64)[rng.integers(0, len(pass_values), n)].astype(np.int32)


def pass_radius_cases():
    out = []
    for rs, ro in ((5.0, 2.0), (2.0, 5.0), (3.0, 3.0)):
        p, s = walk(600, seed=int(10 * rs + ro), size=20.0, sessions=4)
        out.append(case(f"walk_rs{rs:g}_ro{ro:g}", p, s, rs, ro))
    p, s = cluster(400, 3, 25.0, [I32_MIN, I32_MIN + 1, -5, -1, 0, I32_MAX - 1, I32_MAX])
    out.append(case("passes_extreme", p, s, 4.0, 2.5))
    out.append(case("passes_extreme_lt", p, s, 2.5, 4.0))
    p, s = walk(500, seed=5, size=15.0, sessions=3)
    m = len(p[2::3])
    p[0:3 * m:3, :2] = p[2::3, :2]                              # every third node on top of the node two ahead
    out.append(case("radius0_with_duplicates", p, s, 0.0, 0.0))
    out.append(case("radius_inf", p[:300], s[:300], INF, INF))
    out.append(case("radius_inf_same_only", p[:300], s[:300], INF, 0.0))
    return out


def geometry_cases():
    out = []
    p = np.zeros((3000, 3), F32)
    p[:, 0], p[:, 1] = F32(1.5), F32(-2.25)
    p[:, 2] = F32(0.5)
    s = (np.arange(3000) % 2).astype(np.int32)
    out.append(case("coincident_3000", p, s, 0.0, 0.0))
    z = np.array([[0.0, 0.0], [-0.0, 0.0], [0.0, -0.0], [-0.0, -0.0], [1e-45, 0.0], [0.0, -1e-45], [1e-38, 1e-38],
                  [-0.0, 0.0], [2.0, 0.0], [-0.0, -0.0]], np.float64)
    pz = np.concatenate([z, np.zeros((len(z), 1))], 1).astype(F32)
    out.append(case("signed_zeros_r0", pz, np.zeros(len(z), np.int32), 0.0, 0.0))
    out.append(case("signed_zeros_r1", pz, np.arange(len(z)) % 2, 1.0, 0.0))
    big = np.array([1e19, -1e19, 1.5e19, -1.5e19, 1e19, 3e19, -3e19], np.float64)
    rng = np.random.default_rng(9)
    pb = np.zeros((200, 3), F32)
    pb[:, 0] = big[rng.integers(0, len(big), 200)]
    pb[:, 1] = big[rng.integers(0, len(big), 200)]
    pb[::5, 1] = F32(0.0)
    sb = rng.integers(0, 2, 200).astype(np.int32)
    out.append(case("huge_coords_inf", pb, sb, INF, INF))
    out.append(case("huge_coords_r5", pb, sb, 5.0, 5.0))
    out.append(case("huge_coords_mixed", pb, sb, INF, 5.0))
    p, s = walk(3000, seed=11, size=45.0, sessions=4)
    for order in ("trajectory", "reversed", "shuffled", "interleaved"):
        po, so = reorder(p, s, order, seed=12)
        out.append(case(f"order_{order}", po, so, 5.0, 2.0))
    return out


SIZES = [0, 1, 2, 3, 4, 5, 31, 32, 33, 1023, 1024, 1025, 32767, 32768, 32769]
ONLINE_SIZES = [34, 35, 36, 67, 68]


def size_case(n):
    p, s = walk(n, seed=100 + n, sessions=3)
    return case(f"size_{n}", p, s, 5.0, 2.0)


def online_size_case(n):
    """a compact walk so that many candidates j <= n-4 pass against node n-2, some of either pass"""
    p, s = walk(n, seed=200 + n, size=6.0, sessions=2)
    return case(f"online_{n}", p, s, 3.0, 2.0)


def four_level_case():
    """1 048 577 nodes, the first size with four hierarchy levels: serpentine rows of 1024 nodes 1 m apart, rows
    3 m apart (the row above is at a gate tie: dist == 3.0f exactly), a few pairs per node"""
    n = 1_048_577
    k = np.arange(n)
    row, col = k // 1024, k % 1024
    col = np.where(row % 2 == 1, 1023 - col, col)
    poses = np.zeros((n, 3), F32)
    poses[:, 0] = col.astype(F32) - F32(512.0)
    poses[:, 1] = row.astype(F32) * F32(3.0) - F32(1536.0)
    poses[:, 2] = np.where(row % 2 == 1, PI32, F32(0.0))
    poses[k % 4099 == 0, 2] = F32(0.11056483)
    passes = (row // 128).astype(np.int32)
    return case("four_levels_1048577", poses, passes, 3.0, 2.0)


# ---- angles -----------------------------------------------------------------------------------------------------
SPECIAL_THETAS = [0.0, -0.0, np.pi, -np.pi, float(PI32), -float(PI32), float(np.nextafter(PI32, F32(4))),
                  -float(np.nextafter(PI32, F32(4))), float(np.nextafter(PI32, F32(0))), np.pi / 2, -np.pi / 2,
                  1e4, -1e4, 9999.5, -9999.25, 3 * np.pi, 2 * np.pi, -2 * np.pi, 1e-30, -1e-30]


def angle_case(extra=(), seed=31, name="angles"):
    """every ordered pair of the special headings (and `extra`) inside one 1 m cluster: all pairs pass the gate"""
    th = np.array(list(SPECIAL_THETAS) + [float(e) for e in extra], np.float64).astype(F32)
    rng = np.random.default_rng(seed)
    n = len(th)
    poses = np.zeros((n, 3), F32)
    poses[:, :2] = rng.uniform(-0.5, 0.5, (n, 2))
    poses[:, 2] = th
    return case(name, poses, np.zeros(n, np.int32), 5.0, 2.0)


def boundary_heading_case(angles, n=160, seed=41, name="boundary_headings"):
    """n nodes within 1 m of each other in one pass, theta cycling through 0 and the given boundary angles (and their
    negatives): every pair passes, and a pair whose two headings differ is a boundary pair"""
    rng = np.random.default_rng(seed)
    th = np.concatenate([[0.0], np.asarray(angles, np.float64)])
    poses = np.zeros((n, 3), F32)
    poses[:, :2] = rng.uniform(0.0, 0.7, (n, 2))
    poses[:, 2] = th[np.arange(n) % len(th)].astype(F32)
    return case(name, poses, np.zeros(n, np.int32), 5.0, 2.0)


def edge_cases():
    """every reoptimize edge case small enough for the CPU oracle"""
    return tie_345_cases() + tie_cases() + pass_radius_cases() + geometry_cases() + [angle_case()]
