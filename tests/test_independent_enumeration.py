"""CPU: the oracle's candidate-pair enumeration and pair guesses against the independent reference
(``ref_enumeration``) at the edges of the contract (``enum_cases``), bit for bit, and the reference's own checks."""
import math

import numpy as np
import pytest

import enum_cases as EC
import ref_enumeration as R
from oracle import oracle_py as O

F32 = np.float32


def _oracle_list(c, online=False):
    f = O.enumerate_online if online else O.enumerate_pairs
    return f(c["poses"][:, :2], c["passes"], float(c["r_same"]), float(c["r_other"]))


def _reference_list(c, online=False):
    if online:
        return R.enumerate_online(c["poses"][:, :2], c["passes"], c["r_same"], c["r_other"])
    return R.enumerate_reoptimize(c["poses"][:, :2], c["passes"], c["r_same"], c["r_other"])


def _assert_lists_equal(c, online=False):
    ws, wt = _reference_list(c, online)
    gs, gt = _oracle_list(c, online)
    assert len(gs) == len(ws), (c["name"], len(gs), len(ws))
    assert np.array_equal(gs, ws) and np.array_equal(gt, wt), c["name"]
    return ws, wt


# ---- the reference's own checks ------------------------------------------------------------------------------------
def test_gate_distance_of_a_345_layout_is_exact():
    assert R.gate_distance((0.0, 0.0), (3.0, 4.0)) == F32(5.0)
    assert R.gate_distance((100.0, 100.0), (103.0, 104.0)) == F32(5.0)
    assert R.gate(3.0, 4.0, 0, 0.0, 0.0, 0, 5.0, 1.0) and not R.gate(3.0, 4.0, 0, 0.0, 0.0, 1, 5.0, np.nextafter(F32(5), F32(0)))
    # a binary32 layout whose rounded distance equals the radius while the real distance exceeds it
    q = (F32(0.375), F32(-1.25))
    for r in (5.0, 3.0, 2.0):
        p = EC.tie_point(q, r, "tie")
        assert R.gate_distance(q, p) == F32(r) and EC.real_distance_exceeds(q, p, r), r
        assert R.gate_distance(q, EC.tie_point(q, r, "over")) == np.nextafter(F32(r), F32(np.inf))
        assert R.gate_distance(q, EC.tie_point(q, r, "under")) == np.nextafter(F32(r), F32(0))


@pytest.mark.parametrize("name", ["order_shuffled", "coincident_600", "radius0_with_duplicates", "signed_zeros_r0",
                                  "huge_coords_r5", "tie_other_mixed_tie_pos5", "passes_extreme"])
def test_reference_prefilter_equals_brute_force(name):
    if name == "coincident_600":
        c = EC.case(name, np.tile(np.array([[1.5, -2.25, 0.0]], F32), (600, 1)), np.arange(600) % 2, 0.0, 0.0)
    elif name == "tie_other_mixed_tie_pos5":
        c = EC.tie_layout(EC.TIE_CONFIGS[2], 5)
    else:
        c = next(x for x in EC.pass_radius_cases() + EC.geometry_cases() if x["name"] == name)
    xy, ps = c["poses"][:, :2], c["passes"]
    b = R.enumerate_reoptimize(xy, ps, c["r_same"], c["r_other"], method="brute")
    k = R.enumerate_reoptimize(xy, ps, c["r_same"], c["r_other"], method="kd")
    assert len(b[0]) > len(xy) - 1 or name == "huge_coords_r5"
    assert np.array_equal(b[0], k[0]) and np.array_equal(b[1], k[1])


def test_boundary_angle_finder():
    found = R.boundary_angles(0.1, 0.125)
    assert F32(0.10123747) in found and F32(0.11056483) in found
    for g in found:
        cs = (math.cos(float(g)), math.sin(float(g)))
        assert R.near_boundary(cs[0]) or R.near_boundary(cs[1]), g
    for g in (0.11056483, 0.31426188, 1.0480543):           # sin, cos, cos
        assert R.is_boundary_angle(g) and R.is_boundary_angle(-F32(g)), g
    assert not R.is_boundary_angle(0.5) and not R.near_boundary(1.0)


# ---- oracle == reference -------------------------------------------------------------------------------------------
_GROUPS = {
    "tie345": EC.tie_345_cases,
    "ties": EC.tie_cases,
    "passes_radii": EC.pass_radius_cases,
    "geometry": EC.geometry_cases,
    "angles": lambda: [EC.angle_case()],
    # the oracle's loop is O(n^2): 32767 and 32768 (hierarchy boundaries of the CUDA path only) stay in the GPU tier
    "sizes": lambda: [EC.size_case(n) for n in EC.SIZES if n <= 1025 or n == 32769],
}


@pytest.mark.parametrize("group", list(_GROUPS))
def test_oracle_reoptimize_list_equals_reference(group):
    for c in _GROUPS[group]():
        _assert_lists_equal(c)


def test_oracle_online_list_equals_reference():
    cases = [EC.online_size_case(n) for n in EC.ONLINE_SIZES + [2, 3, 4, 5]]
    cases += EC.tie_cases(online=True)[::5] + EC.tie_345_cases() + EC.pass_radius_cases() + EC.geometry_cases()[1:6]
    for c in cases:
        ws, _ = _assert_lists_equal(c, online=True)
        assert len(c["passes"]) < 2 or len(ws) >= 1


def _oracle_guesses(poses, src, tgt):
    g = np.zeros((len(src), 3), F32)
    T = np.zeros((len(src), 4), F32)
    for k, (s, t) in enumerate(zip(src, tgt)):
        g[k] = O.relative_guess(poses[t, :2], float(poses[t, 2]), poses[s, :2], float(poses[s, 2]))
        T[k] = O.guess_matrix(g[k])
    return g, T


@pytest.mark.parametrize("name", ["angles", "boundary_headings", "walk", "ties"])
def test_oracle_guesses_equal_reference(name):
    """relative_guess + guess_matrix of every listed pair: tx, ty with libm cosf / sinf, AngleMod in binary64 and the
    binary64 libm cos / sin, bit for bit — at +-pi, float32(pi) and past it, +-1e4 rad, +-0 and boundary angles"""
    if name == "angles":
        c = EC.angle_case(extra=[0.11056483, -0.31426188, 1.0480543, 1e4 + 0.11056483])
    elif name == "boundary_headings":
        c = EC.boundary_heading_case([0.11056483, -0.31426188, 1.0480543], n=120)
    elif name == "walk":
        c = EC.pass_radius_cases()[0]
    else:
        c = EC.tie_layout(EC.TIE_CONFIGS[0], 3)
    src, tgt = _assert_lists_equal(c)
    wg, wT = R.guesses(c["poses"], src, tgt)
    gg, gT = _oracle_guesses(c["poses"], src, tgt)
    assert gg.tobytes() == wg.tobytes() and gT.tobytes() == wT.tobytes(), name
    if name == "boundary_headings":
        amb = R.near_boundary(np.cos(wg[:, 2].astype(np.float64))) | R.near_boundary(np.sin(wg[:, 2].astype(np.float64)))
        assert amb.sum() > len(src) // 3


def test_angle_mod_edges():
    """AngleMod's rint at the half-turn: float32(pi) wraps to the negative side, pi itself is not representable; far
    angles keep their binary32 value modulo 2 pi"""
    pi32 = EC.PI32
    assert R.angle_mod(pi32) < 0 and R.angle_mod(-pi32) > 0
    assert R.angle_mod(np.nextafter(pi32, F32(0))) > 0
    for a in (pi32, -pi32, F32(1e4), F32(-1e4), F32(9999.5), F32(0.0), F32(-0.0)):
        assert R.angle_mod(a).tobytes() == F32(O.angle_mod(float(a))).tobytes(), a
