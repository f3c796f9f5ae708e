"""Odometry at the edges of the pose-cell plan, and proof that each generated case is an edge.

Every pose-cell kernel turns the odometry of one update into per-plane integer decisions in float64
(``oracle.posecells.path_integration_plan``, ``posecell_network.py:252-267,249,304``): the integer origin of each
plane (``numpy.around``, half to even), the LUT filter (``int(diff*10) < 0`` selects the filter of origin -1), the
theta origin ``floor(vr + .5)``, and the translation bound ``3 + ceil|vt| <= min(X, Y)``.  A wrong decision moves a
whole plane by one cell, and random odometry almost never lands on a boundary.  ``edge_cases`` emits, for a grid
shape, the float64 values on each side of every such boundary (found with ``numpy.nextafter``), plus odometry
across the whole accepted range and beyond it; the GPU tests (test_gpu_posecell_edges.py) run them through every
kernel family.  The tests here check that each pair really straddles its boundary, so that the GPU cases cannot
silently turn into ordinary ones.
"""
from __future__ import annotations

import functools
import math

import numpy as np
import pytest
from scipy import ndimage

from oracle import posecells as opc

VS = opc.PC_CELL_X_SIZE
ERR_LUT_KEY, ERR_RADIUS, ERR_THETA = 1, 2, 4      # PRS_ERR_* of include/pyratslam_b200.h


def _angles(n_th):
    mid = n_th // 2
    a = (np.arange(n_th) - mid) * (2.0 * np.pi / n_th)
    return np.cos(a), np.sin(a)


def plan(shape, vtrans, vrot):
    """The decisions of one update as the kernels make them: ``(ox int[Th], oy int[Th], key int[Th], og, err)``.

    Finite odometry gives exactly ``path_integration_plan``'s numbers.  Non-finite odometry follows the device's
    float -> int conversion (NaN -> 0), where the numpy plan raises; the error bits are those of the header."""
    X, Y, Th = shape
    c, s = _angles(Th)
    with np.errstate(invalid="ignore", over="ignore"):
        vt = vtrans / VS
        vr = vrot / (2.0 * np.pi / Th)
        ex, ey = vt * c, vt * s
        oxd, oyd = np.around(ex), np.around(ey)
        kd = (ex - oxd) * 10.0
        key = np.where(np.isfinite(kd), np.trunc(np.nan_to_num(kd)), 0).astype(np.int64)
        og = math.floor(vr + 0.5) if math.isfinite(vr + 0.5) else None
    err = ERR_LUT_KEY if (key >= 5).any() else 0
    if not (3.0 + math.ceil(abs(vt)) <= min(X, Y) if math.isfinite(vt) else False):
        err |= ERR_RADIUS
    if og is None or not abs(og) <= 64:
        err |= ERR_THETA
    ox, oy = (np.where(np.isfinite(o), o, 0).astype(np.int64) for o in (oxd, oyd))
    return ox, oy, key, og, err


def _walk(v0, n):
    """v0 and its n float64 neighbours on each side, ascending."""
    lo, hi = [], []
    a = b = float(v0)
    for _ in range(n):
        a, b = np.nextafter(a, -np.inf), np.nextafter(b, np.inf)
        lo.append(float(a))
        hi.append(float(b))
    return lo[::-1] + [float(v0)] + hi


def _exact_vtrans(target, coef, n=512):
    """A vtrans with ``(vtrans / 0.2) * coef == target`` exactly in float64, or None."""
    for v in sorted(_walk(target * VS / coef, n), key=lambda v: abs(v - target * VS / coef)):
        if (v / VS) * coef == target:
            return v
    return None


def _straddle(f, v0, n=4096):
    """Adjacent float64 values (a, b), a < b, nearest to v0 with f(a) != f(b)."""
    up = dn = float(v0)
    fu = fd = f(up)
    for _ in range(n):
        u2, d2 = float(np.nextafter(up, np.inf)), float(np.nextafter(dn, -np.inf))
        fu2, fd2 = f(u2), f(d2)
        if fu2 != fu:
            return up, u2
        if fd2 != fd:
            return d2, dn
        up, fu, dn, fd = u2, fu2, d2, fd2
    raise AssertionError("no boundary within %d ulps of %r" % (n, v0))


@functools.lru_cache(maxsize=None)
def edge_cases(shape):
    """Edge odometry for a grid shape: a list of ``(cls, vtrans, vrot, what, group)``.

    Boundary classes come as two rows of one ``group`` (an integer), the adjacent float64 values below and above the
    boundary, whose plans differ in ``what``: ``("ox"|"oy", k)``, ``("key", k)``, ``"og"`` or ``"radius"``.  The half
    origins add the value exactly on the half (``group`` None).  Range classes (``what`` and ``group`` None) are
    single rows.  Some rows are refused by the reference (LUT key 5, a translation beyond the grid, a theta origin
    beyond +-64, non-finite odometry): ``plan(...)[4]`` gives their error bits."""
    X, Y, Th = shape
    c, s = _angles(Th)
    minxy = min(X, Y)
    vr_small = 0.3 * (2.0 * np.pi / Th)                 # og = 0
    out = []
    gid = iter(range(10 ** 6))

    def fits(vt):
        return 3 + math.ceil(abs(vt)) <= minxy

    # integer origin exactly at a half: (vtrans / 0.2) * cos_k (or sin_k) == n + 0.5 for some plane k.  Plane order:
    # far from the axes first, so that the other planes of the same odometry stay away from the LUT hole
    order = sorted(range(Th), key=lambda k: -min(abs(c[k]), abs(s[k])))
    for comp, coefs, targets in (("ox", c, (1.5, -0.5, -2.5, 2.5, -1.5, 3.5)),
                                 ("oy", s, (0.5, -0.5, 2.5, -2.5, 1.5, -3.5))):
        for t in targets:
            for k in order:
                if abs(coefs[k]) < 0.3 or not fits(t / coefs[k]):
                    continue
                v = _exact_vtrans(t, coefs[k])
                if v is None:
                    continue
                # neighbouring vtrans can give the same product: the boundary is where the origin changes
                ci = 0 if comp == "ox" else 1
                lo, hi = _straddle(lambda w: int(plan(shape, w, vr_small)[ci][k]), v)
                if (plan(shape, lo, vr_small)[4] | plan(shape, hi, vr_small)[4]) & ERR_RADIUS:
                    continue
                g = next(gid)
                out.append(("half_" + comp, v, vr_small, (comp, k), None))        # exactly on the half
                for w in (lo, hi):
                    out.append(("half_" + comp, w, vr_small, (comp, k), g))
                break
    # F0 / F-1: int(diff * 10) switches between 0 and -1 (diff near -0.1), origins n = 0, 1, -1, 2
    for n in (0, 1, -1, 2):
        for k in order[: max(1, Th // 4)]:
            if abs(c[k]) < 0.3 or not fits((n - 0.1) / c[k]) or not fits((n - 0.1) / c[k] * 1.01):
                continue
            a, b = _straddle(lambda v: int(plan(shape, v, vr_small)[2][k]), (n - 0.1) * VS / c[k])
            g = next(gid)
            for w in (a, b):
                out.append(("fsel", w, vr_small, ("key", k), g))
            break
    # theta origin: vr + 0.5 exactly an integer m (og = m there, m - 1 just below), og in -8..8 and at +-64 / +-65
    vrs = 2.0 * np.pi / Th
    for m in list(range(-8, 10)) + [-64, 65]:
        a, b = _straddle(lambda v: plan(shape, 0.05, v)[3], (m - 0.5) * vrs)
        g = next(gid)
        for w in (a, b):
            out.append(("og", 0.05, w, "og", g))
    # translation bound: 3 + ceil|vt| == min(X, Y), then one past it; both signs of vtrans
    R = minxy - 3
    for sign in (1.0, -1.0):
        a, b = _straddle(lambda v: plan(shape, v, 0.1 * vrs)[4] & ERR_RADIUS, sign * R * VS)
        g = next(gid)
        for w in (a, b):
            out.append(("radius", w, 0.1 * vrs, "radius", g))
    # wide ranges: translations over the accepted range with both signs, theta origins far out, non-finite odometry
    rng = np.random.default_rng(sum(shape))
    for f in (0.13, 0.37, 0.61, 0.83, 0.97):
        for sign in (1.0, -1.0):
            vt = sign * f * R
            out.append(("vtrans", vt * VS, float(rng.uniform(-0.45, 0.45)) * vrs, None, None))
    for og in (2, 3, 4, 5, 6, 7, 8, 9, 17, 40, 64, 65):
        for sign in (1, -1):
            out.append(("vrot", float(rng.uniform(-0.4, 0.4)) * R * VS / 2, (sign * og + rng.uniform(-0.4, 0.4)) * vrs,
                        None, None))
    for vt, vr in ((np.nan, 0.0), (0.1, np.nan), (np.inf, 0.0), (-np.inf, 0.0), (0.1, np.inf), (0.1, -np.inf),
                   (np.nan, np.nan)):
        out.append(("nonfinite", float(vt), float(vr), None, None))
    return tuple(out)



# ------------------------------------------------------------------ the one-step cases of the GPU tests (oracle side)
NEG_GIS = (-0.005, -0.0005, -0.0, 0.0)


def _f32(a):
    return np.asarray(a, dtype=np.float32).astype(np.float64)


@functools.lru_cache(maxsize=None)
def start_states(shape):
    """(packet after realistic updates, two packets one across the periodic corner, dense random, packet x5), as float32
    values.  The packets are centred on plane Th // 2."""
    X, Y, Th = shape
    net = opc.PoseCellNetwork(shape, global_inhibition=0.05)
    net.inject(1.0, (X // 2, Y // 2, Th // 2))
    for v in [(0.11, 0.02), (0.21, -0.03), (0.07, 0.0)]:
        net.update(v)
    pk = net.posecells
    am = np.unravel_index(pk.argmax(), shape)
    corner = np.roll(pk, (X - 1 - am[0], 0 - am[1], Th - 1 - am[2]), axis=(0, 1, 2))
    # every cell non-zero, over a packet: a uniform random field alone is ill-conditioned in float32 (its filtered
    # planes cancel to a few cells of 1e-6 of the peak; the oracle's answer then rests on the last bits of each sum)
    dense = pk / pk.max() + np.random.default_rng(X * Y * Th).uniform(0.0, 0.3, shape)
    return tuple(_f32(s) for s in (pk, pk + 0.6 * corner, dense, 5.0 * pk))


def start_for(shape, j, row):
    """Start state j for an edge row.  A row about one plane k (a half origin, the F0 / F-1 switch) gets the start
    rolled along theta so that its packet is centred on plane k: a decision in a plane without activity changes nothing
    a test can compare."""
    st = start_states(shape)[j]
    if not isinstance(row[3], tuple):
        return st
    return np.roll(st, row[3][1] - shape[2] // 2, axis=2)


def dog(state):
    return ndimage.correlate(state, opc.diff_gaussian_3d(), mode="wrap")


def _one_step(shape, states, gis, odom):
    """The oracle's update for each case: (state, total, arg-max) or None where the device reports an error."""
    net = opc.PoseCellNetwork(shape)
    out = []
    for st, g, (vt, vr) in zip(states, gis, odom):
        if plan(shape, vt, vr)[4]:
            out.append(None)
            continue
        net.global_inhibition = float(g)
        net.posecells = st.copy()
        am = net.update((vt, vr))
        out.append((net.posecells, net.last_total, am))
    return out


def _away_from_gi(state, g):
    """For gi < 0 inhibition is discontinuous at a == gi (below: -gi, above: a - gi ~ 0).  Scale the state until no cell
    of its DoG response lies within 2e-6 of the peak of gi, so that float32 rounding cannot move a cell across."""
    for _ in range(20):
        pre = dog(state)
        if g >= 0 or np.abs(pre - g).min() > 2e-6 * np.abs(pre).max():
            return state
        state = _f32(state * 1.0137)
    raise AssertionError("no state away from the inhibition threshold")


@functools.lru_cache(maxsize=None)
def one_step_suite(shape, kind):
    """One-step cases of one shape: ``(states, gis, odom, errs, refs, rows)`` -- start states, inhibitions, odometry,
    expected error bits, the oracle's ``(state, total, arg-max)`` (None where the device reports an error) and the edge
    row of each case.

    kind "edges": every edge row on two start states, positive inhibition (a fraction of the DoG peak of the state).
    kind "inhibition": gi in NEG_GIS on the three packet starts, with a spread of accepted edge rows."""
    rows = edge_cases(shape)
    states, gis, odom, of = [], [], [], []
    if kind == "edges":
        fracs = (0.05, 0.15, 0.3, 0.5, 0.7)
        for i, r in enumerate(rows):
            for j in (i % 4, (i + 1) % 4):
                st = start_for(shape, j, r)
                states.append(st)
                gis.append(float(np.float32(fracs[(i + j) % 5] * dog(st).max())))
                odom.append((r[1], r[2]))
                of.append(r)
    else:
        ok = [r for r in rows if plan(shape, r[1], r[2])[4] == 0 and abs(plan(shape, r[1], r[2])[3]) <= 4]
        pick = ok[:: max(1, len(ok) // 7)][:7]
        for g in NEG_GIS:
            for j in (0, 1, 3):
                for r in pick:
                    states.append(_away_from_gi(start_for(shape, j, r), g))
                    gis.append(float(np.float32(g)))
                    odom.append((r[1], r[2]))
                    of.append(r)
    states, gis, odom = np.stack(states), np.array(gis), np.array(odom, dtype=np.float64)
    errs = np.array([plan(shape, vt, vr)[4] for vt, vr in odom])
    return states, gis, odom, errs, _one_step(shape, states, gis, odom), tuple(of)


def _update_with(shape, state, gi, vtrans, vrot, alt=None):
    """``PoseCellNetwork.update`` of the oracle, restated with one decision of the plan overridden: ``alt = (name, k,
    value)`` sets plane k's x origin (``"ox"``), y origin (``"oy"``) or LUT key (``"key"``, which picks F0 or F-1)."""
    X, Y, Th = shape
    pc = dog(state)
    pc[pc < gi] = 0
    pc[pc >= gi] -= gi
    total = np.sum(pc.ravel())
    if total != 0:
        pc /= total
    vt, origins, diff, keys, og = opc.path_integration_plan(vtrans, vrot, Th)
    lut = _lut()
    keys = list(keys)
    if alt is not None:
        name, k, value = alt
        if name == "key":
            keys[k] = value
        else:
            origins[0 if name == "ox" else 1, k] = value
    out = np.empty_like(pc)
    for k in range(Th):
        plane = np.roll(pc[:, :, k], (-int(origins[0, k]), -int(origins[1, k])), axis=(0, 1))
        out[:, :, k] = ndimage.correlate(plane, lut[(keys[k], keys[k])], mode="wrap")
    out[out < 0] = 0
    out = ndimage.correlate1d(out, opc.diff_gaussian_offset_1d(size=7, origin=og), axis=2, mode="wrap")
    out[out < 0] = 0
    return out


@functools.lru_cache(maxsize=None)
def _lut():
    return opc.build_filter_lut_2d()

SHAPES = [(21, 21, 36), (50, 50, 10), (17, 23, 11), (12, 10, 5)]


def _groups(cases):
    groups = {}
    for r in cases:
        if r[4] is not None:
            groups.setdefault(r[4], []).append(r)
    return list(groups.values())


def _what(shape, row):
    ox, oy, key, og, err = plan(shape, row[1], row[2])
    what = row[3]
    if what == "og":
        return og
    if what == "radius":
        return err & ERR_RADIUS
    name, k = what
    return {"ox": ox, "oy": oy, "key": key}[name][k]


@pytest.mark.parametrize("shape", SHAPES)
def test_boundary_pairs_straddle_their_boundary(shape):
    """Each boundary group: adjacent float64 values whose plans differ in the quantity the group is about."""
    groups = _groups(edge_cases(shape))
    assert len(groups) >= 20
    for g in groups:
        vals = [r[1] if r[3] != "og" else r[2] for r in g]
        assert all(float(np.nextafter(a, b)) == b for a, b in zip(vals, vals[1:])), g        # adjacent floats
        assert _what(shape, g[0]) != _what(shape, g[-1]), g


@pytest.mark.parametrize("shape", SHAPES)
def test_half_origins_are_exact_halves(shape):
    """The exact row of each half-origin group puts one plane's offset exactly on n + 0.5, in the numpy plan of the
    oracle and in ours, and the group's two neighbours differ in that plane's origin; numpy's half-to-even and the
    half-away-from-zero rounding give different origins on some of them."""
    X, Y, Th = shape
    c, s = _angles(Th)
    rows = [r for r in edge_cases(shape) if r[0].startswith("half_")]
    triples = [rows[i:i + 3] for i in range(0, len(rows), 3)]
    assert len(triples) >= 8
    n_away_differs = n_negative = 0
    for at, lo, hi in triples:
        assert at[4] is None and lo[4] == hi[4] is not None and at[3] == lo[3] == hi[3]
        comp, k = at[3]
        e = (at[1] / VS) * (c[k] if comp == "ox" else s[k])
        assert e - math.floor(e) == 0.5, at
        vt, origins, diff, keys, og = opc.path_integration_plan(at[1], at[2], Th)
        assert origins[0 if comp == "ox" else 1, k] == np.around(e) == _what(shape, at)
        away = math.copysign(math.floor(abs(e) + 0.5), e)
        n_away_differs += away != np.around(e)
        n_negative += e < 0
        assert _what(shape, lo) != _what(shape, hi)
        assert _what(shape, at) in (_what(shape, lo), _what(shape, hi))
    assert n_away_differs >= 2 and n_negative >= 3


@pytest.mark.parametrize("shape", SHAPES)
def test_plan_matches_the_oracle_plan_on_finite_odometry(shape):
    """``plan`` restates ``path_integration_plan`` (plus the bits of the header) for every finite row."""
    X, Y, Th = shape
    for cls, vtrans, vrot, _, _ in edge_cases(shape):
        if not (math.isfinite(vtrans) and math.isfinite(vrot)):
            assert plan(shape, vtrans, vrot)[4] & (ERR_RADIUS if not math.isfinite(vtrans) else ERR_THETA)
            continue
        ox, oy, key, og, err = plan(shape, vtrans, vrot)
        vt, origins, diff, keys, og2 = opc.path_integration_plan(vtrans, vrot, Th)
        assert np.array_equal(ox, origins[0]) and np.array_equal(oy, origins[1]) and list(key) == keys and og == og2
        assert bool(err & ERR_LUT_KEY) == (max(keys) >= 5)
        assert bool(err & ERR_RADIUS) == (3 + math.ceil(abs(vt)) > min(X, Y))
        assert bool(err & ERR_THETA) == (abs(og) > 64)


@pytest.mark.parametrize("shape", SHAPES)
def test_edge_cases_cover_every_class(shape):
    X, Y, Th = shape
    cases = edge_cases(shape)
    plans = [plan(shape, r[1], r[2]) for r in cases]
    ogs = {p[3] for p in plans if p[3] is not None}
    assert set(range(-8, 9)) <= ogs and {-65, 65, -64, 64} <= ogs
    assert any(9 <= abs(o) < 64 for o in ogs)
    errs = [p[4] for p in plans]
    for bit in (ERR_LUT_KEY, ERR_RADIUS, ERR_THETA):
        assert any(e == bit for e in errs), bit             # each error alone on some row
    assert sum(e == 0 for e in errs) >= 0.6 * len(errs)     # most rows are accepted: their results are compared
    fsel = [p for r, p in zip(cases, plans) if r[0] == "fsel"]
    assert len(fsel) >= 2 and any((p[2] == -1).any() for p in fsel) and any((p[2] == 0).any() for p in fsel)
    vts = [r[1] / VS for r, p in zip(cases, plans) if p[4] == 0]
    R = min(X, Y) - 3
    assert max(vts) == R and min(vts) == -R                 # the largest translation the kernels accept, both signs
    assert any(r[0] == "radius" and p[4] == ERR_RADIUS for r, p in zip(cases, plans))
    assert sum(r[0] == "half_oy" for r in cases) >= 9 and sum(r[0] == "half_ox" for r in cases) >= 9


@pytest.mark.parametrize("shape", SHAPES)
def test_boundary_rows_are_visible_in_the_state(shape):
    """A kernel that decides one plane's origin or LUT filter the way the other side of the boundary does must fail the
    state bar of the GPU tests: for every accepted one-step case whose row is about a plane k, the oracle's state with
    that one decision taken from the row's neighbour across the boundary differs by more than 10x the float32 bar."""
    states, gis, odom, errs, refs, rows = one_step_suite(shape, "edges")
    groups = {}
    for r in edge_cases(shape):
        if isinstance(r[3], tuple):
            groups.setdefault((r[0], r[3]), []).append(r)
    n = 0
    for st, g, (vt, vr), ref, row in zip(states, gis, odom, refs, rows):
        if ref is None or not isinstance(row[3], tuple):
            continue
        name, k = row[3]
        idx = {"ox": 0, "oy": 1, "key": 2}[name]
        mine = plan(shape, vt, vr)[idx][k]
        # the neighbour across the boundary: the other row of the group; for the exact half, the neighbour that differs
        near = [r for r in groups[(row[0], row[3])] if r[4] is not None and (r[4] == row[4] or row[4] is None)
                and abs(r[1] - row[1]) <= 8192 * abs(np.spacing(row[1]))]
        alt = [plan(shape, r[1], r[2])[idx][k] for r in near if plan(shape, r[1], r[2])[idx][k] != mine]
        assert alt, row
        want = _update_with(shape, st, g, vt, vr)
        assert np.array_equal(want, ref[0])                          # the restatement is the oracle, bit for bit
        moved = _update_with(shape, st, g, vt, vr, (name, k, int(alt[0])))
        rel = np.abs(moved - want).max() / np.abs(want).max()
        assert rel > 1e-4, (row, g, rel)
        n += 1
    assert n >= 24
