"""Crafted ensemble records and host experience maps for the ensemble experience-map tests (no reference needed)."""
from __future__ import annotations

import math

import numpy as np

from pyratslam_b200.experience_ensemble import gate
from pyratslam_b200.experience_map import ExperienceMap


def crafted(rng, B, T, pose_size=(6, 5, 7)):
    """``(template [B,T], argmax [B,T,3], odom [T,2])`` on a small grid, so that candidates often lie across its wrap.

    Agent kinds (b % 6): a packet that never moves under one view (matches with the current experience); a cycle of
    views at one cell (repeated closures of the same pairs); a random walk with views from a small set and some frames
    matching no template (-1); uniformly random cells; cells on the grid's faces only; cells on the six neighbours of one
    cell (equal-distance ties).  The odometry has frames below the twist gate and turns beyond +-pi."""
    X, Y, Th = pose_size
    dims = np.array(pose_size)
    tpl = np.zeros((B, T), np.int64)
    am = np.zeros((B, T, 3), np.int64)
    for b in range(B):
        kind = b % 6
        K = int(rng.choice([1, 2, 3, 4, 8, 30]))
        c0 = rng.integers(0, dims)
        if kind == 0:
            tpl[b] = int(rng.integers(0, 3))
            am[b] = c0
        elif kind == 1:
            tpl[b] = np.arange(T) % K
            am[b] = c0
        elif kind == 2:
            steps = rng.integers(-1, 2, (T, 3))
            am[b] = (c0 + np.cumsum(steps, axis=0)) % dims
            tpl[b] = rng.integers(0, K, T)
            tpl[b, rng.random(T) < 0.15] = -1
        elif kind == 3:
            am[b] = rng.integers(0, dims, (T, 3))
            tpl[b] = rng.integers(0, K, T)
        elif kind == 4:
            am[b] = rng.integers(0, 2, (T, 3)) * (dims - 1)
            tpl[b] = rng.integers(0, min(K, 3), T)
        else:
            axis = rng.integers(0, 3, T)
            sign = rng.choice([-1, 1], T)
            cells = np.tile(c0, (T, 1))
            cells[np.arange(T), axis] += sign
            cells[rng.random(T) < 0.2] = c0
            am[b] = cells % dims
            tpl[b] = rng.integers(0, 2, T)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-40, 40, T)], axis=1)
    still = rng.random(T) < 0.25
    odom[still] = rng.choice([0.0, 0.0005], (int(still.sum()), 2))
    return tpl, am, odom


def host_maps(template, argmax, odom, pose_size, delta_pc=1.0):
    """Each agent's ``ExperienceMap(linked=True)`` over its records, tagged as ``RatslamRos.replay_native`` tags (the
    template of the frame before, none at t = 0 or for a negative template), with ``n_exp``, ``exp_id`` and ``em_xy``
    after every frame."""
    moved, tw = gate(odom)
    B, T = template.shape
    maps = []
    n_exp = np.zeros((B, T), np.int64)
    exp_id = np.full((B, T), -1, np.int64)
    em_xy = np.zeros((B, T, 2))
    for b in range(B):
        em = ExperienceMap(linked=True, pc_dims=pose_size, delta_pc=delta_pc)
        for t in range(T):
            if moved[t]:
                vt = int(template[b, t - 1]) if t > 0 else None
                em.update(float(tw[t, 0]), float(tw[t, 1]), tuple(int(c) for c in argmax[b, t]),
                          None if vt is None or vt < 0 else vt)
            n_exp[b, t] = len(em.experiences)
            if em.current_exp is not None:
                exp_id[b, t] = em.current_exp.index
                em_xy[b, t] = em.get_current_point()
        maps.append(em)
    return maps, n_exp, exp_id, em_xy


def arrays(em):
    """A host map's ``(experiences, links)`` as ``ExperienceMap.from_arrays`` takes them."""
    from pyratslam_b200.experience_ensemble import EXPERIENCE_DTYPE, LINK_DTYPE
    ex = np.zeros(len(em.experiences), EXPERIENCE_DTYPE)
    for i, e in enumerate(em.experiences):
        ex[i] = (e.pc_x, e.pc_y, e.pc_th, -1 if e.vt is None else e.vt, e.m_x, e.m_y, e.th)
    li = np.array(em.links, dtype=LINK_DTYPE) if em.links else np.zeros(0, LINK_DTYPE)
    return ex, li


def _angle_diff(a, b):
    d = np.abs(np.asarray(a) - np.asarray(b)) % (2 * math.pi)
    return np.minimum(d, 2 * math.pi - d)


def assert_same_map(got, want, exact_th=True, tol=1e-9, what=""):
    """``got`` and ``want`` (``ExperienceMap`` instances) have the same structure -- experience cells and tags, the
    link (from, to) list in creation order, the loop-closure count and the current experience -- positions and link
    lengths within ``tol``, link headings and facings within ``tol`` modulo 2 pi, and experience headings equal
    (``exact_th``) or within ``tol`` modulo 2 pi."""
    assert len(got.experiences) == len(want.experiences), what
    assert [(e.pc_x, e.pc_y, e.pc_th, e.vt) for e in got.experiences] == \
        [(e.pc_x, e.pc_y, e.pc_th, e.vt) for e in want.experiences], what
    assert [l[:2] for l in got.links] == [l[:2] for l in want.links], what
    assert got.n_loop_closures == want.n_loop_closures, what
    assert (got.current_exp is None) == (want.current_exp is None), what
    if got.current_exp is not None:
        assert got.current_exp.index == want.current_exp.index, what
    if want.experiences:
        gp, wp = np.array(got.get_poses()), np.array(want.get_poses())
        assert np.abs(gp[:, :2] - wp[:, :2]).max() <= tol, (what, np.abs(gp[:, :2] - wp[:, :2]).max())
        if exact_th:
            assert np.array_equal(gp[:, 2], wp[:, 2]), what
        else:
            assert _angle_diff(gp[:, 2], wp[:, 2]).max() <= tol, what
    if want.links:
        gl, wl = np.array([l[2:] for l in got.links]), np.array([l[2:] for l in want.links])
        assert np.abs(gl[:, 0] - wl[:, 0]).max() <= tol, what
        assert _angle_diff(gl[:, 1:], wl[:, 1:]).max() <= tol, what


def loop_recording(rng, T, K=6, moving=40, looping=60):
    """``(frames [T,256,256] uint8, odom [T,2])`` in which loops close: periods of ``moving`` synthetic frames under
    the bench's random odometry, then ``looping`` frames that show K fixed views in a cycle while the twist stays just
    above the 0.001 gate.  The pose-cell packet then stays put, so every revisit of a view closes a loop, and later
    cycles close the same pairs again."""
    from synth import synth_frames
    views = rng.integers(0, 256, (K, 256, 256), dtype=np.uint8)
    frames = synth_frames(rng, T)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    for t in range(T):
        p = t % (moving + looping)
        if p >= moving:
            frames[t] = views[(p - moving) % K]
            odom[t] = (0.0015, 0.0)
    return frames, odom
