"""The view-template -> pose-cell injection (ros_simulate.py:106-108) as the last node of the frame graph: every replay
mode against the oracle's replay with the same coupling, the O(1) arg-max rule on crafted states, templates appended
outside the plans, float64 and the active-set update, and the energies the device node does not take."""
import numpy as np
import pytest

from synth import synth_frames

pytestmark = pytest.mark.gpu

SHAPE = (21, 21, 36)
ROWS = np.arange(33, 96, 2)      # the pixels the 32x32 template is sub-sampled from (view_templates.py:48-57)


def _inputs(T, lag=1):
    """Frames with revisits of the frame `lag` steps back (every third frame) and the bench's odometry range: the packet
    has moved a little since the revisited template was made, so some injections take the arg-max with them."""
    frames = synth_frames(np.random.default_rng(5), T)
    for t in range(4, T, 3):
        frames[t] = frames[t - lag]
    rng = np.random.default_rng(6)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    for t, still in ((9, (0.0005, -0.0002)), (10, (0.0, 0.0)), (30, (0.0, 0.0))):
        if t < T:
            odom[t] = still          # below the 0.001 gate: no pose-cell update for this frame
    return frames, odom


def _oracle_moves(frames, odom, energy):
    """Injections that move the arg-max in the oracle's loop (oracle/drivers.py:replay_run, step by step)."""
    from oracle import drivers as odrv
    from oracle.posecells import PoseCellNetwork
    from oracle.view_templates import ViewTemplates
    pcn = PoseCellNetwork(SHAPE)
    pcn.inject(1, (10, 10, 18))
    vts = ViewTemplates(odrv.X_RANGE, odrv.Y_RANGE, odrv.X_STEP, odrv.Y_STEP, 256, 256, odrv.MATCH_THRESHOLD)
    n = 0
    for t in range(len(frames)):
        lin, ang = float(odom[t, 0]), float(odom[t, 1])
        if abs(lin) > 0.001 or abs(ang) > 0.001:
            pcn.update((lin / odrv.ODOM_FREQ, ang / odrv.ODOM_FREQ))
        pm = tuple(pcn.get_pc_max())
        tm = vts.match(frames[t], *pm)
        pcn.inject(energy, tm.location())
        n += tuple(pcn.get_pc_max()) != pm
    return n


def _pipelined(frames, odom, energy, depth, **kw):
    """pipe_submit / pipe_finish with `depth` frames in flight."""
    from pyratslam_b200 import ros_simulate
    node = ros_simulate.RatslamRos(inject_energy=energy, **kw)
    node._pipe_setup(depth)
    node.vts._grow(len(frames) + depth + 2)
    node._pipe_plans()
    T = len(frames)
    rec = {"template": np.zeros(T, np.int64), "created": np.zeros(T, np.bool_), "argmax": np.zeros((T, 3), np.int64),
           "n_exp": np.zeros(T, np.int64)}

    def finish(t):
        idx, created = node.pipe_finish(t % depth)
        rec["template"][t], rec["created"][t] = idx, created
        rec["argmax"][t] = node.pcn.max_pc
        rec["n_exp"][t] = len(node.em.experiences)

    for t in range(T):
        if t >= depth:
            finish(t - depth)
        node.pipe_submit(t % depth, (float(odom[t, 0]), float(odom[t, 1])), frames[t])
    for t in range(max(T - depth, 0), T):
        finish(t)
    rec["node"] = node
    return rec


def _native(frames, odom, energy, n_plans, **kw):
    from pyratslam_b200 import ros_simulate
    node = ros_simulate.RatslamRos(inject_energy=energy, **kw)
    res = node.replay_native(frames, odom, n_plans=n_plans)
    flat = res["argmax"]
    Y, Th = SHAPE[1], SHAPE[2]
    return {"template": res["template_index"].astype(np.int64), "created": res["created"] != 0,
            "argmax": np.stack([flat // (Y * Th), (flat // Th) % Y, flat % Th], axis=1), "n_exp": node._native_n_exp,
            "node": node}


def _locations(node):
    return [node.vts.templates[i].location() for i in range(len(node.vts.templates))]


def _check(rec, ref, shaped, tol, what):
    for k in ("template", "created", "argmax", "n_exp"):
        assert np.array_equal(np.asarray(rec[k]), ref[k]), (what, k)
    node = rec["node"]
    fs = node.pcn.posecells
    assert np.abs(fs - ref["final_state"]).max() / ref["final_state"].max() <= tol, what
    assert _locations(node) == _locations(shaped), what
    assert tuple(node.pcn.get_pc_max()) == tuple(shaped.pcn.get_pc_max()), what


def test_every_mode_matches_the_oracle():
    from oracle import drivers as odrv
    from pyratslam_b200 import ros_simulate
    T = 80
    frames, odom = _inputs(T)
    moved_by_injection = 0
    for energy in (0.02, 0.3):
        ref = odrv.replay_run(frames, odom, inject_energy=energy)
        moved_by_injection += _oracle_moves(frames, odom, energy)
        shaped = ros_simulate.replay(frames, odom, inject_energy=energy)
        _check(shaped, ref, shaped["node"], 1e-5, ("reference-shaped", energy))
        _check(ros_simulate.replay(frames, odom, fused=True, inject_energy=energy), ref, shaped["node"], 1e-5,
               ("fused", energy))
        _check(ros_simulate.replay(frames, odom, pipelined=True, inject_energy=energy), ref, shaped["node"], 1e-5,
               ("pipelined", energy))
        for depth in (1, 3):
            _check(_pipelined(frames, odom, energy, depth), ref, shaped["node"], 1e-5, ("pipelined", depth, energy))
        for n_plans in (1, 3):
            _check(_native(frames, odom, energy, n_plans), ref, shaped["node"], 1e-5, ("native", n_plans, energy))
        nat_rec = ros_simulate.replay(frames, odom, native=True, inject_energy=energy)
        for k in ("template", "created", "argmax", "n_exp", "em_xy"):
            assert np.array_equal(nat_rec[k], ref[k]), ("replay(native=True)", k, energy)
    # the O(1) arg-max update of the injection node is exercised, not bypassed
    assert moved_by_injection >= 1


def _frame_of(tpl):
    f = np.zeros((256, 256), np.uint8)
    f[np.ix_(ROWS, ROWS)] = tpl
    return f


def test_argmax_rule_on_crafted_states():
    """Ties at a lower / higher flat index than the arg-max, injection at the arg-max itself and a dead network: the
    cached arg-max the node leaves behind is numpy.argmax of the state (first maximum in C order)."""
    from pyratslam_b200 import ros_simulate
    rng = np.random.default_rng(41)
    lib = rng.integers(0, 256, (6, 32, 32), dtype=np.uint8)
    A, lo, hi = (15, 3, 7), (2, 5, 9), (18, 1, 1)
    locs = [lo, hi, A, (7, 7, 7), (0, 0, 0), (20, 20, 35)]
    node = ros_simulate.RatslamRos(inject_energy=0.25)
    node.vts.load_library(lib, locations=locs)

    def run(state, k):
        node.pcn.posecells = state
        idx, created = node.fused_frame(None, _frame_of(lib[k]))
        assert (idx, created) == (k, False)
        ps = node.pcn.posecells
        cached = int(node._f_pcwork[0].item())
        assert cached == int(np.argmax(ps)), (k, cached)
        assert tuple(node.pcn.get_pc_max()) == np.unravel_index(np.argmax(ps), SHAPE)
        # the next image-only frame reports the cached arg-max as the one its match was made with
        node.fused_frame(None, _frame_of(lib[3]))
        assert tuple(node.pcn.max_pc) == np.unravel_index(cached, SHAPE)
        return ps, cached

    base = np.zeros(SHAPE)
    base[A] = 0.5
    base[lo] = base[hi] = 0.25
    ps, c = run(base, 0)                                     # 0.25 + 0.25 == 0.5 at a lower flat index: moves
    assert ps[lo] == 0.5 and c == np.ravel_multi_index(lo, SHAPE)
    ps, c = run(base, 1)                                     # the same tie at a higher flat index: stays
    assert ps[hi] == 0.5 and c == np.ravel_multi_index(A, SHAPE)
    ps, c = run(base, 2)                                     # at the arg-max itself
    assert ps[A] == 0.75 and c == np.ravel_multi_index(A, SHAPE)
    ps, c = run(np.zeros(SHAPE), 5)                          # dead network: arg-max 0, then the injected cell
    assert c == np.ravel_multi_index((20, 20, 35), SHAPE)
    node.inject_energy = 0.0                                 # energy 0 into a dead network: numpy keeps index 0
    ps, c = run(np.zeros(SHAPE), 5)
    assert c == 0 and not ps.any()


def test_templates_appended_outside_the_plans():
    """vis_callback and load_library between plan frames (negative-index and out-of-bounds locations included), then
    plan frames that match those templates: each injects at its stored cell, as the reference-shaped calls do; the
    out-of-bounds one raises IndexError and leaves the state alone."""
    from pyratslam_b200 import ros_simulate
    T = 16
    frames, odom = _inputs(T)
    a, b = ros_simulate.RatslamRos(inject_energy=0.3), ros_simulate.RatslamRos(inject_energy=0.3)

    def plain(node, twist, im):
        if twist is not None:
            node.odom_callback(twist)
            node.spin_once()
        return node.vis_callback(im)

    def both(t, im, twist=None, fused=True):
        got = a.fused_frame(twist, im) if fused else a.vis_callback(im)
        want = plain(b, twist, im)
        assert got == want, (t, got, want)
        assert tuple(a.pcn.get_pc_max()) == tuple(b.pcn.get_pc_max()), t
        return got

    for t in range(6):
        both(t, frames[t], (float(odom[t, 0]), float(odom[t, 1])))
    i6, created = both(6, frames[6], fused=False)             # appended by the reference-shaped call
    assert created
    both(7, frames[8], (float(odom[7, 0]), float(odom[7, 1])))
    assert both(8, frames[6]) == (i6, False)                 # a plan frame matches it: injects at its stored cell
    rng = np.random.default_rng(42)
    lib = rng.integers(0, 256, (40, 32, 32), dtype=np.uint8)
    locs = np.zeros((40, 3))
    locs[:, 0], locs[:, 1], locs[:, 2] = np.arange(40) % 21, (3 * np.arange(40)) % 21, np.arange(40) % 36
    locs[5] = (-1, -2, -3)                                   # numpy negative indices: the cell (20, 19, 33)
    locs[6] = (4.7, -0.5, 35.2)                              # truncated: (4, 0, 35)
    locs[7] = (21, 0, 0)                                     # outside the grid
    for node in (a, b):
        node.vts.load_library(lib, locations=locs)
    for t, k in enumerate((5, 6, 12, 5, 39)):
        both(10 + t, _frame_of(lib[k]), (float(odom[t, 0]), float(odom[t, 1])) if t % 2 else None)
    before = a.pcn.posecells
    for node in (a, b):
        with pytest.raises(IndexError):
            if node is a:
                node.fused_frame(None, _frame_of(lib[7]))
            else:
                node.vis_callback(_frame_of(lib[7]))
    assert np.array_equal(a.pcn.posecells, before)
    both(20, frames[9], (float(odom[11, 0]), float(odom[11, 1])))   # the plans carry on after the error
    assert np.abs(a.pcn.posecells - b.pcn.posecells).max() <= 1e-5 * b.pcn.posecells.max()
    assert _locations(a) == _locations(b)


def test_float64_and_active_set():
    from oracle import drivers as odrv
    from pyratslam_b200 import ros_simulate
    T = 64
    frames, odom = _inputs(T)
    ref = odrv.replay_run(frames, odom, inject_energy=0.3)
    shaped = ros_simulate.replay(frames, odom, inject_energy=0.3, dtype=np.float64)
    _check(shaped, ref, shaped["node"], 1e-12, "float64 reference-shaped")
    _check(ros_simulate.replay(frames, odom, fused=True, inject_energy=0.3, dtype=np.float64), ref, shaped["node"],
           1e-12, "float64 fused")
    _check(_native(frames, odom, 0.3, 2, dtype=np.float64), ref, shaped["node"], 1e-12, "float64 native")
    dense = ros_simulate.replay(frames, odom, native=True, inject_energy=0.3)
    for kw in ({"fused": True}, {"native": True}, {"pipelined": True}):
        act = ros_simulate.replay(frames, odom, inject_energy=0.3, active_set=2, **kw)
        for k in ("template", "created", "argmax", "n_exp", "em_xy"):
            assert np.array_equal(act[k], dense[k]), (kw, k)
        assert np.abs(act["node"].pcn.posecells - ref["final_state"]).max() / ref["final_state"].max() <= 1e-5


def test_negative_energy():
    """fused_frame injects an energy < 0 on the host behind the frame (oracle parity); the pipelined and native replays,
    which inject on the device only, refuse it."""
    from oracle import drivers as odrv
    from pyratslam_b200 import ros_simulate
    T = 24
    frames, odom = _inputs(T)
    ref = odrv.replay_run(frames, odom, inject_energy=-0.01)
    rec = ros_simulate.replay(frames, odom, fused=True, inject_energy=-0.01)
    for k in ("template", "created", "argmax", "n_exp"):
        assert np.array_equal(rec[k], ref[k]), k
    assert np.abs(rec["node"].pcn.posecells - ref["final_state"]).max() / ref["final_state"].max() <= 1e-5
    for kw in ({"pipelined": True}, {"native": True}):
        with pytest.raises(ValueError):
            ros_simulate.replay(frames, odom, inject_energy=-0.01, **kw)
    node = ros_simulate.RatslamRos(inject_energy=-0.01)
    with pytest.raises(ValueError):
        node.replay_native(frames, odom)
