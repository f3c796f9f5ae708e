"""replay_ensemble: B agents with their own match threshold, global inhibition and injection energy over one recording,
each against the oracle's replay loop with that agent's parameters, across the pose-cell kernel families, and against
the single-agent native replay."""
import functools
import math

import numpy as np
import pytest

from synth import synth_frames

pytestmark = pytest.mark.gpu

SHAPE = (21, 21, 36)
THRESHOLDS = (0, 30000, 45000, 45000, 60000, 2 ** 32 - 1)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25, 0.3)          # 0.3: the network dies, its arg-max drops to (0, 0, 0)
MIXED = (None, 0.0, 0.02, 0.3, None, 0.3)


def _inputs(T, lag=1):
    """Frames with revisits of the frame `lag` steps back (every third frame), odometry with frames below the gate."""
    frames = synth_frames(np.random.default_rng(5), T)
    for t in range(4, T, 3):
        frames[t] = frames[t - lag]
    rng = np.random.default_rng(6)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    for t, still in ((9, (0.0005, -0.0002)), (10, (0.0, 0.0)), (30, (0.0, 0.0))):
        if t < T:
            odom[t] = still          # below the 0.001 gate: no pose-cell update for this frame
    return frames, odom


@functools.lru_cache(maxsize=None)
def _oracle(T, threshold, gi, energy):
    """oracle/drivers.py:replay_run with the agent's global inhibition, plus its library."""
    from oracle import drivers as odrv
    from oracle.posecells import PoseCellNetwork
    from oracle.view_templates import ViewTemplates
    frames, odom = _inputs(T)
    pcn = PoseCellNetwork(SHAPE, global_inhibition=gi)
    pcn.inject(1, tuple(math.floor(s / 2) for s in SHAPE))
    vts = ViewTemplates(odrv.X_RANGE, odrv.Y_RANGE, odrv.X_STEP, odrv.Y_STEP, 256, 256, threshold)
    rec = {"template": np.zeros(T, np.int64), "created": np.zeros(T, np.bool_), "argmax": np.zeros((T, 3), np.int64)}
    for t in range(T):
        lin, ang = float(odom[t, 0]), float(odom[t, 1])
        if abs(lin) > 0.001 or abs(ang) > 0.001:
            pcn.update((lin / odrv.ODOM_FREQ, ang / odrv.ODOM_FREQ))
        pc_max = pcn.get_pc_max()
        n0 = len(vts.templates)
        tm = vts.match(frames[t], pc_max[0], pc_max[1], pc_max[2])
        if energy is not None:
            pcn.inject(energy, tm.location())
        rec["template"][t], rec["created"][t], rec["argmax"][t] = tm.get_index(), len(vts.templates) > n0, pc_max
    rec["n_templates"] = len(vts.templates)
    rec["final_state"] = pcn.posecells
    rec["templates"] = np.stack([t.template for t in vts.templates])
    rec["locations"] = np.array([t.location() for t in vts.templates], dtype=np.int64)
    return rec


def _check_agent(out, b, ref, tol, what):
    for k in ("template", "created", "argmax"):
        assert np.array_equal(out[k][b], ref[k]), (what, b, k)
    assert out["n_templates"][b] == ref["n_templates"], (what, b)
    ag = out["agents"]
    assert np.array_equal(ag.templates(b), ref["templates"]), (what, b)
    assert np.array_equal(ag.locations(b), ref["locations"]), (what, b)
    fs, want = ag.posecells(b), ref["final_state"]
    scale = want.max() if want.max() > 0 else 1.0
    assert np.abs(fs - want).max() <= tol * scale, (what, b, np.abs(fs - want).max() / scale)


def test_six_agents_against_the_oracle():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 60
    frames, odom = _inputs(T)
    for energies in ((None,) * 6, MIXED):
        out = replay_ensemble(frames, odom, match_threshold=list(THRESHOLDS), global_inhibition=list(GIS),
                              inject_energy=list(energies))
        assert out["template"].shape == (6, T) and out["argmax"].shape == (6, T, 3)
        for b in range(6):
            _check_agent(out, b, _oracle(T, THRESHOLDS[b], GIS[b], energies[b]), 1e-5, ("float32", energies))
        assert tuple(out["argmax"][5, -1]) == (0, 0, 0)                   # gi = 0.3: the network died
        assert out["n_templates"][5] == 1 and out["n_templates"][0] > out["n_templates"][1]


def test_float64_ensemble():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 60
    frames, odom = _inputs(T)
    sel = (0, 2, 3, 4)
    energies = (None, 0.3, 0.02, None)
    out = replay_ensemble(frames, odom, match_threshold=[THRESHOLDS[i] for i in sel],
                          global_inhibition=[GIS[i] for i in sel], inject_energy=list(energies), dtype=np.float64)
    for j, i in enumerate(sel):
        _check_agent(out, j, _oracle(T, THRESHOLDS[i], GIS[i], energies[j]), 1e-12, "float64")


SETS = [(45000, 0.2, None), (0, 0.1, 0.02), (30000, 0.1745, 0.3), (60000, 0.25, 0.0), (2 ** 32 - 1, 0.05, 0.3)]


@pytest.mark.parametrize("B, path", [(1, "cluster"), (8, "cluster"), (60, "pair"), (300, "resident")])
def test_pose_cell_paths(B, path):
    """Parameter sets repeated round-robin: equal parameters give identical records and bit-identical states on every
    kernel family the ensemble's size selects, and one agent of each set equals the oracle."""
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 48
    frames, odom = _inputs(T)
    sets = [SETS[b % len(SETS)] for b in range(B)]
    out = replay_ensemble(frames, odom, match_threshold=[s[0] for s in sets], global_inhibition=[s[1] for s in sets],
                          inject_energy=[s[2] for s in sets])
    ag = out["agents"]
    assert ag.path == path
    state = ag.state.cpu().numpy()
    for b in range(B):
        first = b % len(SETS)
        if b == first:
            _check_agent(out, b, _oracle(T, *SETS[b]), 1e-5, ("path", path))
        else:
            for k in ("template", "created", "argmax"):
                assert np.array_equal(out[k][b], out[k][first]), (B, b, k)
            assert np.array_equal(state[b], state[first]), (B, b)


@pytest.mark.parametrize("links", [False, True])
def test_single_agent_equals_native_replay(links):
    from pyratslam_b200 import ros_simulate
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 60
    frames, odom = _inputs(T)
    for energy in (None, 0.3):
        want = ros_simulate.replay(frames, odom, native=True, inject_energy=energy, experience_links=links)
        out = replay_ensemble(frames, odom, inject_energy=energy, experience_map=True, experience_links=links)
        for k in ("template", "created", "argmax", "n_exp", "em_xy"):
            assert np.array_equal(out[k][0], want[k]), (links, energy, k)
        assert out["n_templates"][0] == want["n_templates"]
        node = want["node"]
        assert np.array_equal(out["agents"].locations(0),
                              np.array([t.location() for t in node.vts.templates], dtype=np.int64))
        fs = node.pcn.posecells
        assert np.abs(out["agents"].posecells(0) - fs).max() <= 1e-6 * fs.max()


def test_active_set_matches_dense():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 60
    frames, odom = _inputs(T)
    kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED))
    dense = replay_ensemble(frames, odom, **kw)
    act = replay_ensemble(frames, odom, active_set=2, **kw)
    for k in ("template", "created", "argmax", "n_templates"):
        assert np.array_equal(act[k], dense[k]), k
    for b in range(6):
        want = dense["agents"].posecells(b)
        assert np.abs(act["agents"].posecells(b) - want).max() <= 1e-5 * max(want.max(), 1.0)


def test_libraries_of_different_sizes():
    """A threshold-0 agent creates on most frames and spans several groups of 32 templates; in the same sweep another
    agent's library stays at one template."""
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 120
    frames, odom = _inputs(T)
    out = replay_ensemble(frames, odom, match_threshold=[0, 2 ** 32 - 1, 45000], inject_energy=[None, 0.3, 0.02])
    assert out["n_templates"][0] > 64 and out["n_templates"][1] == 1
    for b, (thr, energy) in enumerate(((0, None), (2 ** 32 - 1, 0.3), (45000, 0.02))):
        _check_agent(out, b, _oracle(T, thr, 0.2, energy), 1e-5, "sizes")


def test_lut_hole_raises_at_the_same_frame():
    from pyratslam_b200 import ros_simulate
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _inputs(30)
    bad = odom.copy()
    bad[20] = (1.0, 0.0)             # vtrans = 0.1 after the /10 scaling: the reference's LUT hole
    kw = dict(match_threshold=[45000, 0, 60000], global_inhibition=[0.2, 0.1, 0.25], inject_energy=[None, 0.3, 0.02])
    for T in (21, 30):
        with pytest.raises(KeyError):
            ros_simulate.replay(frames[:T], bad[:T], native=True)
        with pytest.raises(KeyError):
            replay_ensemble(frames[:T], bad[:T], **kw)
    out = replay_ensemble(frames[:20], bad[:20], **kw)        # the frames before it
    want = ros_simulate.replay(frames[:20], bad[:20], native=True)
    for k in ("template", "created", "argmax"):
        assert np.array_equal(out[k][0], want[k]), k


def test_invalid_arguments():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _inputs(8)
    for kw in ({"match_threshold": [1, 2], "global_inhibition": [0.1, 0.2, 0.3]}, {"inject_energy": [0.1, -0.1]},
               {"inject_energy": math.nan}, {"mode": "circular"}, {"n_agents": 2, "match_threshold": [1, 2, 3]}):
        with pytest.raises(ValueError):
            replay_ensemble(frames, odom, **kw)
    with pytest.raises(ValueError):
        replay_ensemble(frames[:, :128], odom)
    with pytest.raises(ValueError):
        replay_ensemble(frames, odom[:5])
