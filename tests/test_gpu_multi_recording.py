"""replay_ensemble over several recordings: agent b replays recording[b] with its own parameters.  Every agent against
the oracle's replay loop and the native replay on its own recording, across the pose-cell kernel families, with the
active set, after its recording has ended, with linked experience maps, and with a LUT hole in one recording."""
import functools
import math

import numpy as np
import pytest

from em_records import assert_same_map, host_maps, loop_recording
from synth import synth_frames

pytestmark = pytest.mark.gpu

SHAPE = (21, 21, 36)
# the settings of test_gpu_ros_ensemble.py: gi = 0.3 kills the network, MIXED mixes injection and none
THRESHOLDS = (0, 30000, 45000, 45000, 60000, 2 ** 32 - 1)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25, 0.3)
MIXED = (None, 0.0, 0.02, 0.3, None, 0.3)
SETS = [(45000, 0.2, None), (0, 0.1, 0.02), (30000, 0.1745, 0.3), (60000, 0.25, 0.0), (2 ** 32 - 1, 0.05, 0.3)]

# (seed, length, still frames): the stills differ per recording, so frames occur where some recordings move and others
# do not; one recording is empty
RECORDINGS = ((5, 50, (9, 10, 30)), (11, 0, ()), (7, 36, (3, 17, 18, 19)), (13, 44, (0, 25)))


@functools.lru_cache(maxsize=None)
def _recording(r):
    """Frames with revisits of the frame before last (every third frame) and odometry with still frames."""
    seed, T, still = RECORDINGS[r]
    rng = np.random.default_rng(seed)
    frames = synth_frames(rng, T) if T else np.zeros((0, 256, 256), np.uint8)
    for t in range(4, T, 3):
        frames[t] = frames[t - 2]
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    for t in still:
        odom[t] = (0.0005, -0.0002) if t % 2 else (0.0, 0.0)      # below the 0.001 gate
    return frames, odom


def _lists(rs):
    return [_recording(r)[0] for r in rs], [_recording(r)[1] for r in rs]


@functools.lru_cache(maxsize=None)
def _oracle(r, threshold, gi, energy, dtype=np.float64):
    """oracle/drivers.py:replay_run on recording r with the agent's parameters, plus its library."""
    from oracle import drivers as odrv
    from oracle.posecells import PoseCellNetwork
    from oracle.view_templates import ViewTemplates
    frames, odom = _recording(r)
    T = len(frames)
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
    rec["templates"] = (np.stack([t.template for t in vts.templates]) if vts.templates
                        else np.zeros((0, 32, 32), np.uint8))
    rec["locations"] = np.array([t.location() for t in vts.templates], dtype=np.int64).reshape(-1, 3)
    return rec


def _check_agent(out, b, ref, tol, what):
    L = len(ref["template"])
    assert out["length"][b] == L, (what, b)
    for k in ("template", "created", "argmax"):
        assert np.array_equal(out[k][b, :L], ref[k]), (what, b, k)
    assert (out["template"][b, L:] == -1).all() and not out["created"][b, L:].any(), (what, b)
    assert (out["argmax"][b, L:] == -1).all(), (what, b)
    assert out["n_templates"][b] == ref["n_templates"], (what, b)
    ag = out["agents"]
    assert np.array_equal(ag.templates(b), ref["templates"]), (what, b)
    assert np.array_equal(ag.locations(b), ref["locations"]), (what, b)
    fs, want = ag.posecells(b), ref["final_state"]
    scale = want.max() if want.max() > 0 else 1.0
    assert np.abs(fs - want).max() <= tol * scale, (what, b, np.abs(fs - want).max() / scale)


# interleaved, not sorted: recordings 0, 2 and 1 (empty) alternate over the agents
REC3 = (0, 2, 1, 2, 0, 0, 2, 1, 0)
REC3_LISTS = (0, 1, 2)


def test_agents_against_the_oracle():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _lists(REC3_LISTS)
    B = len(REC3)
    for energies in ((None,) * 6, MIXED):
        kw = dict(match_threshold=[THRESHOLDS[b % 6] for b in range(B)], global_inhibition=[GIS[b % 6] for b in range(B)],
                  inject_energy=[energies[b % 6] for b in range(B)])
        out = replay_ensemble(frames, odom, recording=list(REC3), **kw)
        assert out["template"].shape == (B, 50) and out["argmax"].shape == (B, 50, 3)
        for b, r in enumerate(REC3):
            _check_agent(out, b, _oracle(r, THRESHOLDS[b % 6], GIS[b % 6], energies[b % 6]), 1e-5, ("float32", energies))
        assert tuple(out["argmax"][5, 49]) == (0, 0, 0)                   # gi = 0.3 on recording 0: the network died


def test_float64_against_the_oracle():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _lists(REC3_LISTS)
    sel = (0, 2, 3, 4, 1)
    rec = (2, 0, 1, 2, 0)
    energies = (None, 0.3, 0.02, None, 0.02)
    out = replay_ensemble(frames, odom, recording=list(rec), match_threshold=[THRESHOLDS[i] for i in sel],
                          global_inhibition=[GIS[i] for i in sel], inject_energy=list(energies), dtype=np.float64)
    for j, i in enumerate(sel):
        _check_agent(out, j, _oracle(rec[j], THRESHOLDS[i], GIS[i], energies[j]), 1e-12, "float64")


def test_one_recording_as_a_list_equals_the_array_form():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _recording(0)
    kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED),
              experience_map="device", experience_links=True)
    a = replay_ensemble(frames, odom, **kw)
    m = replay_ensemble([frames], [odom], recording=0, **kw)
    for k in ("template", "created", "argmax", "n_templates", "n_exp", "exp_id", "em_xy", "n_loop_closures"):
        assert np.array_equal(a[k], m[k]), k
    assert (m["length"] == len(frames)).all()
    assert np.array_equal(a["agents"].state.cpu().numpy(), m["agents"].state.cpu().numpy())
    for b in range(6):
        assert np.array_equal(a["agents"].locations(b), m["agents"].locations(b))


def test_agents_equal_the_native_replay():
    from pyratslam_b200 import ros_simulate
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _lists((0, 2, 3))
    rec = (2, 0, 1, 0, 2, 1)
    thr = (45000, 30000, 45000, 60000, 0, 30000)
    energy = (None, 0.3, 0.02, None, 0.3, None)
    out = replay_ensemble(frames, odom, recording=list(rec), match_threshold=list(thr), inject_energy=list(energy),
                          experience_map=True)
    for b, r in enumerate(rec):
        want = ros_simulate.replay(frames[r], odom[r], native=True, match_threshold=thr[b], inject_energy=energy[b])
        L = len(frames[r])
        for k in ("template", "created", "argmax", "n_exp", "em_xy"):
            assert np.array_equal(out[k][b, :L], want[k]), (b, k)
        assert out["n_templates"][b] == want["n_templates"]
        fs = want["node"].pcn.posecells
        assert np.abs(out["agents"].posecells(b) - fs).max() <= 1e-6 * fs.max(), b


@pytest.mark.parametrize("B, path", [(8, "cluster"), (60, "pair"), (300, "resident")])
def test_pose_cell_paths(B, path):
    """Four recordings with staggered stops and ends (so mixed frames occur on every path), parameter sets round-robin:
    equal (set, recording) pairs give identical records and bit-identical states, and one agent of each pair equals
    the oracle."""
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _lists((0, 2, 3, 1))
    rec = [(b * 3) % 4 for b in range(B)]
    sets = [SETS[(b // 4) % len(SETS)] for b in range(B)]
    out = replay_ensemble(frames, odom, recording=rec, match_threshold=[s[0] for s in sets],
                          global_inhibition=[s[1] for s in sets], inject_energy=[s[2] for s in sets])
    ag = out["agents"]
    assert ag.path == path
    state = ag.state.cpu().numpy()
    first = {}
    lists = (0, 2, 3, 1)
    for b in range(B):
        key = (sets[b], rec[b])
        if key not in first:
            first[key] = b
            _check_agent(out, b, _oracle(lists[rec[b]], *sets[b]), 1e-5, ("path", path))
        else:
            f = first[key]
            for k in ("template", "created", "argmax"):
                assert np.array_equal(out[k][b], out[k][f]), (B, b, k)
            assert np.array_equal(state[b], state[f]), (B, b)


def test_active_set_matches_dense():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _lists(REC3_LISTS)
    B = len(REC3)
    kw = dict(recording=list(REC3), match_threshold=[THRESHOLDS[b % 6] for b in range(B)],
              global_inhibition=[GIS[b % 6] for b in range(B)], inject_energy=[MIXED[b % 6] for b in range(B)])
    dense = replay_ensemble(frames, odom, **kw)
    act = replay_ensemble(frames, odom, active_set=2, **kw)
    for k in ("template", "created", "argmax", "n_templates"):
        assert np.array_equal(act[k], dense[k]), k
    for b in range(B):
        want = dense["agents"].posecells(b)
        assert np.abs(act["agents"].posecells(b) - want).max() <= 1e-5 * max(want.max(), 1.0)


def test_ended_recordings_keep_their_state():
    """The agents of a recording that ended long before the others keep the library, locations and pose cells they had
    at its end: the same as replaying that recording alone with the same agents."""
    from pyratslam_b200.ros_ensemble import replay_ensemble
    long_f, long_o = _recording(0)
    short_f, short_o = long_f[:12], long_o[:12]
    kw = dict(match_threshold=[45000, 0, 30000, 45000], global_inhibition=[0.2, 0.1, 0.1745, 0.2],
              inject_energy=[None, 0.02, 0.3, 0.3])
    both = replay_ensemble([long_f, short_f], [long_o, short_o], recording=[1, 0, 1, 1], **kw)
    alone = replay_ensemble([short_f], [short_o], recording=[0, 0, 0, 0], **kw)
    for b in (0, 2, 3):
        assert both["length"][b] == 12
        for k in ("template", "created", "argmax"):
            assert np.array_equal(both[k][b, :12], alone[k][b]), (b, k)
        assert both["n_templates"][b] == alone["n_templates"][b]
        assert np.array_equal(both["agents"].templates(b), alone["agents"].templates(b))
        assert np.array_equal(both["agents"].locations(b), alone["agents"].locations(b))
        want = alone["agents"].posecells(b)
        assert np.abs(both["agents"].posecells(b) - want).max() <= 1e-6 * want.max(), b


def test_linked_experience_maps_against_the_host():
    """Device maps of agents on three loop-closing recordings of different lengths against host linked maps over each
    agent's own records and odometry: structure exact, floats within 1e-9, before and after iterate(5); past an agent's
    length n_exp and exp_id are -1 and em_xy NaN."""
    from pyratslam_b200.ros_ensemble import replay_ensemble
    recs = [loop_recording(np.random.default_rng(s), T) for s, T in ((3, 240), (4, 170), (9, 200))]
    frames, odom = [f for f, _ in recs], [o for _, o in recs]
    rec = [1, 0, 2, 0, 1, 2]
    kw = dict(recording=rec, match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED))
    dev = replay_ensemble(frames, odom, experience_map="device", experience_links=True, **kw)
    host = replay_ensemble(frames, odom, experience_map=True, experience_links=True, **kw)
    for k in ("template", "created", "argmax", "n_exp"):
        assert np.array_equal(dev[k], host[k]), k
    assert np.array_equal(np.isnan(dev["em_xy"]), np.isnan(host["em_xy"]))
    assert np.nanmax(np.abs(dev["em_xy"] - host["em_xy"])) <= 1e-9
    closing = 0
    for b, r in enumerate(rec):
        L = len(frames[r])
        maps, n_exp, exp_id, em_xy = host_maps(dev["template"][b:b + 1, :L], dev["argmax"][b:b + 1, :L], odom[r], SHAPE)
        assert np.array_equal(dev["n_exp"][b, :L], n_exp[0]) and np.array_equal(dev["exp_id"][b, :L], exp_id[0]), b
        assert np.abs(dev["em_xy"][b, :L] - em_xy[0]).max() <= 1e-9, b
        assert (dev["n_exp"][b, L:] == -1).all() and (dev["exp_id"][b, L:] == -1).all()
        assert np.isnan(dev["em_xy"][b, L:]).all()
        assert dev["n_loop_closures"][b] == maps[0].n_loop_closures, b
        got, want = dev["maps"].experience_map(b), maps[0]
        assert_same_map(got, want, what=b)
        got.iterate(5)
        want.iterate(5)
        assert_same_map(got, want, exact_th=False, what=(b, "iterate"))
        closing += want.n_loop_closures > 0
    assert closing >= 3
    unl = replay_ensemble(frames, odom, experience_map="device", **kw)
    unl_host = replay_ensemble(frames, odom, experience_map=True, **kw)
    for k in ("n_exp", "em_xy"):
        assert np.array_equal(unl[k], unl_host[k], equal_nan=True), k


def test_lut_hole_in_one_recording_raises_like_its_native_replay():
    from pyratslam_b200 import ros_simulate
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = _lists((0, 2))
    bad = odom[1].copy()
    bad[20] = (1.0, 0.0)             # vtrans = 0.1 after the /10 scaling: the reference's LUT hole
    with pytest.raises(KeyError) as native:
        ros_simulate.replay(frames[1], bad, native=True)
    kw = dict(recording=[0, 1, 0, 1], match_threshold=[45000, 0, 60000, 45000], global_inhibition=[0.2, 0.1, 0.25, 0.2],
              inject_energy=[None, 0.3, 0.02, None])
    with pytest.raises(KeyError) as ens:
        replay_ensemble(frames, [odom[0], bad], **kw)
    assert ens.value.args == native.value.args == ((5, 5),)
    out = replay_ensemble(frames, odom, **kw)          # the same agents without the hole run through
    assert (out["length"] == [50, 36, 50, 36]).all()
