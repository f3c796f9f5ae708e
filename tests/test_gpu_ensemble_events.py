"""Message-stream ensemble replay: every agent of replay_ensemble_events / EnsembleSession.feed_events equals the node's
message loop (ros_simulate.replay_events, or the oracle's replay_events_run for inhibitions the node cannot be given)
on streams with several twists per image, images without twists, gated-out twists and trailing odometry -- records,
libraries, locations, pose cells and maps -- across dtypes, pose-cell paths, injection, several recordings and
sessions fed in pieces."""
import functools

import numpy as np
import pytest

from em_records import assert_same_map, loop_recording
from event_oracle import replay_events_run

pytestmark = pytest.mark.gpu

THRESHOLDS = (0, 30000, 45000, 45000, 60000, 2 ** 32 - 1)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25, 0.3)          # 0.3: the network dies
MIXED = (None, 0.0, 0.02, 0.3, None, 0.3)
SETS = [(45000, 0.2, None), (0, 0.1, 0.02), (30000, 0.1745, 0.3), (60000, 0.25, 0.0), (2 ** 32 - 1, 0.05, 0.3)]


@functools.lru_cache(maxsize=None)
def _events(seed, T, lo=1, hi=4, trailing=3):
    """T images of a recording that closes loops, each after lo..hi twists (every seventh after none); one twist in
    eight is below the 0.001 gate; ``trailing`` twists after the last image."""
    rng = np.random.default_rng(seed)
    frames, odom = loop_recording(rng, T, moving=30, looping=30)
    ev, ns = [], 0

    def stamp():
        nonlocal ns
        ns += 1000
        return (ns // 10 ** 9, ns % 10 ** 9)
    for t in range(T):
        k = 0 if t % 7 == 3 else int(rng.integers(lo, hi + 1))
        for j in range(k):
            if rng.random() < 0.125:
                tw = (0.0005, 0.0)
            elif odom[t, 0] < 0.01:                  # a looping frame: stay just above the gate
                tw = (0.0015, 0.0)
            else:
                tw = (float(rng.uniform(0, 3)), float(rng.uniform(-1, 1)))
            ev.append(("odom", stamp(), tw))
        ev.append(("image", stamp(), frames[t]))
    for _ in range(trailing):
        ev.append(("odom", stamp(), (float(rng.uniform(0, 3)), float(rng.uniform(-1, 1)))))
    return tuple(ev)


@functools.lru_cache(maxsize=None)
def _node(key, threshold=45000, energy=None, links=False):
    from pyratslam_b200 import ros_simulate
    return ros_simulate.replay_events(list(_events(*key)), fused=False, match_threshold=threshold, inject_energy=energy,
                                      experience_links=links)


@functools.lru_cache(maxsize=None)
def _oracle(key, threshold, gi, energy):
    return replay_events_run(list(_events(*key)), match_threshold=threshold, global_inhibition=gi, inject_energy=energy)


def _check_node(out, b, node, what, tol=1e-6):
    for k in ("template", "created", "argmax"):
        assert np.array_equal(out[k][b, :out["length"][b]], node[k]), (what, b, k)
    assert out["n_templates"][b] == node["n_templates"], (what, b)
    ag, nd = out["agents"], node["node"]
    assert np.array_equal(ag.templates(b), np.stack([t.template for t in nd.vts.templates])), (what, b)
    assert np.array_equal(ag.locations(b), np.array([t.location() for t in nd.vts.templates], dtype=np.int64))
    fs = nd.pcn.posecells
    assert np.abs(ag.posecells(b) - fs).max() <= tol * fs.max(), (what, b)


def _check_oracle(out, b, ref, tol, what):
    for k in ("template", "created", "argmax"):
        assert np.array_equal(out[k][b, :out["length"][b]], ref[k]), (what, b, k)
    assert out["n_templates"][b] == ref["n_templates"], (what, b)
    ag = out["agents"]
    assert np.array_equal(ag.templates(b), ref["templates"]), (what, b)
    assert np.array_equal(ag.locations(b), ref["locations"]), (what, b)
    fs, want = ag.posecells(b), ref["final_state"]
    scale = want.max() if want.max() > 0 else 1.0
    assert np.abs(fs - want).max() <= tol * scale, (what, b, np.abs(fs - want).max() / scale)


@pytest.mark.parametrize("energies", [(None,) * 6, MIXED])
def test_agents_equal_their_message_loops(energies):
    from pyratslam_b200.ros_ensemble import replay_ensemble_events
    key = (1, 60)
    out = replay_ensemble_events(list(_events(*key)), match_threshold=list(THRESHOLDS), global_inhibition=list(GIS),
                                 inject_energy=list(energies), experience_map="device")
    assert out["template"].shape == (6, 60) and (out["length"] == 60).all()
    node = _node(key, THRESHOLDS[3], energies[3])
    _check_node(out, 3, node, energies)
    for b in range(6):
        _check_oracle(out, b, _oracle(key, THRESHOLDS[b], GIS[b], energies[b]), 1e-5, ("oracle", energies))
        assert np.array_equal(out["n_exp"][b], node["n_exp"]) and np.array_equal(out["em_xy"][b], node["em_xy"])
    ev = _events(*key)
    assert sum(e[0] == "odom" and max(map(abs, e[2])) > 0.001 for e in ev) > 60 + 30     # more updates than images


def test_float64():
    from pyratslam_b200.ros_ensemble import replay_ensemble_events
    key = (2, 40)
    sel = (0, 2, 3, 4)
    energies = (None, 0.3, 0.02, None)
    out = replay_ensemble_events(list(_events(*key)), match_threshold=[THRESHOLDS[i] for i in sel],
                                 global_inhibition=[GIS[i] for i in sel], inject_energy=list(energies),
                                 dtype=np.float64)
    for j, i in enumerate(sel):
        _check_oracle(out, j, _oracle(key, THRESHOLDS[i], GIS[i], energies[j]), 1e-12, "float64")


@pytest.mark.parametrize("B, path, active_set", [(8, "cluster", 0), (60, "pair", 0), (300, "resident", 0),
                                                 (6, None, 2)])
def test_pose_cell_paths_and_active_set(B, path, active_set):
    from pyratslam_b200.ros_ensemble import replay_ensemble_events
    key = (3, 40)
    sets = [SETS[b % len(SETS)] for b in range(B)]
    out = replay_ensemble_events(list(_events(*key)), match_threshold=[s[0] for s in sets],
                                 global_inhibition=[s[1] for s in sets], inject_energy=[s[2] for s in sets],
                                 active_set=active_set)
    ag = out["agents"]
    assert path is None or ag.path == path
    state = ag.state.cpu().numpy()
    _check_node(out, 0, _node(key, *SETS[0][::2]), path)
    for b in range(B):
        first = b % len(SETS)
        if b == first:
            _check_oracle(out, b, _oracle(key, *SETS[b]), 1e-5, (path, active_set))
        else:
            for k in ("template", "created", "argmax"):
                assert np.array_equal(out[k][b], out[k][first]), (B, b, k)
            assert np.array_equal(state[b], state[first]), (B, b)


def test_linked_maps_equal_the_node():
    from pyratslam_b200.ros_ensemble import replay_ensemble_events
    key = (4, 150)
    params = [(45000, None), (30000, 0.3), (60000, 0.02)]
    out = replay_ensemble_events(list(_events(*key)), match_threshold=[p[0] for p in params],
                                 inject_energy=[p[1] for p in params], experience_map="device", experience_links=True)
    closed = 0
    for b, (thr, energy) in enumerate(params):
        node = _node(key, thr, energy, True)
        _check_node(out, b, node, ("links", b))
        assert np.array_equal(out["n_exp"][b], node["n_exp"]), b
        assert np.abs(out["em_xy"][b] - node["em_xy"]).max() <= 1e-9, b
        em = node["node"].em
        assert out["n_loop_closures"][b] == em.n_loop_closures
        closed += em.n_loop_closures > 0
        got = out["maps"].experience_map(b)
        assert_same_map(got, em, what=b)
        got.iterate(5)
        em.iterate(5)
        assert_same_map(got, em, exact_th=False, what=(b, "iterate"))
    assert closed >= 1


def test_four_recordings_at_different_rates():
    from pyratslam_b200.ros_ensemble import replay_ensemble_events
    keys = [(5, 30, 1, 1, 0), (6, 24, 3, 3, 2), (7, 40, 0, 2, 5), (8, 12, 5, 5, 1)]
    streams = [list(_events(*k)) for k in keys]
    rec = [0, 1, 2, 3, 3, 2, 1, 0]
    sets = [SETS[b % len(SETS)] for b in range(8)]
    kw = dict(match_threshold=[s[0] for s in sets], global_inhibition=[s[1] for s in sets],
              inject_energy=[s[2] for s in sets], experience_map="device", experience_links=True)
    out = replay_ensemble_events(streams, recording=rec, **kw)
    assert out["length"].tolist() == [keys[r][1] for r in rec] and out["template"].shape == (8, 40)
    for b, r in enumerate(rec):
        one = replay_ensemble_events(streams[r], **{k: (v[b] if isinstance(v, list) else v) for k, v in kw.items()})
        L = out["length"][b]
        for k in ("template", "created", "argmax", "n_exp", "exp_id", "em_xy"):
            assert np.array_equal(out[k][b, :L], one[k][0]), (b, k)
        assert (out["template"][b, L:] == -1).all() and np.isnan(out["em_xy"][b, L:]).all()
        assert out["n_templates"][b] == one["n_templates"][0]
        want = one["agents"].posecells(0)
        assert np.abs(out["agents"].posecells(b) - want).max() <= 1e-6 * max(want.max(), 1.0), b
        assert_same_map(out["maps"].experience_map(b), one["maps"].experience_map(0), what=b)
        if sets[b] == SETS[0]:
            _check_node(out, b, _node(keys[r], 45000, None, True), ("recording", r))


def _cut(events, cuts):
    return [list(events[i:j]) for i, j in zip((0,) + cuts, cuts + (len(events),))]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_session_in_pieces_equals_one_call(dtype):
    from pyratslam_b200 import rosbag_io as rb
    from pyratslam_b200.ros_ensemble import EnsembleSession, replay_ensemble_events
    head = (9, 20, 1, 1, 0)                  # alternates: fed as arrays with feed
    ev = list(_events(*head)) + list(_events(10, 80))
    kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED), dtype=dtype,
              experience_map="device", experience_links=True)
    want = replay_ensemble_events(ev, **kw)
    n_head = len(_events(*head))
    rest = ev[n_head:]
    odom_runs = [i for i in range(1, len(rest) - 1) if rest[i][0] == rest[i - 1][0] == "odom"]
    cuts = (1, odom_runs[0], odom_runs[3], odom_runs[3] + 1, odom_runs[20], len(rest) - 2)   # inside odometry runs
    s = EnsembleSession(capacity=32, **kw)
    frames, odom, _ = rb.events_to_arrays(ev[:n_head])
    outs = [s.feed(frames, odom)]
    outs += [s.feed_events(p) for p in _cut(rest, cuts)]
    assert s.capacity > 32 and s.frames_fed.tolist() == [100]
    for k in ("template", "created", "argmax", "n_exp", "exp_id", "em_xy"):
        got = np.concatenate([o[k] for o in outs], axis=1)
        assert np.array_equal(got, want[k]), k
    assert np.array_equal(s.n_templates, want["n_templates"])
    assert np.array_equal(s.n_loop_closures, want["n_loop_closures"])
    ag, wg = s.agents, want["agents"]
    for b in range(6):
        assert np.array_equal(ag.templates(b), wg.templates(b)), b
        assert np.array_equal(ag.locations(b), wg.locations(b)), b
        assert np.array_equal(ag.posecells(b), wg.posecells(b)), b
        got_m, want_m = s.maps.experience_map(b), want["maps"].experience_map(b)
        assert_same_map(got_m, want_m, what=b)
        got_m.iterate(5)
        want_m.iterate(5)
        assert_same_map(got_m, want_m, exact_th=False, what=(b, "iterate"))
    s.close()
    with pytest.raises(RuntimeError):
        s.feed_events(rest[:2])


def test_alternating_stream_equals_replay_ensemble():
    from pyratslam_b200 import rosbag_io as rb
    from pyratslam_b200.ros_ensemble import replay_ensemble, replay_ensemble_events
    ev = list(_events(11, 120, 1, 1, 0))
    frames, odom, _ = rb.events_to_arrays(ev)
    kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED),
              experience_map="device", experience_links=True)
    want = replay_ensemble(frames, odom, **kw)
    got = replay_ensemble_events(ev, **kw)
    for k in ("template", "created", "argmax", "n_exp", "exp_id", "em_xy", "n_templates", "n_loop_closures"):
        assert np.array_equal(got[k], want[k]), k
    for b in range(6):
        assert np.array_equal(got["agents"].posecells(b), want["agents"].posecells(b)), b
        assert_same_map(got["maps"].experience_map(b), want["maps"].experience_map(b), what=b)


def test_lut_hole_on_an_odometry_only_tick():
    from pyratslam_b200 import ros_simulate
    from pyratslam_b200.ros_ensemble import replay_ensemble_events
    ev = list(_events(12, 20, 2, 2, 0))
    img = [i for i, e in enumerate(ev) if e[0] == "image"]
    i = img[11] - 2                               # the first of two twists before image 11: an odometry-only tick
    assert ev[i][0] == ev[i + 1][0] == "odom"
    bad = ev[:i] + [("odom", ev[i][1], (1.0, 0.0))] + ev[i + 1:]       # vtrans = 0.1: the reference's LUT hole
    kw = dict(match_threshold=[45000, 0, 60000], global_inhibition=[0.2, 0.1, 0.25], inject_energy=[None, 0.3, 0.02])
    for stream in (bad, ev + [("odom", ev[-1][1], (1.0, 0.0))]):       # mid-stream and in trailing odometry
        with pytest.raises(KeyError):
            ros_simulate.replay_events(stream)
        with pytest.raises(KeyError):
            replay_ensemble_events(stream, **kw)


def test_cli_all_messages_reports_what_the_node_reports(tmp_path, capsys):
    from pyratslam_b200 import ros_ensemble, ros_simulate
    from pyratslam_b200 import rosbag_io as rb
    path = str(tmp_path / "run.bag")
    rb.write_events(path, list(_events(13, 40, 3, 3, 2)))
    want = ros_simulate.replay_bag(path)
    for extra in ([], ["--chunk", "7"]):
        ros_ensemble.main([path, "--all-messages"] + extra)
        line = capsys.readouterr().out.strip()
        assert ("templates %d " % want["n_templates"]) in line and ("created %d/40 " % want["created"].sum()) in line
        assert line.endswith("experiences %d" % len(want["node"].em.experiences)), line
