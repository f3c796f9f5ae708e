"""EnsembleSession: agents fed in pieces equal replay_ensemble on the concatenated recordings -- records, libraries,
locations, pose cells and linked device maps -- through library and map growth, over several recordings fed unevenly,
across recordings (continuation), beyond 65535 frames, and on a pose-cell error."""
import numpy as np
import pytest

from em_records import assert_same_map, loop_recording

pytestmark = pytest.mark.gpu

SHAPE = (21, 21, 36)
THRESHOLDS = (0, 30000, 45000, 45000, 60000, 2 ** 32 - 1)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25, 0.3)          # 0.3: the network dies
MIXED = (None, 0.0, 0.02, 0.3, None, 0.3)
MAP_KEYS = ("n_exp", "exp_id", "em_xy")


def _settings(B):
    return dict(match_threshold=[THRESHOLDS[b % 6] for b in range(B)], global_inhibition=[GIS[b % 6] for b in range(B)],
                inject_energy=[MIXED[b % 6] for b in range(B)])


def _feed(s, frames, odom, chunks):
    """Feed one recording in pieces of the given sizes (the last piece takes the rest); concatenated outputs."""
    outs, t = [], 0
    for n in list(chunks) + [len(frames)]:
        n = min(n, len(frames) - t)
        outs.append(s.feed(frames[t:t + n], odom[t:t + n]))
        t += n
    return {k: np.concatenate([o[k] for o in outs], axis=1) for k in ("template", "created", "argmax") + MAP_KEYS
            if k in outs[0]}


def _same(got, s, want, agents, what, maps=True):
    for k in ("template", "created", "argmax") + MAP_KEYS:
        if k in got:
            assert np.array_equal(got[k], want[k], equal_nan=True), (what, k)
    assert np.array_equal(s.n_templates, want["n_templates"]), what
    ag, wg = s.agents, want["agents"]
    assert ag.path == wg.path
    for b in agents:
        assert np.array_equal(ag.templates(b), wg.templates(b)), (what, b)
        assert np.array_equal(ag.locations(b), wg.locations(b)), (what, b)
        assert np.array_equal(ag.posecells(b), wg.posecells(b)), (what, b)
    if maps and "maps" in want:
        assert np.array_equal(s.n_loop_closures, want["n_loop_closures"]), what
        for b in agents:
            got_m, want_m = s.maps.experience_map(b), want["maps"].experience_map(b)
            assert_same_map(got_m, want_m, what=(what, b))
            got_m.iterate(5)
            want_m.iterate(5)
            assert_same_map(got_m, want_m, exact_th=False, what=(what, b, "iterate"))


@pytest.mark.parametrize("B, dtype, active_set, path", [(6, np.float32, 0, "cluster"), (6, np.float64, 0, None),
                                                        (60, np.float32, 0, "pair"), (300, np.float32, 0, "resident"),
                                                        (6, np.float32, 2, None)])
def test_chunked_equals_one_shot(B, dtype, active_set, path):
    from pyratslam_b200.ros_ensemble import EnsembleSession, replay_ensemble
    frames, odom = loop_recording(np.random.default_rng(3), 300)
    kw = dict(_settings(B), dtype=dtype, active_set=active_set, experience_map="device", experience_links=True)
    want = replay_ensemble(frames, odom, **kw)
    s = EnsembleSession(**kw)
    got = _feed(s, frames, odom, (1, 7, 64, 0))
    assert path is None or s.agents.path == path
    assert s.frames_fed.tolist() == [300]
    assert (want["n_loop_closures"] > 0).sum() >= 3
    _same(got, s, want, range(min(B, 6)), (B, dtype, active_set))
    s.close()
    with pytest.raises(RuntimeError):
        s.feed(frames[:1], odom[:1])


def test_growth_mid_session():
    """Threshold 0 creates a template on most frames: from 32 templates the libraries and the map workspace grow
    several times."""
    from test_gpu_ros_ensemble import _inputs
    from pyratslam_b200.ros_ensemble import EnsembleSession, replay_ensemble
    frames, odom = _inputs(300)
    kw = dict(_settings(6), experience_map="device", experience_links=True)
    want = replay_ensemble(frames, odom, **kw)
    s = EnsembleSession(capacity=32, **kw)
    caps, rows, outs = [], [], []
    for t in range(0, 300, 40):
        outs.append(s.feed(frames[t:t + 40], odom[t:t + 40]))
        caps.append(s.capacity)
        rows.append(s._E)
    assert len(set(caps)) >= 3 and caps == sorted(caps) and caps[-1] >= want["n_templates"].max(), caps
    assert len(set(rows)) >= 3, rows
    got = {k: np.concatenate([o[k] for o in outs], axis=1) for k in ("template", "created", "argmax") + MAP_KEYS}
    _same(got, s, want, range(6), "growth")


def _feed_unevenly(R, rec, **kw):
    """Every recording fed in four feeds of different sizes, some zero; per agent its concatenated records."""
    from test_gpu_multi_recording import _recording
    from pyratslam_b200.ros_ensemble import EnsembleSession
    s = EnsembleSession(n_recordings=R, recording=rec, **kw)
    plan = [(5, 0, 1, 30), (0, 0, 20, 0), (1, 0, 0, 7), (44, 0, 15, 7)]    # frames per recording in each feed
    t = [0] * R
    got = [{k: [] for k in ("template", "created", "argmax")} for _ in rec]
    for sizes in plan:
        fr, od = [], []
        for r in range(R):
            f, o = _recording(r)
            n = min(sizes[r], len(f) - t[r])
            fr.append(f[t[r]:t[r] + n])
            od.append(o[t[r]:t[r] + n])
            t[r] += n
        out = s.feed(fr, od)
        for b, r in enumerate(rec):
            L = out["length"][b]
            assert L == len(fr[r])
            for k in got[b]:
                got[b][k].append(out[k][b, :L])
            assert (out["template"][b, L:] == -1).all() and (out["argmax"][b, L:] == -1).all()
    assert t == [len(_recording(r)[0]) for r in range(R)] and s.frames_fed.tolist() == t
    return s, [{k: np.concatenate(v) for k, v in g.items()} for g in got]


def test_several_recordings_fed_unevenly():
    """The RECORDINGS of test_gpu_multi_recording.py (staggered stills, one empty) fed unevenly: every agent equals the
    native replay of its recording (float32) and the oracle (float64)."""
    from test_gpu_multi_recording import RECORDINGS, _oracle, _recording
    from pyratslam_b200 import ros_simulate
    R = len(RECORDINGS)
    rec = [3, 0, 2, 1, 0, 2, 3, 0, 2]
    thr = [THRESHOLDS[b % 6] for b in range(len(rec))]
    energy = [MIXED[b % 6] for b in range(len(rec))]
    s, got = _feed_unevenly(R, rec, match_threshold=thr, inject_energy=energy)
    for b, r in enumerate(rec):
        f, o = _recording(r)
        want = ros_simulate.replay(f, o, native=True, match_threshold=thr[b], inject_energy=energy[b]) if len(f) else None
        for k in ("template", "created", "argmax"):
            assert len(got[b][k]) == len(f) and (want is None or np.array_equal(got[b][k], want[k])), (b, k)
        assert s.n_templates[b] == (want["n_templates"] if want else 0)
        if want:
            fs = want["node"].pcn.posecells
            assert np.abs(s.agents.posecells(b) - fs).max() <= 1e-6 * fs.max(), b
    kw = _settings(len(rec))
    s, got = _feed_unevenly(R, rec, dtype=np.float64, **kw)
    ag = s.agents
    for b, r in enumerate(rec):
        ref = _oracle(r, THRESHOLDS[b % 6], GIS[b % 6], MIXED[b % 6])
        for k in ("template", "created", "argmax"):
            assert np.array_equal(got[b][k], ref[k]), (b, k)
        assert s.n_templates[b] == ref["n_templates"]
        assert np.array_equal(ag.templates(b), ref["templates"]) and np.array_equal(ag.locations(b), ref["locations"])
        scale = ref["final_state"].max() if ref["final_state"].max() > 0 else 1.0
        assert np.abs(ag.posecells(b) - ref["final_state"]).max() <= 1e-12 * scale, b


def test_continuation_across_recordings():
    from pyratslam_b200.ros_ensemble import EnsembleSession, replay_ensemble
    frames, odom = loop_recording(np.random.default_rng(3), 240)
    a, b = slice(0, 120), slice(120, 240)
    kw = dict(_settings(6), experience_map="device", experience_links=True)
    want = replay_ensemble(frames, odom, **kw)
    s = EnsembleSession(**kw)
    first = s.feed(frames[a], odom[a])
    after_a = s.n_loop_closures
    second = s.feed(frames[b], odom[b])
    assert (s.n_loop_closures > after_a).any()
    got = {k: np.concatenate([first[k], second[k]], axis=1) for k in ("template", "created", "argmax") + MAP_KEYS}
    _same(got, s, want, range(6), "continuation")
    unl = dict(_settings(6), experience_map="device")
    want = replay_ensemble(frames, odom, **unl)
    s = EnsembleSession(**unl)
    got = [s.feed(frames[a], odom[a]), s.feed(frames[b], odom[b])]
    for k in ("n_exp", "exp_id", "em_xy"):
        assert np.array_equal(np.concatenate([g[k] for g in got], axis=1), want[k]), k
    assert s.maps is None


def test_beyond_65535_frames():
    from synth import synth_frames
    from pyratslam_b200.ros_ensemble import EnsembleSession, capacity_for
    K, chunk, T = 20, 4096, 70000
    base = synth_frames(np.random.default_rng(8), K)
    s = EnsembleSession(match_threshold=0, global_inhibition=[0.1, 0.2, 0.25], inject_energy=[None, 0.3, 0.02])
    rng = np.random.default_rng(9)
    for t in range(0, T, chunk):
        n = min(chunk, T - t)
        odom = np.stack([rng.uniform(0, 3, n), rng.uniform(-1, 1, n)], axis=1)
        out = s.feed(base[np.arange(t, t + n) % K], odom)
        assert out["template"].shape == (3, n)
    assert s.frames_fed.tolist() == [T]
    assert (s.n_templates == K).all(), s.n_templates
    assert s.capacity == capacity_for(chunk + K - 1), s.capacity


def test_lut_hole_raises_and_closes():
    from test_gpu_ros_ensemble import _inputs
    from pyratslam_b200.ros_ensemble import EnsembleSession, replay_ensemble
    frames, odom = _inputs(40)
    bad = odom.copy()
    bad[20] = (1.0, 0.0)             # vtrans = 0.1 after the /10 scaling: the reference's LUT hole
    kw = dict(match_threshold=[45000, 0, 60000], global_inhibition=[0.2, 0.1, 0.25], inject_energy=[None, 0.3, 0.02])
    with pytest.raises(KeyError) as one:
        replay_ensemble(frames, bad, **kw)
    replay_ensemble(frames[:20], bad[:20], **kw)            # the frame before it is fine
    s = EnsembleSession(**kw)
    s.feed(frames[:8], bad[:8])
    s.feed(frames[8:16], bad[8:16])
    with pytest.raises(KeyError) as ses:
        s.feed(frames[16:24], bad[16:24])                    # the third chunk holds frame 20
    assert ses.value.args == one.value.args == ((5, 5),)
    with pytest.raises(RuntimeError):
        s.feed(frames[24:], bad[24:])
