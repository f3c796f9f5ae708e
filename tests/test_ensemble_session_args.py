"""EnsembleSession without CUDA: the feed's input validation, the refusal of the host experience map, the library
growth rule, the chunked bag reader and the CLI's --chunk."""
import numpy as np
import pytest

from pyratslam_b200 import ros_ensemble
from pyratslam_b200.ros_ensemble import MAX_CAPACITY, EnsembleSession, capacity_for, feed_inputs, grow_capacity


def _frames(t):
    return np.zeros((t, 256, 256), np.uint8), np.zeros((t, 2))


def test_feed_inputs_one_recording():
    f, o = _frames(3)
    fr, od = feed_inputs(f, o, 1)
    assert len(fr) == 1 and fr[0].shape == (3, 256, 256) and od[0].dtype == np.float64
    fr, od = feed_inputs(*_frames(0), 1)
    assert fr[0].shape == (0, 256, 256)
    for bad in ((f.astype(np.int16), o), (f[:, :128], o), (f, o[:2]), (f, o[:, :1]), (f[0], o[:1]), ([f], [o]),
                (f, [[0.0, "x"]] * 3)):
        with pytest.raises(ValueError):
            feed_inputs(*bad, 1)


def test_feed_inputs_several_recordings():
    (f3, o3), (f0, o0) = _frames(3), _frames(0)
    fr, od = feed_inputs([f3, f0, f3[:1]], [o3, o0, o3[:1]], 3)
    assert [len(f) for f in fr] == [3, 0, 1] and [len(o) for o in od] == [3, 0, 1]
    for frames, odom in (((f3, f0), (o3,)),              # list lengths disagree
                         ((f3, f0), (o3, o0)),            # two recordings for a session of three
                         (f3, o3),                        # arrays for a session of three
                         ((f3, f0, f3), (o3, o0, o3[:2])),
                         ((f3, f0, f3.astype(np.float32)), (o3, o0, o3))):
        with pytest.raises(ValueError):
            feed_inputs(list(frames), list(odom), 3) if isinstance(frames, tuple) else feed_inputs(frames, odom, 3)


def test_session_refuses_the_host_experience_map_and_bad_arguments():
    for kw in ({"experience_map": True}, {"experience_map": "host"}, {"n_recordings": 0}, {"n_recordings": 1.5},
               {"capacity": 0}, {"capacity": MAX_CAPACITY + 1}, {"capacity": 33.5},
               {"n_recordings": 2, "recording": [0, 2]}, {"match_threshold": [1, 2], "global_inhibition": [1, 2, 3]}):
        with pytest.raises(ValueError):
            EnsembleSession(**kw)


def test_growth_rule_doubles():
    assert grow_capacity(32, 0, 20) == (32, 20)                 # fits: no growth
    assert grow_capacity(32, 10, 30) == (64, 30)                # doubled
    assert grow_capacity(64, 10, 500) == (capacity_for(510), 500)   # more than doubling needs
    assert grow_capacity(4096 + 32, 7, 4096) == (4096 + 32, 4096)   # templates, not frames, decide


def test_growth_rule_clamps_and_splits():
    assert grow_capacity(40000, 30000, 20000) == (MAX_CAPACITY, 20000)
    assert grow_capacity(MAX_CAPACITY, 65000, 1000) == (MAX_CAPACITY, 536)    # a sub-run that fits
    assert grow_capacity(60000, 65000, 1000) == (MAX_CAPACITY, 536)
    assert grow_capacity(MAX_CAPACITY, MAX_CAPACITY, 5) == (MAX_CAPACITY, 0)  # full: the session raises
    cap, n, t, runs = 32, 0, 70000, []
    while t:                    # the worst case, a template per frame, splits where the sweep's limit is reached
        cap, run = grow_capacity(cap, n, t)
        runs.append(run)
        n, t = n + run, t - run
        if n == MAX_CAPACITY:
            break
    assert cap == MAX_CAPACITY and sum(runs) == MAX_CAPACITY and t == 70000 - MAX_CAPACITY


@pytest.mark.parametrize("chunk", [1, 4, 5, 23, 100])
def test_iter_frames_equals_events_to_arrays(tmp_path, chunk):
    from pyratslam_b200 import rosbag_io as rb
    rng = np.random.default_rng(3)
    T = 23
    frames = rng.integers(0, 256, (T, 256, 256), dtype=np.uint8)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    path = str(tmp_path / "run.bag")
    rb.write_run(path, frames, odom)
    want_f, want_o, _ = rb.events_to_arrays(rb.read_events(path))
    pieces = list(rb.iter_frames(path, chunk))
    assert [len(f) for f, _ in pieces] == [min(chunk, T - i) for i in range(0, T, chunk)]
    assert np.array_equal(np.concatenate([f for f, _ in pieces]), want_f)
    assert np.array_equal(np.concatenate([o for _, o in pieces]), want_o)
    with pytest.raises(ValueError):
        next(rb.iter_frames(path, 0))


def test_cli_chunk(monkeypatch, capsys):
    calls = []

    def fake(bags, chunk, image_topic, odom_topic, recording, **kw):
        calls.append((list(bags), chunk, recording, kw["n_agents"]))
        B = kw["n_agents"]
        return np.arange(B), np.zeros(B, np.int64), np.array([7] * len(bags)), [(1, 2, 3)] * B, None
    monkeypatch.setattr(ros_ensemble, "_replay_chunked", fake)
    ros_ensemble.main(["a.bag", "b.bag", "--chunk", "256", "--match-threshold", "1,2"])
    assert calls == [(["a.bag", "b.bag"], 256, [0, 0, 1, 1], 4)]
    lines = capsys.readouterr().out.splitlines()
    assert len(lines) == 4 and lines[2].startswith("bag b.bag  agent 2  match_threshold 1 ")
    assert "created 0/7  final arg-max (1, 2, 3)" in lines[2]
    for bad in ("0", "-3", "x", "2.5"):
        with pytest.raises(SystemExit):
            ros_ensemble.main(["a.bag", "--chunk", bad])
