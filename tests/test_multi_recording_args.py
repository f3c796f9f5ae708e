"""replay_ensemble over several recordings, without a GPU: the `recording` argument's broadcasting and validation, the
list forms of frames and odom (all checked before the first CUDA call), the per-recording unlinked dead reckoning and
the command line's cross product of bags and settings."""
import numpy as np
import pytest

from pyratslam_b200 import experience_ensemble as xens
from pyratslam_b200 import ros_ensemble
from pyratslam_b200.experience_map import ExperienceMap


def test_recording_broadcasting():
    assert ros_ensemble.agent_recordings(0, 3, 1).tolist() == [0, 0, 0]
    assert ros_ensemble.agent_recordings(np.int64(2), 2, 3).tolist() == [2, 2]
    rec = ros_ensemble.agent_recordings([2, 0, 1, 0], 4, 3)
    assert rec.dtype == np.int64 and rec.tolist() == [2, 0, 1, 0]
    assert ros_ensemble.agent_recordings(np.array([1, 1]), 2, 2).tolist() == [1, 1]
    assert ros_ensemble._recording_count(0) is None and ros_ensemble._recording_count([0, 1, 1]) == 3


@pytest.mark.parametrize("recording, B, R", [
    (3, 2, 3),                # out of range
    (-1, 2, 3),
    ([0, 1], 3, 2),           # length disagrees with B
    ([0, 2], 2, 2),
    ([0, 1.0], 2, 2),         # not integers
    (True, 2, 2),
    ("0", 1, 1),
    (None, 1, 1),
])
def test_invalid_recordings(recording, B, R):
    with pytest.raises(ValueError):
        ros_ensemble.agent_recordings(recording, B, R)


def _rec(T):
    return np.zeros((T, 256, 256), np.uint8), np.zeros((T, 2))


def _lists(*Ts):
    recs = [_rec(T) for T in Ts]
    return [f for f, _ in recs], [o for _, o in recs]


@pytest.mark.parametrize("args, kw", [
    (_lists(4, 3), {"recording": [0, 2]}),                                  # index out of range
    (_lists(4, 3), {"recording": [0, 1, 1], "match_threshold": [1, 2]}),   # recording and parameters disagree
    (_lists(4, 3), {"recording": [0, 1], "n_agents": 3}),                   # recording and n_agents disagree
    (_lists(4, 3), {"recording": [0, 1.5]}),
    ((_lists(4, 3)[0], _lists(4)[1]), {}),                                  # list lengths disagree
    ((_lists(4, 3)[0], _rec(4)[1]), {}),                                    # odom not a list
    ((_lists(4, 3)[0], [np.zeros((4, 2)), np.zeros((2, 2))]), {}),         # odom length of recording 1
    (([np.zeros((4, 256, 256), np.uint8), np.zeros((3, 128, 128), np.uint8)], _lists(4, 3)[1]), {}),  # bad shape
    (([np.zeros((4, 256, 256), np.uint8), np.zeros((3, 256, 256), np.float32)], _lists(4, 3)[1]), {}),
    (([np.zeros((4, 256, 256), np.uint8), np.zeros((3, 256, 256), np.uint8)], [np.zeros((4, 2)), np.zeros((3, 3))]),
     {}),
    (_rec(4), {"recording": 1}),                                            # single arrays take recording 0 only
    (_rec(4), {"recording": [0, 1]}),
    (_lists(4, 3), {"recording": [0, 1], "inject_energy": [0.1, -1.0]}),
    (_lists(4, 3), {"recording": 1, "mode": "circular"}),
    (([np.broadcast_to(np.zeros((1, 256, 256), np.uint8), (1 << 16, 256, 256)), np.zeros((2, 256, 256), np.uint8)],
      [np.zeros((1 << 16, 2)), np.zeros((2, 2))]), {"recording": [0, 1]}),   # the longest recording is too long
])
def test_multi_replay_refuses_before_any_cuda_call(args, kw, monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("CUDA was touched before the arguments were checked")
    monkeypatch.setattr(ros_ensemble.nat, "require_cuda", no_cuda)
    monkeypatch.setattr(ros_ensemble.nat, "lib", no_cuda)
    with pytest.raises(ValueError):
        ros_ensemble.replay_ensemble(*args, **kw)


def test_a_list_of_single_frames_is_still_one_recording(monkeypatch):
    """A list of 2-D frames is one recording as before (the list form is a list of 3-D recordings)."""
    seen = {}

    def stop(*a, **k):
        seen["cuda"] = True
        raise RuntimeError("stop")
    monkeypatch.setattr(ros_ensemble.nat, "require_cuda", stop)
    with pytest.raises(RuntimeError):
        ros_ensemble.replay_ensemble([np.zeros((256, 256), np.uint8)] * 3, np.zeros((3, 2)))
    assert seen["cuda"]


def _host_dead_reckoning(odom):
    em = ExperienceMap()
    n, xy = [], []
    for lin, ang in odom:
        if abs(lin) > 0.001 or abs(ang) > 0.001:
            em.update(lin / 10.0, ang / 10.0, (0, 0, 0))
        n.append(len(em.experiences))
        xy.append(em.get_current_point() if em.current_exp is not None else (0.0, 0.0))
    return np.array(n), np.array(xy).reshape(-1, 2)


def test_unlinked_maps_per_recording():
    """Without links each recording's dead reckoning is computed once and broadcast to its agents; past a recording's
    end the map stays as it was (the frames there are not-moved frames)."""
    rng = np.random.default_rng(8)
    lengths = (30, 0, 12)
    odoms = [np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1) for T in lengths]
    odoms[0][[3, 4, 20]] = 0.0
    odoms[2][7] = (0.0005, 0.0)
    T, R = max(lengths), len(lengths)
    moved, tw = np.zeros((T, R), np.uint8), np.zeros((T, R, 2))
    for r, o in enumerate(odoms):
        moved[:len(o), r], tw[:len(o), r] = xens.gate(o)
    rec_of = np.array([2, 0, 1, 2, 0])
    out = xens._maps(np.full((T, 5), -1), np.zeros((T, 5), np.int64), moved, tw, (21, 21, 36), False, 1.0, 0.5,
                     rec_of=rec_of)
    assert out["maps"] is None and not out["n_loop_closures"].any()
    for b, r in enumerate(rec_of):
        n, xy = _host_dead_reckoning(odoms[r])
        L = len(odoms[r])
        assert np.array_equal(out["n_exp"][b, :L], n) and np.array_equal(out["em_xy"][b, :L], xy), b
        assert np.array_equal(out["exp_id"][b], out["n_exp"][b] - 1)
        if L:
            assert (out["n_exp"][b, L:] == n[-1]).all() and (out["em_xy"][b, L:] == xy[-1]).all()
        else:
            assert not out["n_exp"][b].any() and not out["em_xy"][b].any()


def _fake_cli(monkeypatch, bags):
    """main() with the bags and the replay replaced: returns the replay's calls."""
    from pyratslam_b200 import rosbag_io
    lengths = {name: T for name, T in bags}
    monkeypatch.setattr(rosbag_io, "read_events", lambda bag, **kw: bag)
    monkeypatch.setattr(rosbag_io, "events_to_arrays",
                        lambda bag: (np.full((lengths[bag], 256, 256), len(bag), np.uint8),
                                     np.zeros((lengths[bag], 2)), None))
    calls = []

    def fake(frames, odom, n_agents=None, recording=0, **kw):
        calls.append(dict(frames=frames, odom=odom, n_agents=n_agents, recording=recording, **kw))
        T = max(len(f) for f in frames) if isinstance(frames, list) else len(frames)
        return {"argmax": np.zeros((n_agents, T, 3), np.int64), "n_templates": np.arange(n_agents),
                "created": np.zeros((n_agents, T), bool)}
    monkeypatch.setattr(ros_ensemble, "replay_ensemble", fake)
    return calls


def test_cli_one_bag_is_unchanged(monkeypatch, capsys):
    calls = _fake_cli(monkeypatch, [("a.bag", 5)])
    ros_ensemble.main(["a.bag", "--match-threshold", "1,2", "--global-inhibition", "0.1,0.2,0.3"])
    (c,) = calls
    assert isinstance(c["frames"], np.ndarray) and c["recording"] == 0 and c["n_agents"] == 6
    lines = capsys.readouterr().out.splitlines()
    assert len(lines) == 6 and lines[0].startswith("agent 0  match_threshold 1  global_inhibition 0.1  inject_energy none")
    assert not any("bag" in line for line in lines)


def test_cli_cross_product_of_bags_and_settings(monkeypatch, capsys):
    calls = _fake_cli(monkeypatch, [("a.bag", 5), ("bb.bag", 3), ("c.bag", 0)])
    ros_ensemble.main(["a.bag", "bb.bag", "c.bag", "--match-threshold", "1,2", "--inject-energy", "none,0.3"])
    (c,) = calls
    assert [len(f) for f in c["frames"]] == [5, 3, 0] and len(c["odom"]) == 3
    assert c["n_agents"] == 12 and c["recording"] == [0] * 4 + [1] * 4 + [2] * 4
    assert c["match_threshold"] == [1.0, 1.0, 2.0, 2.0] * 3
    assert c["inject_energy"] == [None, 0.3] * 6
    lines = capsys.readouterr().out.splitlines()
    assert len(lines) == 12
    assert lines[0].startswith("bag a.bag  agent 0  match_threshold 1 ")
    assert lines[5].startswith("bag bb.bag  agent 5  match_threshold 1 ") and "inject_energy 0.3" in lines[5]
    assert "created 0/3" in lines[5] and "final arg-max (0, 0, 0)" in lines[5]
    assert lines[11].startswith("bag c.bag  agent 11  match_threshold 2 ") and "final arg-max None" in lines[11]
