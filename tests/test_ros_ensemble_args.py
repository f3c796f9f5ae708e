"""replay_ensemble's per-agent argument broadcasting and validation: all of it happens before the first CUDA call, so it
runs without a GPU."""
import math

import numpy as np
import pytest

from pyratslam_b200 import ros_ensemble


def test_broadcasting_keeps_thresholds():
    B, thr, gi, en = ros_ensemble.agent_parameters()
    assert B == 1 and thr.tolist() == [45000] and gi.tolist() == [0.2] and en == [None]
    B, thr, gi, en = ros_ensemble.agent_parameters(n_agents=3, match_threshold=30000.7, inject_energy=0.3)
    assert B == 3 and thr.tolist() == [30000.7] * 3 and gi.tolist() == [0.2] * 3 and en == [0.3] * 3
    B, thr, gi, en = ros_ensemble.agent_parameters(match_threshold=[0, -5, 2.0 ** 40, 45000, -0.5, np.int64(7)],
                                                   global_inhibition=np.linspace(0.05, 0.25, 6),
                                                   inject_energy=[None, 0, 0.02, np.float32(0.5), None, None])
    assert B == 6
    # the caller's numbers, unclamped: a negative threshold creates on every frame, as ViewTemplates.match does
    assert thr.dtype == np.float64 and thr.tolist() == [0, -5, 2.0 ** 40, 45000, -0.5, 7]
    assert np.array_equal(gi, np.linspace(0.05, 0.25, 6))
    assert en == [None, 0.0, 0.02, 0.5, None, None]
    assert ros_ensemble.agent_parameters(n_agents=2, global_inhibition=(0.1, 0.3))[0] == 2


def test_capacity():
    assert ros_ensemble.capacity_for(0) == 32
    assert ros_ensemble.capacity_for(31) == 32
    assert ros_ensemble.capacity_for(32) == 64
    assert ros_ensemble.capacity_for(2000) == 2016


@pytest.mark.parametrize("kw", [
    {"match_threshold": [1, 2], "global_inhibition": [0.1, 0.2, 0.3]},       # lengths disagree
    {"n_agents": 3, "inject_energy": [None, 0.1]},                            # n_agents disagrees
    {"n_agents": 0},
    {"match_threshold": []},
    {"inject_energy": -0.01},
    {"inject_energy": [0.1, math.inf]},
    {"inject_energy": [0.1, math.nan]},
    {"inject_energy": "0.1"},
    {"match_threshold": math.nan},
    {"match_threshold": [0, -math.inf]},
    {"match_threshold": [0, math.inf]},
    {"global_inhibition": [0.1, math.inf]},
    {"global_inhibition": True},
])
def test_invalid_parameters(kw):
    with pytest.raises(ValueError):
        ros_ensemble.agent_parameters(**kw)


def _frames(T):
    return np.zeros((T, 256, 256), np.uint8), np.zeros((T, 2))


@pytest.mark.parametrize("args, kw", [
    (_frames(4), {"inject_energy": [0.1, -1.0]}),
    (_frames(4), {"mode": "circular"}),
    ((np.zeros((4, 128, 128), np.uint8), np.zeros((4, 2))), {}),
    ((np.zeros((4, 256, 256), np.float32), np.zeros((4, 2))), {}),
    ((np.zeros((4, 256, 256), np.uint8), np.zeros((3, 2))), {}),
    ((np.zeros((4, 256, 256), np.uint8), np.zeros((4, 3))), {}),
    ((np.broadcast_to(np.zeros((1, 256, 256), np.uint8), (1 << 16, 256, 256)), np.zeros((1 << 16, 2))), {}),  # too long
])
def test_replay_refuses_before_any_cuda_call(args, kw, monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("CUDA was touched before the arguments were checked")
    monkeypatch.setattr(ros_ensemble.nat, "require_cuda", no_cuda)
    monkeypatch.setattr(ros_ensemble.nat, "lib", no_cuda)
    with pytest.raises(ValueError):
        ros_ensemble.replay_ensemble(*args, **kw)
