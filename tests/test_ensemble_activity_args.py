"""The pose-cell activity capture without CUDA: its settings are validated before any CUDA call, ``activity_entry`` reads
one entry of a result, and the CLI's --activity-threshold asks for counts only and prints them."""
import math

import numpy as np
import pytest

from pyratslam_b200 import ros_ensemble
from pyratslam_b200.ros_ensemble import activity_entry, activity_parameters


def test_settings_accepted():
    assert activity_parameters() == (None, 128)
    assert activity_parameters(0.002, 0) == (0.002, 0)
    assert activity_parameters(np.float32(0.5), np.int64(7)) == (0.5, 7)
    assert activity_parameters(-1, 21 * 21 * 36) == (-1.0, 21 * 21 * 36)
    assert activity_parameters(0.002, 500, pose_size=(50, 50, 10)) == (0.002, 500)
    assert activity_parameters(None, 128)[0] is None


BAD = [
    {"activity_threshold": math.nan},
    {"activity_threshold": math.inf},
    {"activity_threshold": -math.inf},
    {"activity_threshold": True},
    {"activity_threshold": np.bool_(False)},
    {"activity_threshold": "0.002"},
    {"activity_threshold": [0.002]},
    {"activity_threshold": 0.002, "max_active_cells": -1},
    {"activity_threshold": 0.002, "max_active_cells": 21 * 21 * 36 + 1},
    {"activity_threshold": 0.002, "max_active_cells": 4.0},
    {"activity_threshold": 0.002, "max_active_cells": True},
    {"activity_threshold": 0.002, "max_active_cells": None},
    {"max_active_cells": "8"},
]


@pytest.mark.parametrize("kw", BAD)
def test_settings_refused(kw):
    with pytest.raises(ValueError):
        activity_parameters(**kw)


def _no_cuda(monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("CUDA was touched before the arguments were checked")
    monkeypatch.setattr(ros_ensemble.nat, "require_cuda", no_cuda)
    monkeypatch.setattr(ros_ensemble.nat, "lib", no_cuda)


@pytest.mark.parametrize("kw", BAD)
def test_replays_and_sessions_refuse_before_any_cuda_call(kw, monkeypatch):
    _no_cuda(monkeypatch)
    frames, odom = np.zeros((4, 256, 256), np.uint8), np.zeros((4, 2))
    with pytest.raises(ValueError):
        ros_ensemble.replay_ensemble(frames, odom, **kw)
    with pytest.raises(ValueError):
        ros_ensemble.replay_ensemble_events([("odom", 0.0, (1.0, 0.0)), ("image", 0.1, frames[0])], **kw)
    with pytest.raises(ValueError):
        ros_ensemble.EnsembleSession(n_agents=2, **kw)


def test_bound_follows_the_grid(monkeypatch):
    _no_cuda(monkeypatch)
    with pytest.raises(ValueError):
        ros_ensemble.EnsembleSession(pose_size=(10, 10, 4), activity_threshold=0.0, max_active_cells=401)
    assert activity_parameters(0.0, 400, pose_size=(10, 10, 4)) == (0.0, 400)


def test_activity_entry():
    # two agents, three images: agent 0 has 2, 0 and 1 kept cells, agent 1 one image and then nothing
    out = {"activity_count": np.array([[2, 0, 5], [1, -1, -1]]),
           "activity_ptr": np.array([0, 2, 2, 3, 4, 4, 4]),
           "activity_cell": np.array([[1, 2, 3], [1, 2, 4], [0, 0, 1], [5, 5, 5]]),
           "activity_value": np.array([0.1, 0.2, 0.3, 0.4])}
    idx, val = activity_entry(out, 0, 0)
    assert idx.tolist() == [[1, 2, 3], [1, 2, 4]] and val.tolist() == [0.1, 0.2]
    idx, val = activity_entry(out, 0, 1)
    assert idx.shape == (0, 3) and val.shape == (0,)
    idx, val = activity_entry(out, 1, 0)
    assert idx.tolist() == [[5, 5, 5]] and val.tolist() == [0.4]
    assert activity_entry(out, 1, 2)[0].shape == (0, 3)
    for b, i in ((2, 0), (0, 3), (-1, 0)):
        with pytest.raises(IndexError):
            activity_entry(out, b, i)


def test_cli_activity_threshold(monkeypatch, capsys):
    seen = []

    def fake(bags, chunk, image_topic, odom_topic, recording, acc=None, **kw):
        seen.append((kw.get("activity_threshold"), kw.get("max_active_cells"), acc is not None))
        B = kw["n_agents"]
        ros_ensemble._activity_stats({"activity_count": np.array([[3, 5, -1], [0, 0, 0]][:B])}, acc)
        ros_ensemble._activity_stats({"activity_count": np.array([[4], [2]][:B])}, acc)
        return np.arange(B), np.zeros(B, np.int64), np.array([4] * len(bags)), [(1, 2, 3)] * B, None
    monkeypatch.setattr(ros_ensemble, "_replay_chunked", fake)
    ros_ensemble.main(["a.bag", "--chunk", "3", "--match-threshold", "1,2", "--activity-threshold", "0.002"])
    assert seen == [(0.002, 0, True)]
    lines = capsys.readouterr().out.splitlines()
    assert lines[0].endswith("active cells mean 4.0 max 5")
    assert lines[1].endswith("active cells mean 0.5 max 2")
    ros_ensemble.main(["a.bag", "--chunk", "3"])
    assert seen[1] == (None, None, False) and "active cells" not in capsys.readouterr().out
