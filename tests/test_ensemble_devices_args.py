"""Agents split over several devices, without CUDA: the split of shard_agents, the reassign's moves across shards
against a brute-force run of its three steps, and the refusal of bad `devices` arguments before any CUDA call."""
import itertools

import numpy as np
import pytest

from pyratslam_b200 import _native as nat
from pyratslam_b200 import ros_ensemble
from pyratslam_b200.ros_ensemble import (ShardedEnsembleSession, _split, plan_agent_moves, replay_ensemble,
                                         replay_ensemble_events, shard_agents)


@pytest.fixture
def no_cuda(monkeypatch):
    """Fails the test if anything reaches CUDA."""
    def refuse(*a, **k):
        raise AssertionError("reached CUDA")
    monkeypatch.setattr(nat, "require_cuda", refuse)
    monkeypatch.setattr(ros_ensemble.torch.cuda, "device_count", refuse)
    monkeypatch.setattr(ros_ensemble.torch.cuda, "mem_get_info", refuse)


@pytest.fixture
def fake_devices(monkeypatch):
    monkeypatch.setattr(nat, "require_cuda", lambda: None)
    monkeypatch.setattr(ros_ensemble.torch.cuda, "device_count", lambda: 8)


@pytest.mark.parametrize("rec_of, n", [([0] * 7, 3), ([2, 0, 1, 0, 2, 2, 1, 0, 1, 1], 4), ([3, 1, 0, 2], 4),
                                       ([1, 0, 1, 0, 1], 1), (list(np.random.default_rng(0).integers(0, 5, 64)), 8)])
def test_split(rec_of, n, fake_devices):
    rec_of = np.asarray(rec_of)
    B = len(rec_of)
    shards = shard_agents(rec_of, list(range(n)))
    assert len(shards) == n
    agents = np.concatenate([a for a, _ in shards])
    assert sorted(agents.tolist()) == list(range(B))                     # every agent in exactly one shard
    assert np.array_equal(agents, np.argsort(rec_of, kind="stable"))    # contiguous pieces of the recording order
    sizes = [len(a) for a, _ in shards]
    assert max(sizes) - min(sizes) <= 1
    for a, recs in shards:
        assert np.array_equal(recs, np.unique(rec_of[a]))               # its recordings, in global order
        local = np.searchsorted(recs, rec_of[a])
        assert np.array_equal(recs[local], rec_of[a]) and (np.diff(local) >= 0).all()
        assert local[0] == 0


def test_split_repeated_devices(fake_devices):
    shards = shard_agents([0, 1, 1, 2, 2, 2], [0, 0, 0])
    assert [a.tolist() for a, _ in shards] == [[0, 1], [2, 3], [4, 5]]
    assert [r.tolist() for _, r in shards] == [[0, 1], [1, 2], [2]]     # recordings 1 and 2 span two shards


@pytest.mark.parametrize("devices", [[], (), [True], [0, False], [0.0], [1.5], ["0"], "0", 0, None, [-1], [0, 1, 2]])
def test_split_refuses(devices, no_cuda):
    with pytest.raises(ValueError):
        shard_agents([0, 0], devices)


def test_split_checks_the_device_range(monkeypatch):
    monkeypatch.setattr(nat, "require_cuda", lambda: None)
    monkeypatch.setattr(ros_ensemble.torch.cuda, "device_count", lambda: 2)
    assert len(shard_agents([0, 0, 0], [0, 1, 1])) == 3
    with pytest.raises(ValueError, match="cuda:2"):
        shard_agents([0, 0, 0], [0, 2])


def _simulate(parents, shards):
    """The three steps of ShardedEnsembleSession.reassign on labels: every agent's state is its own index."""
    held = [np.array(a) for a, _ in shards]                             # held[s][j]: the state of shard s's agent j
    local, cross = plan_agent_moves(parents, shards)
    stages = [(t, dst, held[s][src].copy()) for s, t, src, dst in cross]        # 1. export before the call
    for s, (dst, src) in enumerate(local):                                       # 2. in-shard copies, all at once
        assert len(set(dst.tolist())) == len(dst) and not (dst == src).any()
        held[s][dst] = held[s][src].copy()
    seen = set()
    for t, dst, rows in stages:                                                  # 3. import
        for j in dst:
            assert (t, int(j)) not in seen                              # each child is written once
            seen.add((t, int(j)))
        held[t][dst] = rows
    out = np.empty(len(parents), np.int64)
    for (a, _), h in zip(shards, held):
        out[a] = h
    return out, local, cross


def _check(parents, shards):
    got, local, cross = _simulate(parents, shards)
    assert np.array_equal(got, np.asarray(parents)), (parents, got)
    n_moves = sum(len(d) for d, _ in local) + sum(len(d) for _, _, _, d in cross)
    assert n_moves == int((np.asarray(parents) != np.arange(len(parents))).sum())
    for s, t, src, dst in cross:
        assert s != t and len(src) == len(dst)
    return cross


def test_moves_swaps_and_cycles_across_shards():
    rec_of = np.zeros(9, np.int64)
    shards = _split(rec_of, 3)                                          # [0 1 2] [3 4 5] [6 7 8]
    cases = {"identity": list(range(9)),
             "swap": [3, 1, 2, 0, 4, 5, 6, 7, 8],                       # 0 <-> 3 across shards 0 and 1
             "cycle": [6, 1, 2, 0, 4, 5, 3, 7, 8],                      # 0 <- 6 <- 3 <- 0 over three shards
             "mixed": [1, 0, 8, 5, 3, 4, 2, 2, 2],                      # in-shard swap, in-shard cycle, cross clones
             "one_remote_parent": [7] * 9}                              # many children of one remote parent
    for name, par in cases.items():
        cross = _check(par, shards)
        if name == "one_remote_parent":
            assert [(s, t, len(src)) for s, t, src, _ in cross] == [(2, 0, 3), (2, 1, 3)]
            assert all((src == 1).all() for _, _, src, _ in cross)     # agent 7 is shard 2's local agent 1


def test_moves_brute_force():
    """Every mapping of 5 agents over 2 and 3 shards, and random ones of larger ensembles with several recordings."""
    for n in (2, 3):
        shards = _split(np.zeros(5, np.int64), n)
        for par in itertools.product(range(5), repeat=5):
            _check(list(par), shards)
    rng = np.random.default_rng(1)
    for _ in range(200):
        B = int(rng.integers(2, 40))
        rec_of = rng.integers(0, 4, B)
        shards = _split(rec_of, int(rng.integers(1, min(B, 6) + 1)))
        par = np.arange(B)
        for r in np.unique(rec_of):                                     # a parent replays its child's recording
            mine = np.nonzero(rec_of == r)[0]
            par[mine] = rng.choice(mine, len(mine))
        _check(par, shards)


def _frames(t):
    return np.zeros((t, 256, 256), np.uint8), np.zeros((t, 2))


@pytest.mark.parametrize("devices", [[], [True], [0, 1.0], "01", [0, 0, 0]])
def test_entry_points_refuse_devices_before_cuda(devices, no_cuda):
    f, o = _frames(4)
    events = [("odom", 0.0, (0.1, 0.0)), ("image", 0.5, f[0])]
    with pytest.raises(ValueError):
        replay_ensemble(f, o, n_agents=2, devices=devices)
    with pytest.raises(ValueError):
        replay_ensemble([f, f[:2]], [o, o[:2]], recording=[0, 1], devices=devices)
    with pytest.raises(ValueError):
        replay_ensemble_events(events, n_agents=2, devices=devices)
    with pytest.raises(ValueError):
        ShardedEnsembleSession(devices, n_agents=2)


def test_sharded_session_refuses_bad_arguments_before_cuda(no_cuda):
    for kw in ({"experience_map": True}, {"n_recordings": 0}, {"capacity": 0},
               {"n_recordings": 2, "recording": [0, 2]}, {"match_threshold": [1, 2], "global_inhibition": [1, 2, 3]}):
        with pytest.raises(ValueError):
            ShardedEnsembleSession([0, 0], n_agents=2, **kw)


def test_cli_passes_devices(monkeypatch, tmp_path):
    seen = {}

    def fake_replay(frames, odom, **kw):
        seen.update(kw)
        B = kw["n_agents"]
        return {"n_templates": np.ones(B, np.int64), "created": np.zeros((B, 1), np.bool_),
                "argmax": np.zeros((B, 1, 3), np.int64)}

    from pyratslam_b200 import rosbag_io
    monkeypatch.setattr(ros_ensemble, "replay_ensemble", fake_replay)
    monkeypatch.setattr(rosbag_io, "read_events", lambda *a, **k: [])
    monkeypatch.setattr(rosbag_io, "events_to_arrays", lambda ev: _frames(1) + (None,))
    ros_ensemble.main(["x.bag", "--match-threshold", "1,2,3", "--devices", "0,1"])
    assert seen["devices"] == [0, 1]
