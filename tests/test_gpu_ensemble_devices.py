"""Agents split over several devices (ShardedEnsembleSession, replay_ensemble(devices=...)): every result key and every
`agents` and `maps` accessor equals one device's, with the same pose-cell family forced on both sides (shard sizes
may select another), through uneven multi-recording feeds, message streams, injection on and off, linked maps, the
activity capture, library growth in one shard and reassigns across shards; without forcing, sampled agents equal the
native replay.  Two or three shards on one device run everywhere; [0, 1] and all devices need two GPUs."""
import contextlib

import numpy as np
import pytest
import torch

from em_records import loop_recording

pytestmark = pytest.mark.gpu

_N = torch.cuda.device_count() if torch.cuda.is_available() else 0
_MULTI = pytest.mark.skipif(_N < 2, reason="needs two GPUs, %d visible" % _N)
DEVICES = [pytest.param([0, 0], id="0,0"), pytest.param([0, 0, 0], id="0,0,0"),
           pytest.param([0, 1], id="0,1", marks=_MULTI), pytest.param(list(range(max(_N, 2))), id="all", marks=_MULTI)]
THRESHOLDS = (45000, 30000, 60000, 45000, 0, 30000)
GIS = (0.2, 0.1, 0.25, 0.1745, 0.1, 0.2)
MIXED = (None, 0.3, 0.02, None, 0.3, 0.0)


@contextlib.contextmanager
def forced(path="generic"):
    """Both sides' pose-cell networks on one kernel family (bench_tools/multi_recording_replay.py's pattern)."""
    from pyratslam_b200 import ros_ensemble
    orig = ros_ensemble.PoseCellEnsemble

    class Forced(orig):
        def __init__(self, *a, **k):
            super().__init__(*a, **k)
            self.force_path(path)

    ros_ensemble.PoseCellEnsemble = Forced
    try:
        yield
    finally:
        ros_ensemble.PoseCellEnsemble = orig


def _settings(B, energies=MIXED):
    return dict(match_threshold=[THRESHOLDS[b % 6] for b in range(B)], global_inhibition=[GIS[b % 6] for b in range(B)],
                inject_energy=[energies[b % 6] for b in range(B)])


def _same_result(got, want, what):
    assert set(got) == set(want), (what, sorted(set(got) ^ set(want)))
    for k, v in want.items():
        if k in ("agents", "maps"):
            continue
        assert got[k].dtype == v.dtype and got[k].shape == v.shape, (what, k, got[k].shape, v.shape)
        assert np.array_equal(got[k], v, equal_nan=v.dtype.kind == "f"), (what, k)


def _same_agents(s, t, B, what):
    """Sessions (or results) s and t hold the same agents: libraries, locations, pose cells and linked maps."""
    ga, wa = s["agents"] if isinstance(s, dict) else s.agents, t["agents"] if isinstance(t, dict) else t.agents
    assert len(ga) == len(wa) == B and np.array_equal(ga.n_templates, wa.n_templates), what
    for b in range(B):
        assert np.array_equal(ga.templates(b), wa.templates(b)), (what, b)
        assert np.array_equal(ga.locations(b), wa.locations(b)), (what, b)
        assert np.array_equal(ga.posecells(b), wa.posecells(b)), (what, b)
    gm, wm = s["maps"] if isinstance(s, dict) else s.maps, t["maps"] if isinstance(t, dict) else t.maps
    assert (gm is None) == (wm is None), what
    if gm is None:
        return
    assert len(gm) == len(wm) == B
    for k in ("n_experiences", "n_links", "current", "n_loop_closures"):
        assert np.array_equal(getattr(gm, k), getattr(wm, k)), (what, k)
    for b in range(B):
        assert gm.experiences(b).tobytes() == wm.experiences(b).tobytes(), (what, b)
        assert gm.links(b).tobytes() == wm.links(b).tobytes(), (what, b)
        assert gm.experience_map(b).n_loop_closures == wm.experience_map(b).n_loop_closures


@pytest.mark.parametrize("devices", DEVICES)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("energies", [MIXED, (None,) * 6], ids=["inject", "no_inject"])
def test_one_recording(devices, dtype, energies):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames, odom = loop_recording(np.random.default_rng(3), 140)
    B = 7
    kw = dict(_settings(B, energies), dtype=dtype, experience_map="device", experience_links=True,
              activity_threshold=0.002, max_active_cells=24)
    with forced():
        one = replay_ensemble(frames, odom, **kw)
        got = replay_ensemble(frames, odom, devices=devices, **kw)
    _same_result(got, one, "one recording")
    _same_agents(got, one, B, "one recording")
    assert (one["n_loop_closures"] > 0).any() and (one["activity_count"] > 0).any()
    assert got["agents"].path == ["generic"] * len(devices)
    if len(devices) > 1:
        with pytest.raises(RuntimeError, match="posecells"):
            got["agents"].state


def _pieces(recs, cuts):
    """Feeds of four recordings: piece i of recording r is frames [cuts[r][i], cuts[r][i + 1])."""
    out = []
    for i in range(len(cuts[0]) - 1):
        out.append(([recs[r][0][cuts[r][i]:cuts[r][i + 1]] for r in range(4)],
                    [recs[r][1][cuts[r][i]:cuts[r][i + 1]] for r in range(4)]))
    return out


@pytest.mark.parametrize("devices", DEVICES)
def test_four_recordings_fed_unevenly(devices):
    """Pieces of different lengths, empty ones among them; recording 3's agents create on every frame (threshold 0),
    the others only on their first, so only the last shard's libraries grow past the initial 32."""
    from pyratslam_b200.ros_ensemble import EnsembleSession, ShardedEnsembleSession
    recs = [loop_recording(np.random.default_rng(s), T) for s, T in ((4, 90), (5, 60), (6, 75), (7, 110))]
    rec = [3, 0, 1, 2, 3, 0, 1, 2, 3, 1, 0]
    B = len(rec)
    thr = [0 if r == 3 else 2 ** 32 - 1 for r in rec]
    kw = dict(match_threshold=thr, global_inhibition=[GIS[b % 6] for b in range(B)],
              inject_energy=[MIXED[b % 6] for b in range(B)], n_recordings=4, recording=rec, dtype=np.float32,
              experience_map="device", experience_links=True, activity_threshold=0.002, max_active_cells=16)
    cuts = [[0, 30, 30, 55, 80, 90], [0, 0, 25, 40, 60, 60], [0, 20, 41, 60, 75, 75], [0, 20, 50, 70, 90, 110]]
    with forced():
        s, t = ShardedEnsembleSession(devices, **kw), EnsembleSession(**kw)
        for i, (fr, od) in enumerate(_pieces(recs, cuts)):
            _same_result(s.feed(fr, od), t.feed(fr, od), ("piece", i))
    assert np.array_equal(s.frames_fed, t.frames_fed)
    for k in ("n_templates", "n_experiences", "n_loop_closures", "match_threshold", "global_inhibition"):
        assert np.array_equal(getattr(s, k), getattr(t, k)), k
    assert s.inject_energy == t.inject_energy and (s.B, s.R, s.pose_size) == (t.B, t.R, t.pose_size)
    caps = [sh.capacity for sh in s._shards]
    assert caps[-1] > 32 and caps[:-1] == [32] * (len(caps) - 1), caps
    _same_agents(s, t, B, "pieces")
    s.close()
    t.close()
    with pytest.raises(RuntimeError):
        s.feed(*_pieces(recs, cuts)[0])


def _events(frames, odom):
    ev = []
    for i in range(len(frames)):
        ev.append(("odom", 2.0 * i, (float(odom[i, 0]), float(odom[i, 1]))))
        if i % 3 != 2:                                 # runs of odometry without an image
            ev.append(("image", 2.0 * i + 1, frames[i]))
    return ev


@pytest.mark.parametrize("devices", DEVICES)
def test_feed_events(devices):
    from pyratslam_b200.ros_ensemble import EnsembleSession, ShardedEnsembleSession, replay_ensemble_events
    streams = [_events(*loop_recording(np.random.default_rng(s), T)) for s, T in ((8, 100), (9, 70))]
    rec = [1, 0, 1, 0, 0, 1]
    kw = dict(_settings(6), n_recordings=2, recording=rec, experience_map="device", experience_links=True,
              activity_threshold=0.002, max_active_cells=8)
    with forced():
        s, t = ShardedEnsembleSession(devices, **kw), EnsembleSession(**kw)
        for lo, hi in ((0, 50), (50, 51), (51, None)):
            ev = [st[lo:hi] for st in streams]
            _same_result(s.feed_events(ev), t.feed_events(ev), ("events", lo))
        _same_agents(s, t, 6, "events")
        del kw["n_recordings"]
        got = replay_ensemble_events(streams, devices=devices, **kw)
        want = replay_ensemble_events(streams, **kw)
    _same_result(got, want, "replay_ensemble_events")
    _same_agents(got, want, 6, "replay_ensemble_events")


@pytest.mark.parametrize("devices", DEVICES)
def test_reassign_across_shards(devices):
    """Parents on other shards -- swaps and cycles between shards, one remote parent of several children, a child whose
    shard must grow to take its parent's library and map -- injection switched on in a shard that had none, then two
    feeds: everything equals one device given the same reassign."""
    from pyratslam_b200.ros_ensemble import EnsembleSession, ShardedEnsembleSession
    frames, odom = loop_recording(np.random.default_rng(10), 200)
    B = 9
    # agents 0-4 never create after their first frame and inject nothing, so the first shard's libraries stay at 32
    # templates while agents 6-8 create on every frame
    M = 2 ** 32 - 1
    kw = dict(match_threshold=[M, M, M, M, M, 30000, 0, 0, 0],
              global_inhibition=[0.2, 0.1, 0.25, 0.1745, 0.2, 0.1, 0.2, 0.1, 0.2],
              inject_energy=[None, None, None, None, None, 0.3, 0.3, None, 0.02], dtype=np.float32,
              experience_map="device", experience_links=True)
    par = [7, 5, 0, 4, 3, 1, 2, 6, 6]   # 0 <- 7 (a larger library), 1 <- 5 <- 1 swap, cycle 3 -> 4 -> 3, 6 <- 2 <- 0
    with forced():
        s, t = ShardedEnsembleSession(devices, **kw), EnsembleSession(**kw)
        for lo in range(0, 70, 10):
            for x in (s, t):
                x.feed(frames[lo:lo + 10], odom[lo:lo + 10])
        assert t.n_templates[7] > 32 >= s._shards[0].capacity
        new_energy = [0.3, 0.02, None, None, 0.3, 0.02, None, 0.3, 0.3]
        for x in (s, t):
            x.reassign(par, inject_energy=new_energy)
        for k in ("n_templates", "n_experiences", "n_loop_closures", "match_threshold", "global_inhibition"):
            assert np.array_equal(getattr(s, k), getattr(t, k)), k
        assert s.inject_energy == t.inject_energy == new_energy
        assert s._shards[0].capacity > 32
        _same_agents(s, t, B, "after reassign")
        for lo, hi in ((70, 90), (90, 200)):
            _same_result(s.feed(frames[lo:hi], odom[lo:hi]), t.feed(frames[lo:hi], odom[lo:hi]), ("after", lo))
        _same_agents(s, t, B, "fed after reassign")
        with pytest.raises(ValueError):
            s.reassign([1] * B, match_threshold=float("nan"))
        s.reassign(list(range(B)))
    s.close()
    with pytest.raises(RuntimeError):
        s.reassign(list(range(B)))


@pytest.mark.parametrize("devices", DEVICES)
def test_agents_equal_the_native_replay(devices):
    from pyratslam_b200 import ros_simulate
    from pyratslam_b200.ros_ensemble import replay_ensemble
    recs = [loop_recording(np.random.default_rng(s), T) for s, T in ((11, 60), (12, 45))]
    rec = [1, 0, 0, 1, 1, 0, 1, 0]
    B = len(rec)
    st = _settings(B)
    del st["global_inhibition"]                       # replay() runs the default inhibition
    out = replay_ensemble([f for f, _ in recs], [o for _, o in recs], recording=rec, devices=devices, **st)
    for b in (0, 1, B // 2, B - 1):
        f, o = recs[rec[b]]
        want = ros_simulate.replay(f, o, native=True, match_threshold=st["match_threshold"][b],
                                   inject_energy=st["inject_energy"][b])
        for k in ("template", "created", "argmax"):
            assert np.array_equal(out[k][b, :len(f)], want[k]), (b, k)
        assert out["n_templates"][b] == want["n_templates"]
        fs = want["node"].pcn.posecells
        assert np.abs(out["agents"].posecells(b) - fs).max() <= 1e-6 * fs.max(), b


@pytest.mark.parametrize("devices", DEVICES)
def test_lut_hole_closes_every_shard(devices):
    from pyratslam_b200.ros_ensemble import EnsembleSession, ShardedEnsembleSession
    recs = [loop_recording(np.random.default_rng(s), 50) for s in (13, 14)]
    bad = recs[1][1].copy()
    bad[20] = (1.0, 0.0)             # vtrans = 0.1 after the /10 scaling: the reference's LUT hole
    kw = dict(_settings(6), n_recordings=2, recording=[0, 1, 0, 1, 0, 0])
    fr, od = [recs[0][0], recs[1][0]], [recs[0][1], bad]
    with pytest.raises(KeyError) as one:
        EnsembleSession(**kw).feed(fr, od)
    s = ShardedEnsembleSession(devices, **kw)
    with pytest.raises(KeyError) as got:
        s.feed(fr, od)
    assert got.value.args == one.value.args == ((5, 5),)
    assert all(sh._closed for sh in s._shards)
    with pytest.raises(RuntimeError):
        s.feed(fr, od)


def test_device_range():
    from pyratslam_b200.ros_ensemble import ShardedEnsembleSession, replay_ensemble, shard_agents
    n = torch.cuda.device_count()
    with pytest.raises(ValueError, match="cuda:%d" % n):
        shard_agents([0, 0], [0, n])
    with pytest.raises(ValueError, match="cuda:%d" % n):
        ShardedEnsembleSession([n], n_agents=2)
    frames, odom = loop_recording(np.random.default_rng(1), 4)
    with pytest.raises(ValueError, match="cuda:%d" % n):
        replay_ensemble(frames, odom, n_agents=2, devices=[0, n])


def test_one_shard_is_one_device():
    """devices=[0]: the wrapper alone, agents in another order than their recordings'; `state` in the caller's order."""
    from pyratslam_b200.ros_ensemble import replay_ensemble
    recs = [loop_recording(np.random.default_rng(s), 40) for s in (15, 16)]
    kw = dict(_settings(5), recording=[1, 0, 1, 0, 0])
    args = ([f for f, _ in recs], [o for _, o in recs])
    got, want = replay_ensemble(*args, devices=[0], **kw), replay_ensemble(*args, **kw)
    _same_result(got, want, "one shard")
    assert torch.equal(got["agents"].state, want["agents"].state)
