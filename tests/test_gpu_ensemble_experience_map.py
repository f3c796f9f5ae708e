"""Linked experience maps built on the device (experience_ensemble, csrc/experience_map.cu) against the host class
ExperienceMap(linked=True): crafted records, ensemble replays that close loops, and the single-agent native replay."""
import numpy as np
import pytest

from em_records import assert_same_map, crafted, host_maps, loop_recording

pytestmark = pytest.mark.gpu

SMALL = (6, 5, 7)
ROS = (21, 21, 36)
THRESHOLDS = (0, 30000, 45000, 45000, 60000, 2 ** 32 - 1)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25, 0.3)
MIXED = (None, 0.0, 0.02, 0.3, None, 0.3)


def _check(out, template, argmax, odom, shape, delta_pc=1.0, what=""):
    """out (the device maps) against a host map per agent: structure exact, floats within 1e-9, before and after
    iterate(5)."""
    maps, n_exp, exp_id, em_xy = host_maps(template, argmax, odom, shape, delta_pc)
    assert np.array_equal(out["n_exp"], n_exp), what
    assert np.array_equal(out["exp_id"], exp_id), what
    assert out["em_xy"].shape == em_xy.shape
    if em_xy.size:
        assert np.abs(out["em_xy"] - em_xy).max() <= 1e-9, what
    assert np.array_equal(out["n_loop_closures"], [em.n_loop_closures for em in maps]), what
    dev = out["maps"]
    assert len(dev) == len(maps)
    for b, want in enumerate(maps):
        got = dev.experience_map(b)
        assert_same_map(got, want, what=(what, b))
        assert len(dev.experiences(b)) == len(want.experiences) and len(dev.links(b)) == len(want.links)
        got.iterate(5)
        want.iterate(5)
        assert_same_map(got, want, exact_th=False, what=(what, b, "iterate"))
    return maps


@pytest.mark.parametrize("delta_pc", [0, 1.0, 1.5])
def test_crafted_records(delta_pc):
    from pyratslam_b200.experience_ensemble import ensemble_experience_maps
    tpl, am, odom = crafted(np.random.default_rng(11), 257, 160, SMALL)
    out = ensemble_experience_maps(tpl, am, odom, SMALL, linked=True, delta_pc=delta_pc)
    maps = _check(out, tpl, am, odom, SMALL, delta_pc, delta_pc)
    closures = sum(em.n_loop_closures for em in maps)
    repeated = sum(em.n_loop_closures - (len(em.links) - len(em.experiences) + 1) for em in maps if em.experiences)
    assert closures > 1000 and repeated > 500, (closures, repeated)
    assert all(out["n_exp"][b, -1] <= 2 for b in range(0, 257, 6))       # the packet that never moves


@pytest.mark.parametrize("T", [0, 1, 2, 7])
def test_short_and_still_records(T):
    from pyratslam_b200.experience_ensemble import ensemble_experience_maps
    tpl, am, odom = crafted(np.random.default_rng(T), 9, T, SMALL)
    _check(ensemble_experience_maps(tpl, am, odom, SMALL, linked=True), tpl, am, odom, SMALL, what=T)
    out = ensemble_experience_maps(tpl, am, np.zeros((T, 2)), SMALL, linked=True)     # nobody moves
    assert not out["n_exp"].any() and (out["exp_id"] == -1).all() and not out["em_xy"].any()
    assert out["em_xy"].shape == (9, T, 2) and not out["n_loop_closures"].any()


def test_sparse_template_ids():
    """Template ids far beyond the frame count (records from another source) give the same maps, reported with the
    caller's ids, and a workspace that does not grow with the ids."""
    from pyratslam_b200.experience_ensemble import ensemble_experience_maps
    tpl, am, odom = crafted(np.random.default_rng(21), 40, 120, SMALL)
    sparse = np.where(tpl >= 0, tpl * 7919 + 2 ** 40, tpl)
    out = ensemble_experience_maps(sparse, am, odom, SMALL, linked=True)
    _check(out, sparse, am, odom, SMALL, what="sparse")
    assert out["maps"]._v["vt_head"].shape[0] <= 120


def test_ensemble_replay_against_the_host_maps():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 240
    frames, odom = loop_recording(np.random.default_rng(3), T)
    kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED))
    dev = replay_ensemble(frames, odom, experience_map="device", experience_links=True, **kw)
    host = replay_ensemble(frames, odom, experience_map=True, experience_links=True, **kw)
    for k in ("template", "created", "argmax", "n_exp"):
        assert np.array_equal(dev[k], host[k]), k
    assert np.abs(dev["em_xy"] - host["em_xy"]).max() <= 1e-9
    _check(dev, dev["template"], dev["argmax"], odom, ROS, what="replay")
    assert (dev["n_loop_closures"] > 0).sum() >= 4, dev["n_loop_closures"]
    dev = replay_ensemble(frames, odom, experience_map="device", **kw)
    host = replay_ensemble(frames, odom, experience_map=True, **kw)
    for k in ("n_exp", "em_xy"):
        assert np.array_equal(dev[k], host[k]), k
    assert dev["maps"] is None and not dev["n_loop_closures"].any()


def test_single_agent_equals_native_replay():
    from pyratslam_b200 import ros_simulate
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 240
    frames, odom = loop_recording(np.random.default_rng(4), T)
    want = ros_simulate.replay(frames, odom, native=True, experience_links=True)
    out = replay_ensemble(frames, odom, experience_map="device", experience_links=True)
    assert np.array_equal(out["n_exp"][0], want["n_exp"])
    assert np.abs(out["em_xy"][0] - want["em_xy"]).max() <= 1e-9
    em = want["node"].em
    assert em.n_loop_closures > 0 and out["n_loop_closures"][0] == em.n_loop_closures
    got = out["maps"].experience_map(0)
    assert_same_map(got, em)
    got.iterate(5)
    em.iterate(5)
    assert_same_map(got, em, exact_th=False)
