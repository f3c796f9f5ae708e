"""The host side of the ensemble experience maps: the shared dead reckoning of unlinked maps, ExperienceMap.from_arrays
and the validation of replay_ensemble's experience_map argument (no GPU needed)."""
import numpy as np
import pytest

from em_records import arrays, assert_same_map, crafted, host_maps

from pyratslam_b200.experience_ensemble import ensemble_experience_maps, gate
from pyratslam_b200.experience_map import ExperienceMap
from pyratslam_b200.ros_ensemble import _experience_maps

SHAPE = (6, 5, 7)


@pytest.mark.parametrize("T", [0, 1, 2, 97])
def test_unlinked_maps_equal_the_host_replay(T):
    tpl, am, odom = crafted(np.random.default_rng(T), 13, T, SHAPE)
    got = ensemble_experience_maps(tpl, am, odom, SHAPE, linked=False)
    moved, tw = gate(odom)
    n_exp, em_xy = _experience_maps({"template": tpl, "argmax": am}, moved, tw, SHAPE, False)
    assert np.array_equal(got["n_exp"], n_exp) and np.array_equal(got["em_xy"], em_xy)
    assert np.array_equal(got["exp_id"], n_exp - 1)
    assert np.array_equal(got["n_loop_closures"], np.zeros(13)) and got["maps"] is None


@pytest.mark.parametrize("delta_pc", [0, 1.0, 1.5])
def test_from_arrays_rebuilds_the_map(delta_pc):
    rng = np.random.default_rng(7)
    tpl, am, odom = crafted(rng, 12, 150, SHAPE)
    maps = host_maps(tpl, am, odom, SHAPE, delta_pc)[0]
    more_tpl, more_am, more_odom = crafted(rng, 12, 50, SHAPE)
    moved, tw = gate(more_odom)
    closures = 0
    for b, em in enumerate(maps):
        ex, li = arrays(em)
        got = ExperienceMap.from_arrays(ex, li, em.current_exp.index if em.current_exp else -1,
                                        rel=(em.rel_x, em.rel_y, em.rel_th),
                                        accum=(em.accum_delta_x, em.accum_delta_y, em.accum_delta_th),
                                        n_loop_closures=em.n_loop_closures, pc_dims=SHAPE, delta_pc=delta_pc)
        assert_same_map(got, em, tol=0, what=b)
        for m in (got, em):
            m.iterate(5)
        assert got.get_poses() == em.get_poses() and got.links == em.links
        for t in range(50):
            if moved[t]:
                vt = int(more_tpl[b, t])
                args = (float(tw[t, 0]), float(tw[t, 1]), tuple(int(c) for c in more_am[b, t]), vt if vt >= 0 else None)
                em.update(*args)
                got.update(*args)
        assert_same_map(got, em, tol=0, what=b)
        assert got.get_poses() == em.get_poses() and got.links == em.links
        assert (got.rel_x, got.rel_y, got.rel_th) == (em.rel_x, em.rel_y, em.rel_th)
        assert (got.accum_delta_x, got.accum_delta_y, got.accum_delta_th) == \
            (em.accum_delta_x, em.accum_delta_y, em.accum_delta_th)
        closures += em.n_loop_closures
    assert closures > 0


@pytest.mark.parametrize("value", ["host", "Device", None, 2, "True", 0, 1, 1.0])
def test_bad_experience_map_values_raise_before_cuda(value):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    frames = np.zeros((4, 256, 256), np.uint8)
    with pytest.raises(ValueError, match="experience_map"):
        replay_ensemble(frames, np.zeros((4, 2)), experience_map=value)


def test_bad_records_raise():
    tpl, am, odom = crafted(np.random.default_rng(1), 3, 10, SHAPE)
    bad_cell = am.copy()
    bad_cell[1, 4, 2] = SHAPE[2]
    for args in ((tpl[:, :5], am, odom), (tpl, am[:, :, :2], odom), (tpl, am, odom[:4]), (tpl, bad_cell, odom),
                 (tpl.astype(float), am, odom)):
        with pytest.raises(ValueError):
            ensemble_experience_maps(*args, SHAPE, linked=True)
