"""Host side of the in-frame injection: template location -> C-order flat pose cell, with the rules of
PoseCellEnsemble.inject (int() truncation, numpy negative indices, -1 where inject raises IndexError).  No GPU."""
import numpy as np

from pyratslam_b200.view_templates import flat_cell_index

SHAPE = (21, 21, 36)


def _flat(x, y, th):
    return x * 21 * 36 + y * 36 + th


def test_integer_locations_are_c_order_flat_indices():
    loc = [(0, 0, 0), (10, 10, 18), (20, 20, 35), (3, 4, 5)]
    assert flat_cell_index(loc, SHAPE).tolist() == [_flat(*c) for c in loc]
    assert flat_cell_index(np.zeros((0, 3)), SHAPE).tolist() == []


def test_truncation_toward_zero():
    got = flat_cell_index([(2.9, 3.5, 35.99), (-0.5, 0.7, -0.99), (20.999, 0.0, 1.2)], SHAPE)
    assert got.tolist() == [_flat(2, 3, 35), _flat(0, 0, 0), _flat(20, 0, 1)]


def test_negative_indices_wrap_like_numpy():
    got = flat_cell_index([(-1, -21, -36), (-1.5, 2, -0.2), (-21, -1, 0)], SHAPE)
    assert got.tolist() == [_flat(20, 0, 0), _flat(20, 2, 0), _flat(0, 20, 0)]


def test_out_of_bounds_and_non_finite_are_invalid():
    bad = [(21, 0, 0), (0, 21, 0), (0, 0, 36), (-22, 0, 0), (0, -22.5, 0), (0, 0, -37), (np.nan, 0, 0),
           (0, np.inf, 0), (1e300, 0, 0)]
    assert flat_cell_index(bad, SHAPE).tolist() == [-1] * len(bad)
    # one bad coordinate invalidates only its own row
    assert flat_cell_index([(1, 2, 3), (1, 2, 36), (1, 2, 35)], SHAPE).tolist() == [_flat(1, 2, 3), -1, _flat(1, 2, 35)]


def test_matches_the_inject_rule_cell_by_cell():
    """Every location the host inject accepts maps to the cell it writes; every other one to -1."""
    rng = np.random.default_rng(3)
    loc = rng.uniform(-40, 60, (2000, 3))
    got = flat_cell_index(loc, SHAPE)
    for (x, y, th), g in zip(loc, got):
        c = [int(v) for v in (x, y, th)]
        c = [v + n if -n <= v < 0 else v for v, n in zip(c, SHAPE)]
        ok = all(0 <= v < n for v, n in zip(c, SHAPE))
        assert g == (np.ravel_multi_index(c, SHAPE) if ok else -1)
