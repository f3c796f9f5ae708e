"""EnsembleSession.reassign's validation: every refusal happens before the first CUDA call, so it runs without a GPU;
omitted settings are the parents', ``inject_energy=None`` turns injection off."""
import math

import numpy as np
import pytest

from pyratslam_b200 import ros_ensemble
from pyratslam_b200.ros_ensemble import KEEP, EnsembleSession, reassign_parameters

THR = np.array([30000.0, 45000.0, 60000.0, 0.0])
GI = np.array([0.1, 0.2, 0.25, 0.3])
EN = [None, 0.02, 0.3, None]


def test_omitted_settings_are_the_parents():
    par, thr, gi, en = reassign_parameters([1, 1, 3, 2], [0] * 4, THR, GI, EN)
    assert par.tolist() == [1, 1, 3, 2]
    assert thr.tolist() == [45000, 45000, 0, 60000]
    assert gi.tolist() == [0.2, 0.2, 0.3, 0.25]
    assert en == [0.02, 0.02, None, 0.3]
    par, thr, gi, en = reassign_parameters(range(4), [0] * 4, THR, GI, EN, KEEP, KEEP, KEEP)
    assert thr.tolist() == THR.tolist() and gi.tolist() == GI.tolist() and en == EN


def test_given_settings_replace_the_copied_ones():
    _, thr, gi, en = reassign_parameters([0, 0, 0, 0], [0] * 4, THR, GI, EN, new_threshold=[1, 2, 3, 4],
                                         new_inhibition=0.15)
    assert thr.tolist() == [1, 2, 3, 4] and gi.tolist() == [0.15] * 4 and en == [None] * 4
    _, _, _, en = reassign_parameters([1, 1, 2, 2], [0] * 4, THR, GI, EN, new_energy=None)     # None: no injection
    assert en == [None] * 4
    _, _, _, en = reassign_parameters([0, 3, 0, 3], [0] * 4, THR, GI, EN, new_energy=[0.1, None, 0, 0.5])
    assert en == [0.1, None, 0.0, 0.5]


def test_parents_within_each_recording():
    rec = [0, 0, 1, 1]
    assert reassign_parameters([1, 0, 3, 3], rec, THR, GI, EN)[0].tolist() == [1, 0, 3, 3]
    with pytest.raises(ValueError, match="recording"):
        reassign_parameters([2, 1, 2, 3], rec, THR, GI, EN)


class _NoCuda:
    def __getattr__(self, name):
        raise AssertionError("CUDA was touched before the arguments were checked")


def _session(monkeypatch, rec=(0, 0, 0, 0), closed=False):
    """A session's host half with the native layer and torch's CUDA replaced by tripwires."""
    def no_cuda(*a, **k):
        raise AssertionError("CUDA was touched before the arguments were checked")
    monkeypatch.setattr(ros_ensemble.nat, "require_cuda", no_cuda)
    monkeypatch.setattr(ros_ensemble.nat, "lib", no_cuda)
    monkeypatch.setattr(ros_ensemble, "torch", _NoCuda())
    s = EnsembleSession.__new__(EnsembleSession)
    s._plan = None
    s._closed = closed
    s.B = len(rec)
    s._rec_of = np.array(rec, np.int64)
    s._thr, s._gi, s._energies = THR.copy(), GI.copy(), list(EN)
    return s


@pytest.mark.parametrize("parents, kw", [
    ([0, 1, 2], {}),                                       # wrong length
    ([0, 1, 2, 3, 0], {}),
    ([0, 1, 2.0, 3], {}),                                  # not an integer
    ([0, 1, True, 3], {}),
    ([0, 1, "2", 3], {}),
    ("0123", {}),
    (5, {}),
    ([0, 1, 2, 4], {}),                                    # out of range
    ([0, 1, -1, 3], {}),
    ([0, 1, 2, 3], {"match_threshold": [1, 2]}),           # refused by agent_parameters
    ([0, 1, 2, 3], {"match_threshold": math.nan}),
    ([0, 1, 2, 3], {"global_inhibition": [0.1, 0.2, math.inf, 0.1]}),
    ([0, 1, 2, 3], {"inject_energy": -0.5}),
    ([0, 1, 2, 3], {"inject_energy": [0.1, None, math.nan, None]}),
    ([0, 1, 2, 3], {"inject_energy": "0.1"}),
])
def test_reassign_refuses_before_any_cuda_call(parents, kw, monkeypatch):
    s = _session(monkeypatch)
    with pytest.raises(ValueError):
        s.reassign(parents, **kw)
    assert s._thr.tolist() == THR.tolist() and s._energies == EN        # nothing changed


def test_reassign_refuses_a_parent_of_another_recording(monkeypatch):
    s = _session(monkeypatch, rec=(0, 0, 1, 1))
    with pytest.raises(ValueError, match="recording"):
        s.reassign([0, 2, 2, 3])


def test_closed_session_refuses(monkeypatch):
    s = _session(monkeypatch, closed=True)
    with pytest.raises(RuntimeError):
        s.reassign([0, 1, 2, 3])


def test_settings_properties_are_copies(monkeypatch):
    s = _session(monkeypatch)
    thr = s.match_threshold
    thr[0] = -1
    assert s.match_threshold.tolist() == THR.tolist()
    assert s.global_inhibition.tolist() == GI.tolist()
    assert s.inject_energy == EN
    assert repr(KEEP) == "KEEP"
