"""EnsembleSession.reassign: after the call agent b is agent parents[b] as it was before it, with the parent's or the
given settings.  A child fed on equals its parent in a twin session that made no call -- records, libraries, locations,
pose cells and linked maps -- through appends and library growth, for the identity, clones, swaps, cycles, one parent
for all and a child that held more templates than its parent; with new settings each child equals the oracle's loop
run with its parent's settings up to the call and its own after it."""
import functools
import math

import numpy as np
import pytest

from em_records import assert_same_map, loop_recording

pytestmark = pytest.mark.gpu

SHAPE = (21, 21, 36)
THRESHOLDS = (0, 30000, 45000, 45000, 60000, 2 ** 32 - 1)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25, 0.3)          # 0.3: the network dies
MIXED = (None, 0.0, 0.02, 0.3, None, 0.3)
RECORD_KEYS = ("template", "created", "score", "argmax", "n_exp", "exp_id", "em_xy")
CONFIGS = [(6, np.float32, "cluster"), (6, np.float64, None), (60, np.float32, "pair"), (300, np.float32, "resident")]


def _settings(B):
    return dict(match_threshold=[THRESHOLDS[b % 6] for b in range(B)], global_inhibition=[GIS[b % 6] for b in range(B)],
                inject_energy=[MIXED[b % 6] for b in range(B)])


def _mapping(name, B):
    par = list(range(B))
    head = {"identity": par[:6], "clones": [0, 0, 2, 2, 4, 1], "swaps": [1, 0, 3, 2, 5, 4], "cycle": [1, 2, 0, 3, 4, 5],
            "more_templates": [5, 1, 2, 3, 4, 5]}      # agent 0 (threshold 0) holds ~40 templates, agent 5 one
    if name == "one_parent":
        return [3] * B
    par[:6] = head[name]
    if B > 6 and name != "identity":
        par[B - 1] = 0                                 # a move far from the others: another recording slice of rows
    return par


def _check_children(got, s, want, t, par, agents, what, maps=True):
    """Agent b of session s (fed `got`) equals agent par[b] of the twin t (fed `want`)."""
    for b in agents:
        p = par[b]
        for k in RECORD_KEYS:
            if k in got:
                assert np.array_equal(got[k][b], want[k][p], equal_nan=True), (what, b, k)
        assert s.n_templates[b] == t.n_templates[p], (what, b)
        assert np.array_equal(s.agents.templates(b), t.agents.templates(p)), (what, b)
        assert np.array_equal(s.agents.locations(b), t.agents.locations(p)), (what, b)
        assert np.array_equal(s.agents.posecells(b), t.agents.posecells(p)), (what, b)
        assert s.match_threshold[b] == t.match_threshold[p] and s.global_inhibition[b] == t.global_inhibition[p]
        assert s.inject_energy[b] == t.inject_energy[p]
        if maps:
            assert s.n_loop_closures[b] == t.n_loop_closures[p], (what, b)
            gm, wm = s.maps.experience_map(b), t.maps.experience_map(p)
            assert_same_map(gm, wm, what=(what, b))
            gm.iterate(5)
            wm.iterate(5)
            assert_same_map(gm, wm, exact_th=False, what=(what, b, "iterate"))


def _checked_agents(par, B):
    moved = [b for b in range(B) if par[b] != b]
    return sorted(set(range(6)) | set(moved[:4]) | set(moved[-2:]))


@pytest.mark.parametrize("B, dtype, path", CONFIGS)
@pytest.mark.parametrize("name", ["identity", "clones", "swaps", "cycle", "one_parent", "more_templates"])
def test_children_continue_as_their_parents(B, dtype, path, name):
    from pyratslam_b200.ros_ensemble import EnsembleSession
    frames, odom = loop_recording(np.random.default_rng(3), 150)
    kw = dict(_settings(B), dtype=dtype, active_set=2, experience_map="device", experience_links=True)
    s, t = EnsembleSession(**kw), EnsembleSession(**kw)
    assert path is None or s.agents.path == path
    for x in (s, t):
        x.feed(frames[:40], odom[:40])
    assert s.capacity == 64 and s.n_templates[0] > 32 and s.n_templates[5] == 1    # a partly filled second group
    par = _mapping(name, B)
    s.reassign(par)
    agents = _checked_agents(par, B)
    # appends, then a feed that grows the libraries (threshold 0 creates on most frames) and the map workspace
    for lo, hi in ((40, 50), (50, 150)):
        got, want = s.feed(frames[lo:hi], odom[lo:hi]), t.feed(frames[lo:hi], odom[lo:hi])
        _check_children(got, s, want, t, par, agents, (name, B, lo))
    assert s.capacity > 64
    assert (t.n_loop_closures > 0).any()
    s.close()
    t.close()
    with pytest.raises(RuntimeError):
        s.reassign(range(B))


@functools.lru_cache(maxsize=None)
def _oracle_cached(seed, T, cut, before, after):
    frames, odom = loop_recording(np.random.default_rng(seed), T)
    return _oracle(frames, odom, cut, before, after)


def _oracle(frames, odom, cut, before, after):
    """oracle/drivers.py's loop with the agent's (threshold, inhibition, energy) `before` for frames [0, cut) and
    `after` from then on, plus its library."""
    from oracle import drivers as odrv
    from oracle.posecells import PoseCellNetwork
    from oracle.view_templates import ViewTemplates
    T = len(frames)
    thr, gi, energy = before
    pcn = PoseCellNetwork(SHAPE, global_inhibition=gi)
    pcn.inject(1, tuple(math.floor(s / 2) for s in SHAPE))
    vts = ViewTemplates(odrv.X_RANGE, odrv.Y_RANGE, odrv.X_STEP, odrv.Y_STEP, 256, 256, thr)
    rec = {"template": np.zeros(T, np.int64), "created": np.zeros(T, np.bool_), "argmax": np.zeros((T, 3), np.int64)}
    for t in range(T):
        if t == cut:
            vts.match_threshold, pcn.global_inhibition, energy = after
        lin, ang = float(odom[t, 0]), float(odom[t, 1])
        if abs(lin) > 0.001 or abs(ang) > 0.001:
            pcn.update((lin / odrv.ODOM_FREQ, ang / odrv.ODOM_FREQ))
        pc_max = pcn.get_pc_max()
        n0 = len(vts.templates)
        tm = vts.match(frames[t], pc_max[0], pc_max[1], pc_max[2])
        if energy is not None:
            pcn.inject(energy, tm.location())
        rec["template"][t], rec["created"][t], rec["argmax"][t] = tm.get_index(), len(vts.templates) > n0, pc_max
    rec["n_templates"] = len(vts.templates)
    rec["final_state"] = pcn.posecells
    rec["templates"] = np.stack([t.template for t in vts.templates])
    rec["locations"] = np.array([t.location() for t in vts.templates], dtype=np.int64)
    return rec


# (initial energies, parents, new thresholds, new inhibitions, new energies): thresholds up and down, inhibitions
# changed (into the dying 0.3 too), energies None -> value and value -> None, a session without injection that gains it
# and one whose injection ends
CASES = {
    "mixed": (list(MIXED), [1, 0, 2, 2, 5, 3], [45000, 0, 60000, 30000, 45000, 30000], [0.1, 0.3, 0.2, 0.1745, 0.25, 0.05],
              [0.02, None, None, 0.3, 0.02, None]),
    "gains": ([None] * 6, [0, 0, 2, 3, 3, 5], "keep", "keep", [0.3, None, 0.02, 0.0, 0.3, 0.02]),
    "loses": (list(MIXED), [3, 1, 2, 3, 3, 5], [30000] * 6, "keep", None),
}


@pytest.mark.parametrize("dtype, tol", [(np.float32, 1e-5), (np.float64, 1e-12)])
@pytest.mark.parametrize("case", sorted(CASES))
def test_new_settings_against_the_oracle(dtype, tol, case):
    from pyratslam_b200.ros_ensemble import KEEP, EnsembleSession
    energies, par, thr1, gi1, en1 = CASES[case]
    frames, odom = loop_recording(np.random.default_rng(5), 60)
    cut = 30
    s = EnsembleSession(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=energies,
                        dtype=dtype, active_set=2)
    first = s.feed(frames[:cut], odom[:cut])
    keep = lambda v: KEEP if isinstance(v, str) else v                    # noqa: E731
    s.reassign(par, match_threshold=keep(thr1), global_inhibition=keep(gi1), inject_energy=keep(en1))
    thr_now = [THRESHOLDS[p] for p in par] if isinstance(thr1, str) else thr1
    gi_now = [GIS[p] for p in par] if isinstance(gi1, str) else gi1
    en_now = [None] * 6 if en1 is None else en1
    assert s.match_threshold.tolist() == thr_now and s.global_inhibition.tolist() == gi_now
    assert s.inject_energy == en_now
    second = s.feed(frames[cut:], odom[cut:])
    for b in range(6):
        p = par[b]
        ref = _oracle_cached(5, 60, cut, (THRESHOLDS[p], GIS[p], energies[p]), (thr_now[b], gi_now[b], en_now[b]))
        for k in ("template", "created", "argmax"):
            assert np.array_equal(first[k][p], ref[k][:cut]), (case, b, k)
            assert np.array_equal(second[k][b], ref[k][cut:]), (case, b, k)
        assert s.n_templates[b] == ref["n_templates"], (case, b)
        assert np.array_equal(s.agents.templates(b), ref["templates"]), (case, b)
        assert np.array_equal(s.agents.locations(b), ref["locations"]), (case, b)
        fs, want = s.agents.posecells(b), ref["final_state"]
        scale = want.max() if want.max() > 0 else 1.0
        assert np.abs(fs - want).max() <= tol * scale, (case, b, np.abs(fs - want).max() / scale)
    s.close()


def test_several_recordings():
    from pyratslam_b200.ros_ensemble import EnsembleSession
    recs = [loop_recording(np.random.default_rng(r), 90) for r in (7, 8)]
    rec = [0, 1, 0, 1, 0, 1, 1, 0]
    kw = dict(_settings(8), recording=rec, n_recordings=2, dtype=np.float32, active_set=2, experience_map="device",
              experience_links=True)
    s, t = EnsembleSession(**kw), EnsembleSession(**kw)
    for x in (s, t):
        x.feed([recs[0][0][:30], recs[1][0][:20]], [recs[0][1][:30], recs[1][1][:20]])
    with pytest.raises(ValueError, match="recording"):
        s.reassign([1, 1, 2, 3, 4, 5, 6, 7])
    par = [4, 5, 0, 1, 0, 3, 6, 2]                     # within each recording: a swap, a clone, a cycle
    s.reassign(par)
    got = s.feed([recs[0][0][30:], recs[1][0][20:]], [recs[0][1][30:], recs[1][1][20:]])
    want = t.feed([recs[0][0][30:], recs[1][0][20:]], [recs[0][1][30:], recs[1][1][20:]])
    _check_children(got, s, want, t, par, range(8), "R = 2")


def test_message_streams_continue_the_parents_tag():
    """feed_events after a reassign: a child's next experience is tagged with its parent's last template (the
    forward-filled tag), not its own, so its map continues as the parent's in the twin session."""
    from pyratslam_b200.ros_ensemble import EnsembleSession
    frames, odom = loop_recording(np.random.default_rng(9), 120)
    events = []
    for i in range(len(frames)):
        events.append(("odom", 2.0 * i, (float(odom[i, 0]), float(odom[i, 1]))))
        if i % 3 != 2:                                # runs of odometry without an image
            events.append(("image", 2.0 * i + 1, frames[i]))
    cut = next(i for i, ev in enumerate(events) if ev[1] >= 100.0 and ev[0] == "odom" and events[i - 1][0] == "odom")
    B = 6
    kw = dict(_settings(B), dtype=np.float32, active_set=2, experience_map="device", experience_links=True)
    s, t = EnsembleSession(**kw), EnsembleSession(**kw)
    for x in (s, t):
        x.feed_events(events[:cut])                   # the piece ends on odometry after its last image
    par = [2, 0, 2, 5, 1, 3]
    last = s._prev_tpl[s._rows]
    assert any(last[b] != last[par[b]] for b in range(B))
    s.reassign(par)
    got, want = s.feed_events(events[cut:]), t.feed_events(events[cut:])
    _check_children(got, s, want, t, par, range(B), "events")


def test_maps_continue_the_parents_host_map():
    """Each child's linked map equals its parent's host ExperienceMap taken before the call, continued on the host over
    the child's later records, before and after relaxation."""
    from pyratslam_b200.experience_ensemble import gate
    from pyratslam_b200.ros_ensemble import EnsembleSession
    frames, odom = loop_recording(np.random.default_rng(11), 200)
    B, cut = 6, 80
    s = EnsembleSession(**_settings(B), dtype=np.float64, active_set=2, experience_map="device", experience_links=True)
    first = s.feed(frames[:cut], odom[:cut])
    par = [3, 3, 0, 1, 4, 2]
    host = [s.maps.experience_map(p) for p in par]
    last = [int(first["template"][p, -1]) for p in par]
    s.reassign(par, match_threshold=[45000, 30000, 60000, 0, 45000, 30000])
    got = s.feed(frames[cut:], odom[cut:])
    moved, tw = gate(odom[cut:])
    for b in range(B):
        em, tpl = host[b], np.concatenate([[last[b]], got["template"][b]])
        for t in range(len(moved)):
            if moved[t]:
                em.update(float(tw[t, 0]), float(tw[t, 1]), tuple(int(c) for c in got["argmax"][b, t]),
                          None if tpl[t] < 0 else int(tpl[t]))
        gm = s.maps.experience_map(b)
        assert_same_map(gm, em, what=b)
        assert gm.n_loop_closures == s.n_loop_closures[b]
        gm.iterate(5)
        em.iterate(5)
        assert_same_map(gm, em, exact_th=False, what=(b, "iterate"))
    assert (s.n_loop_closures > 0).any()
