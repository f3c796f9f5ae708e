"""The ensemble's pose-cell activity capture: per image, every agent's cells above the threshold in the state its match
was made with, against the oracle's ``nonzero(pc > 0.002)`` right after the update and before the injection; its exact
invariants; off against on; truncation; the pose-cell kernel families; and sessions fed in pieces."""
import functools
import math

import numpy as np
import pytest

from synth import synth_frames

pytestmark = pytest.mark.gpu

SHAPE = (21, 21, 36)
N = 21 * 21 * 36
THR = 0.002
THRESHOLDS = (0, 30000, 45000, 45000, 60000, 2 ** 32 - 1)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25, 0.3)          # 0.3: the network dies
MIXED = (None, 0.0, 0.02, 0.3, None, 0.3)
SETS = [(45000, 0.2, None), (0, 0.1, 0.02), (30000, 0.1745, 0.3), (60000, 0.25, 0.0), (2 ** 32 - 1, 0.05, 0.3)]


def _inputs(T, seed=5):
    """Frames with revisits (every third frame), odometry with frames below the 0.001 gate."""
    frames = synth_frames(np.random.default_rng(seed), T)
    for t in range(4, T, 3):
        frames[t] = frames[t - 1]
    rng = np.random.default_rng(seed + 1)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    for t in (9, 10, 30):
        if t < T:
            odom[t] = (0.0, 0.0)
    return frames, odom


@functools.lru_cache(maxsize=None)
def _oracle(T, threshold, gi, energy, shape=SHAPE):
    """The oracle's replay loop; per frame the state the match was made with (after the update, before the
    injection) and the arg-max."""
    from oracle import drivers as odrv
    from oracle.posecells import PoseCellNetwork
    from oracle.view_templates import ViewTemplates
    frames, odom = _inputs(T)
    pcn = PoseCellNetwork(shape, global_inhibition=gi)
    pcn.inject(1, tuple(math.floor(s / 2) for s in shape))
    vts = ViewTemplates(odrv.X_RANGE, odrv.Y_RANGE, odrv.X_STEP, odrv.Y_STEP, 256, 256, threshold)
    states, amax = [], []
    for t in range(T):
        lin, ang = float(odom[t, 0]), float(odom[t, 1])
        if abs(lin) > 0.001 or abs(ang) > 0.001:
            pcn.update((lin / odrv.ODOM_FREQ, ang / odrv.ODOM_FREQ))
        states.append(pcn.posecells.copy())
        pc_max = pcn.get_pc_max()
        amax.append(pc_max)
        tm = vts.match(frames[t], pc_max[0], pc_max[1], pc_max[2])
        if energy is not None:
            pcn.inject(energy, tm.location())
    return np.stack(states), np.array(amax)


def _entry(out, b, i):
    from pyratslam_b200.ros_ensemble import activity_entry
    return activity_entry(out, b, i)


def _check_oracle(out, b, states, tol, what):
    """Every frame of agent b against the oracle's states: the same cells except within tol*max of the threshold,
    values within tol*max, and the count is the number of cells."""
    for t, pc in enumerate(states):
        idx, val = _entry(out, b, t)
        scale = max(pc.max(), 1e-300)
        assert out["activity_count"][b, t] == len(idx), (what, b, t)
        want = np.argwhere(pc > THR)
        got = {tuple(c) for c in idx}
        ref = {tuple(c) for c in want}
        for c in got ^ ref:
            assert abs(pc[c] - THR) <= tol * scale, (what, b, t, c, pc[c])
        for c, v in zip(idx, val):
            assert abs(v - pc[tuple(c)]) <= tol * scale, (what, b, t, tuple(c))
        assert [tuple(c) for c in idx] == sorted(got), (what, b, t)          # C order


def _check_invariants(out, b, what):
    """Exact: where the entry holds every cell above the threshold, the arg-max record is the first maximum of them."""
    K = out.get("_k", N)
    for t in range(out["activity_count"].shape[1]):
        c = out["activity_count"][b, t]
        if 0 < c <= K:
            idx, val = _entry(out, b, t)
            assert tuple(idx[int(np.argmax(val))]) == tuple(out["argmax"][b, t]), (what, b, t)


def _same_entries(a, b_out, rows_a, rows_b, what):
    for ra, rb in zip(rows_a, rows_b):
        n = a["activity_count"].shape[1]
        assert np.array_equal(a["activity_count"][ra], b_out["activity_count"][rb][:n]), (what, ra, rb)
        for i in range(n):
            ia, va = _entry(a, ra, i)
            ib, vb = _entry(b_out, rb, i)
            assert np.array_equal(ia, ib) and np.array_equal(va, vb), (what, ra, rb, i)


@pytest.mark.parametrize("dtype, tol", [(np.float32, 1e-5), (np.float64, 1e-12)])
def test_six_agents_against_the_oracle(dtype, tol):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 60
    frames, odom = _inputs(T)
    for energies in ((None,) * 6, MIXED):
        kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(energies),
                  dtype=dtype)
        off = replay_ensemble(frames, odom, **kw)
        out = replay_ensemble(frames, odom, activity_threshold=THR, max_active_cells=N, **kw)
        assert "activity_count" not in off
        # off against on: the capture only reads
        for k in ("template", "created", "score", "argmax", "n_templates"):
            assert np.array_equal(out[k], off[k]), (k, energies)
        assert np.array_equal(out["agents"].state.cpu().numpy(), off["agents"].state.cpu().numpy())
        assert out["activity_count"].shape == (6, T) and out["activity_ptr"].shape == (6 * T + 1,)
        assert out["activity_cell"].dtype == np.int64 and out["activity_value"].dtype == np.float64
        for b in range(6):
            states, amax = _oracle(T, THRESHOLDS[b], GIS[b], energies[b])
            _check_oracle(out, b, states, tol, (dtype, energies))
            _check_invariants(out, b, (dtype, energies))
            if energies[b] is None:      # nothing changes the state after the last match
                fs = out["agents"].posecells(b)
                idx, val = _entry(out, b, T - 1)
                assert np.array_equal(idx, np.argwhere(fs > THR)) and np.array_equal(val, fs[fs > THR])
        assert out["activity_count"][5, -1] == 0                             # gi = 0.3: the network died
        assert (out["activity_count"] > 0).sum() > T


def test_truncation_and_counts_only():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 40
    frames, odom = _inputs(T)
    kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED),
              activity_threshold=THR)
    full = replay_ensemble(frames, odom, max_active_cells=N, **kw)
    four = replay_ensemble(frames, odom, max_active_cells=4, **kw)
    zero = replay_ensemble(frames, odom, max_active_cells=0, **kw)
    assert np.array_equal(four["activity_count"], full["activity_count"])
    assert np.array_equal(zero["activity_count"], full["activity_count"])
    assert (full["activity_count"] > 4).any()
    assert zero["activity_cell"].shape == (0, 3) and zero["activity_value"].shape == (0,)
    assert not zero["activity_ptr"].any()
    for b in range(6):
        for t in range(T):
            i4, v4 = _entry(four, b, t)
            i_, v_ = _entry(full, b, t)
            assert np.array_equal(i4, i_[:4]) and np.array_equal(v4, v_[:4]), (b, t)
        four["_k"] = 4
        _check_invariants(four, b, "K=4")


@pytest.mark.parametrize("B, path", [(8, "cluster"), (60, "pair"), (300, "resident")])
def test_pose_cell_paths(B, path):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 48
    frames, odom = _inputs(T)
    sets = [SETS[b % len(SETS)] for b in range(B)]
    out = replay_ensemble(frames, odom, match_threshold=[s[0] for s in sets], global_inhibition=[s[1] for s in sets],
                          inject_energy=[s[2] for s in sets], activity_threshold=THR, max_active_cells=N)
    assert out["agents"].path == path
    for b in range(len(SETS)):
        _check_oracle(out, b, _oracle(T, *SETS[b])[0], 1e-5, path)
        _check_invariants(out, b, path)
    first = [b % len(SETS) for b in range(B)]
    _same_entries(out, out, first, range(B), path)


def test_active_set_gives_the_dense_cells():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    T = 60
    frames, odom = _inputs(T)
    kw = dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED),
              activity_threshold=THR, max_active_cells=N)
    act = replay_ensemble(frames, odom, active_set=2, **kw)
    for b in range(6):
        _check_oracle(act, b, _oracle(T, THRESHOLDS[b], GIS[b], MIXED[b])[0], 1e-5, "active_set=2")
        _check_invariants(act, b, "active_set=2")


def test_large_grid():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    shape = (50, 50, 10)
    T = 16
    frames, odom = _inputs(T)
    out = replay_ensemble(frames, odom, match_threshold=[45000, 0], global_inhibition=[0.2, 0.1],
                          inject_energy=[None, 0.02], pose_size=shape, activity_threshold=THR,
                          max_active_cells=50 * 50 * 10)
    for b, (thr, gi, e) in enumerate(((45000, 0.2, None), (0, 0.1, 0.02))):
        _check_oracle(out, b, _oracle(T, thr, gi, e, shape)[0], 1e-5, ("50x50x10", out["agents"].path))
        _check_invariants(out, b, "50x50x10")


def _session_kw():
    return dict(match_threshold=list(THRESHOLDS), global_inhibition=list(GIS), inject_energy=list(MIXED),
                activity_threshold=THR, max_active_cells=64)


def _concat(outs, B):
    """The activity of several feeds per agent: per image (count, cells, values)."""
    rows = [[] for _ in range(B)]
    for out in outs:
        for b in range(B):
            for i in range(int(out["length"][b])):
                idx, val = _entry(out, b, i)
                rows[b].append((int(out["activity_count"][b, i]), idx, val))
            assert (out["activity_count"][b, int(out["length"][b]):] == -1).all()
    return rows


def _one_call(out, B):
    return [[(int(out["activity_count"][b, i]),) + tuple(_entry(out, b, i))
             for i in range(out["activity_count"].shape[1] if "length" not in out else int(out["length"][b]))]
            for b in range(B)]


def _equal_rows(got, want, what):
    assert len(got) == len(want), what
    for b, (g, w) in enumerate(zip(got, want)):
        assert len(g) == len(w), (what, b)
        for i, (x, y) in enumerate(zip(g, w)):
            assert x[0] == y[0] and np.array_equal(x[1], y[1]) and np.array_equal(x[2], y[2]), (what, b, i)


def test_session_feeds_concatenate_and_grow():
    from pyratslam_b200.ros_ensemble import EnsembleSession, replay_ensemble
    T = 150
    frames, odom = _inputs(T)
    want = replay_ensemble(frames, odom, **_session_kw())
    s = EnsembleSession(**_session_kw())
    outs, t0 = [], 0
    for n in (1, 7, 64, 0, T - 72):
        outs.append(s.feed(frames[t0:t0 + n], odom[t0:t0 + n]))
        t0 += n
    assert s.capacity > 32                        # the threshold-0 agent outgrew the first libraries
    s.close()
    _equal_rows(_concat(outs, 6), _one_call(want, 6), "feeds")


def test_four_recordings_fed_unevenly():
    from pyratslam_b200.ros_ensemble import EnsembleSession, replay_ensemble
    lens = (30, 12, 4, 25)
    recs = [_inputs(n, seed=11 + 2 * r) for r, n in enumerate(lens)]
    recording = [0, 1, 2, 3, 0, 1, 3, 3]
    kw = dict(match_threshold=[0, 45000, 30000, 60000, 45000, 0, 45000, 0], global_inhibition=0.2,
              inject_energy=[None, 0.02, None, 0.3, 0.02, None, None, 0.3], activity_threshold=THR, max_active_cells=64)
    want = replay_ensemble([f for f, _ in recs], [o for _, o in recs], recording=recording, **kw)
    for b, r in enumerate(recording):
        assert (want["activity_count"][b, lens[r]:] == -1).all() and (want["activity_count"][b, :lens[r]] >= 0).all()
    s = EnsembleSession(n_recordings=4, recording=recording, **kw)
    outs, at = [], [0] * 4
    for piece in ((5, 12, 0, 1), (20, 0, 0, 3), (5, 0, 4, 21)):
        outs.append(s.feed([recs[r][0][at[r]:at[r] + n] for r, n in enumerate(piece)],
                           [recs[r][1][at[r]:at[r] + n] for r, n in enumerate(piece)]))
        at = [a + n for a, n in zip(at, piece)]
    s.close()
    _equal_rows(_concat(outs, 8), _one_call(want, 8), "uneven")


def test_feed_events_equals_feed():
    from pyratslam_b200.ros_ensemble import EnsembleSession
    T = 40
    frames, odom = _inputs(T)
    events = []
    for t in range(T):
        events.append(("odom", 0.1 * t, (float(odom[t, 0]), float(odom[t, 1]))))
        events.append(("image", 0.1 * t + 0.05, frames[t]))
    a = EnsembleSession(**_session_kw())
    b = EnsembleSession(**_session_kw())
    got = [a.feed_events(events[:30]), a.feed_events(events[30:])]
    want = [b.feed(frames[:15], odom[:15]), b.feed(frames[15:], odom[15:])]
    a.close()
    b.close()
    _equal_rows(_concat(got, 6), _concat(want, 6), "events")


def test_reassign_keeps_the_capture():
    from pyratslam_b200.ros_ensemble import EnsembleSession
    T = 50
    frames, odom = _inputs(T)
    s = EnsembleSession(**_session_kw())
    s.feed(frames[:20], odom[:20])
    parents = [0, 0, 2, 2, 4, 4]
    s.reassign(parents)
    out = s.feed(frames[20:], odom[20:])
    _same_entries(out, out, parents, range(6), "reassign")
    s.reassign(parents, inject_energy=None)           # an injection change makes the plan again; it still captures
    out = s.feed(frames[20:30], odom[20:30])
    assert out["activity_count"].shape == (6, 10) and (out["activity_count"] >= 0).all()
    s.close()
