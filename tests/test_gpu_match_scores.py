"""Best match scores of every path that makes the create-or-match decision on the device -- the single-agent frame plans
(fused, pipelined, native), ensembles of one and of several recordings, sessions that grow their libraries, and
message-stream replay -- against a view-template-only oracle, at every frame and for every agent.

The decisions alone barely constrain the score: most frames are either near-revisits or new places tens of thousands
away from any threshold, so a sweep that is off by thousands still decides the same way.  The crafted recordings below
put exact, known scores where the sweep can go wrong: exact revisits (0), copies darkened in the compared rows (the
darkening's sum), brighter-by-one pixels (255 each, the uint8 wrap), saturated pixels, row shifts of every offset in
[-8, 8] (7 is inside the search window, 8 is not), all-zero and all-255 frames while libraries end in a partly filled
group of 32 (a slot past the live count must not take part), and ties between groups (the lower index wins).  The
thresholds sit on both sides of those scores, including negative ones: ``min(scores) > threshold`` creates on every
frame then, as the reference does.

A library and its scores depend only on the frames and the threshold, not on the pose cells, so the oracle here replays
the view templates alone: one pass of ``oracle.view_templates.library_scores`` per frame over the recording's earlier
templates, and per threshold only the decisions.  The CPU tests check it against
``oracle.view_templates.ViewTemplates``."""
import functools

import numpy as np
import pytest

ROWS = np.arange(33, 96, 2)      # image rows and columns of the 32x32 template (ros_simulate's mask on 256x256 frames)
WIN = slice(8, 24)               # template rows compared with a stored template at offset 0
S_EDGE = 3000                    # the exact best score of each recording's edge frame (300 pixels darkened by 10)
GIS = (0.05, 0.1, 0.1745, 0.2, 0.25)
# thresholds on both sides of the crafted scores: ties score 255, the edge frame S_EDGE, revisits 0, the largest
# possible score (an all-255 template against an all-zero frame) is 130560
EDGES = (S_EDGE - 1, S_EDGE - 0.5, S_EDGE, S_EDGE + 0.5, 0, -0.5, -1, 2 ** 32 - 1, 2 ** 40, 254.5, 255, -1e9)
NONNEG = (0, 0.5, 254, 255, 255.5, S_EDGE, 1000, 30000, 45000, 58000, 60000, 62000, 65280, 130559, 2 ** 32 - 1, 2 ** 40)


def template(frame):
    return frame[np.ix_(ROWS, ROWS)]


@functools.lru_cache(maxsize=None)
def crafted_recording(seed, T):
    """``(frames uint8 [T,256,256], odom [T,2])`` with the crafted frames at fixed places (T >= 110):

    * 5, 40, 70: S1, S2 = S1 + 1 on a set K of 256 compared pixels, S3 = S2 + 1 on the other 256; 80: S1 + 1 on one
      pixel of K ties S1 and S2 (255 each), 81: S2 + 1 on one pixel outside K ties S2 and S3;
    * 20: the edge frame's source, 82: the source with 300 compared pixels darkened by 10 (best score ``S_EDGE``);
    * 83 and 84: an all-zero and an all-255 frame; 85..101: frame 50 shifted by 2·o image rows, o = -8..8;
    * from 102 on a seeded mix of new places, exact revisits, darker copies, brighter-by-one copies, shifted copies and
      more all-zero / all-255 frames.
    Every other frame is a new place; 4 % of the pixels of a new place are 0 and 4 % are 255."""
    assert T >= 110
    rng = np.random.default_rng(seed)
    frames = np.empty((T, 256, 256), np.uint8)

    def fresh():
        f = rng.integers(0, 256, (256, 256), dtype=np.uint8)
        u = rng.random((256, 256))
        f[u < 0.04] = 0
        f[u > 0.96] = 255
        return f

    def with_template(f, tpl):
        f = f.copy()
        f[np.ix_(ROWS, ROWS)] = tpl
        return f

    win = [(r, c) for r in range(WIN.start, WIN.stop) for c in range(32)]
    perm = rng.permutation(len(win))
    K, K2 = [win[i] for i in perm[:256]], [win[i] for i in perm[256:]]

    def bump(tpl, pixels, d):
        tpl = tpl.astype(np.int16)
        for r, c in pixels:
            tpl[r, c] += d
        assert tpl.min() >= 0 and tpl.max() <= 255
        return tpl.astype(np.uint8)

    for t in range(80):
        frames[t] = fresh()
    s1 = template(frames[5]).copy()
    s1[WIN] = np.minimum(s1[WIN], 253)                       # room for two +1 steps
    frames[5] = with_template(frames[5], s1)
    s2 = bump(s1, K, 1)
    frames[40] = with_template(fresh(), s2)
    frames[70] = with_template(fresh(), bump(s2, K2, 1))
    frames[80] = with_template(fresh(), bump(s1, K[:1], 1))
    frames[81] = with_template(fresh(), bump(s2, K2[:1], 1))
    src = template(frames[20]).copy()
    src[WIN] = np.maximum(src[WIN], 10)
    frames[20] = with_template(frames[20], src)
    frames[82] = with_template(fresh(), bump(src, [win[i] for i in rng.permutation(len(win))[:300]], -10))
    frames[83] = 0
    frames[84] = 255
    for o in range(-8, 9):
        frames[93 + o] = np.roll(frames[50], 2 * o, axis=0)
    for t in range(102, T):
        u = rng.random()
        j = int(rng.integers(0, t))
        if u < 0.3:
            frames[t] = fresh()
        elif u < 0.45:
            frames[t] = frames[j]
        elif u < 0.65:
            dark = rng.integers(0, 4, (256, 256), dtype=np.int16)
            frames[t] = np.clip(frames[j].astype(np.int16) - dark, 0, 255).astype(np.uint8)
        elif u < 0.75:
            tpl = template(frames[j])
            ok = [p for p in win if tpl[p] < 255]
            pick = rng.permutation(len(ok))[:int(rng.choice([1, 2, 3, 5]))]
            frames[t] = with_template(frames[j], bump(tpl, [ok[i] for i in pick], 1))
        elif u < 0.93:
            frames[t] = np.roll(frames[j], 2 * int(rng.integers(-8, 9)), axis=0)
        else:
            frames[t] = 0 if u < 0.965 else 255
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    odom[rng.random(T) < 0.1] = (0.0005, 0.0)               # below the 0.001 gate: no pose-cell update
    frames.setflags(write=False)
    odom.setflags(write=False)
    return frames, odom


@functools.lru_cache(maxsize=None)
def _pair_scores(seed, T):
    """``M[i, j]``: the score of frame j's template against frame i's stored template, i < j (uint64)."""
    from oracle.view_templates import library_scores
    tpl = np.stack([template(f) for f in crafted_recording(seed, T)[0]])
    M = np.zeros((T, T), np.uint64)
    for j in range(1, T):
        M[:j, j] = library_scores(tpl[:j], tpl[j])
    return M


@functools.lru_cache(maxsize=None)
def vt_oracle(seed, T, threshold):
    """``ViewTemplates.match`` (oracle/view_templates.py) over the templates of ``crafted_recording(seed, T)``: per
    frame the best score (-1 for an empty library), the template index and whether it was created; the library's frame
    numbers; and the frames that matched a best score reached by two templates in different groups of 32."""
    M = _pair_scores(seed, T)
    out = {"score": np.full(T, -1, np.int64), "template": np.zeros(T, np.int64), "created": np.zeros(T, np.bool_)}
    lib, ties = [], []
    for j in range(T):
        if lib:
            sc = M[lib, j]
            best = int(sc.min())
            idx = int(np.argmin(sc))
            out["score"][j] = best
        if not lib or best > threshold:
            out["template"][j] = len(lib)
            out["created"][j] = True
            lib.append(j)
        else:
            out["template"][j] = idx
            same = np.nonzero(sc == best)[0]
            if len(same) > 1 and same[-1] // 32 != same[0] // 32:
                ties.append(j)
    out["library"] = np.array(lib, np.int64)
    out["ties"] = ties
    return out


def _library(key, ref):
    frames = crafted_recording(*key)[0]
    return np.stack([template(frames[i]) for i in ref["library"]])


def _check(got, b, key, threshold, what):
    """Agent b of an ensemble replaying ``crafted_recording(*key)``: its score, template and created over the
    recording's frames against the oracle, nothing past them, and its library."""
    ref = vt_oracle(*key, threshold)
    n = key[1]
    for k in ("score", "template", "created"):
        bad = np.nonzero(got[k][b, :n] != ref[k])[0]
        assert len(bad) == 0, (what, b, threshold, k, bad[:5], got[k][b, bad[:5]], ref[k][bad[:5]])
    assert (got["score"][b, n:] == -1).all() and (got["template"][b, n:] == -1).all(), (what, b)
    assert not got["created"][b, n:].any(), (what, b)
    if "agents" in got:
        assert np.array_equal(got["agents"].templates(b), _library(key, ref)), (what, b, threshold)


# ---------------------------------------------------------------------------------------------------- CPU

EDGE_KEY = (11, 120)


def test_oracle_helper_equals_view_templates():
    """The pairwise-score oracle equals oracle.view_templates.ViewTemplates frame by frame, library included."""
    from oracle.view_templates import ViewTemplates
    frames, _ = crafted_recording(*EDGE_KEY)
    for thr in (-1, 0, 255, S_EDGE, 45000, 2 ** 40):
        ref = vt_oracle(*EDGE_KEY, thr)
        vts = ViewTemplates((32, 96), (32, 96), 2, 2, 256, 256, thr)
        for t in range(len(frames)):
            vals = [tm.match(template(frames[t])) for tm in vts.templates]
            n0 = len(vts.templates)
            tm = vts.match(frames[t], 0, 0, 0)
            assert ref["score"][t] == (int(min(vals)) if vals else -1), (thr, t)
            assert ref["template"][t] == tm.get_index() and ref["created"][t] == (len(vts.templates) > n0), (thr, t)
        assert np.array_equal(_library(EDGE_KEY, ref), np.stack([tm.template for tm in vts.templates])), thr


def test_crafted_scores():
    """The crafted frames score what they were made to score, so the thresholds of the GPU tests sit on their edges."""
    frames, _ = crafted_recording(*EDGE_KEY)
    assert (template(frames[83]) == 0).all() and (template(frames[84]) == 255).all()
    assert (template(frames[5]) == 0).any() and (template(frames[5]) == 255).any()
    ref = vt_oracle(*EDGE_KEY, 0)
    assert ref["created"][:80].all()                   # new places: library index = frame number up to 80
    assert ref["score"][80] == ref["score"][81] == 255
    tie = vt_oracle(*EDGE_KEY, 255)                    # the ties match the lower index, across groups of 32
    assert tie["template"][80] == 5 and tie["template"][81] == 40 and {80, 81} <= set(tie["ties"])
    edge = vt_oracle(*EDGE_KEY, S_EDGE)
    assert edge["score"][82] == S_EDGE and not edge["created"][82] and edge["template"][82] == 20
    assert vt_oracle(*EDGE_KEY, S_EDGE - 0.5)["created"][82]
    assert ref["score"][83] > 0 and ref["score"][84] > 0 and ref["created"][:83].sum() % 32 != 0
    for o in range(-8, 9):                             # row offsets 7 are inside the window, 8 are not
        assert (ref["score"][93 + o] == 0) == (abs(o) <= 7), o
    neg = vt_oracle(*EDGE_KEY, -1)
    assert neg["created"].all() and (neg["score"][1:] >= 0).all() and (neg["score"] == 0).any()


def test_thresholds_reach_the_device_unclamped():
    from pyratslam_b200.ros_ensemble import agent_parameters
    _, thr, _, _ = agent_parameters(match_threshold=list(EDGES))
    assert thr.dtype == np.float64 and thr.tolist() == [float(v) for v in EDGES]


# ---------------------------------------------------------------------------------------------------- GPU


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["plain", "fused", "pipelined", "native"])
@pytest.mark.parametrize("threshold", [-1, 255, S_EDGE, 45000])
def test_single_agent_paths(mode, threshold):
    """ros_simulate.replay in every mode: per-frame score, template and created, the library and last_score."""
    from pyratslam_b200 import ros_simulate
    frames, odom = crafted_recording(*EDGE_KEY)
    ref = vt_oracle(*EDGE_KEY, threshold)
    rec = ros_simulate.replay(frames, odom, fused=mode == "fused", pipelined=mode == "pipelined",
                              native=mode == "native", match_threshold=threshold)
    for k in ("score", "template", "created"):
        bad = np.nonzero(rec[k] != ref[k])[0]
        assert len(bad) == 0, (mode, threshold, k, bad[:5], rec[k][bad[:5]], ref[k][bad[:5]])
    vts = rec["node"].vts
    assert vts.last_score == int(ref["score"][-1])
    assert rec["n_templates"] == len(ref["library"])
    got = np.stack([tm.template for tm in vts.templates])
    assert np.array_equal(got, _library(EDGE_KEY, ref)), (mode, threshold)


def _stream(key, seed=4):
    """``crafted_recording(*key)`` as a message stream: one to three twists before each image, none before every fifth
    image, one trailing twist."""
    frames, _ = crafted_recording(*key)
    rng = np.random.default_rng(seed)
    ev, ns = [], 0
    for t in range(len(frames)):
        for _ in range(0 if t % 5 == 2 else int(rng.integers(1, 4))):
            ns += 1000
            ev.append(("odom", (0, ns), (float(rng.uniform(0, 3)), float(rng.uniform(-1, 1)))))
        ns += 1000
        ev.append(("image", (0, ns), frames[t]))
    ev.append(("odom", (0, ns + 1000), (0.77, 0.2)))
    return ev


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["frames", "events"])
def test_threshold_edges(entry):
    """One ensemble, one agent per threshold on either side of the crafted scores: a threshold equal to a best score
    matches, half a unit below it creates, a negative threshold creates on every frame (exact revisits included)."""
    from pyratslam_b200.ros_ensemble import replay_ensemble, replay_ensemble_events
    refs = [vt_oracle(*EDGE_KEY, thr) for thr in EDGES]
    met = {thr for thr, ref in zip(EDGES, refs) if ((ref["score"] == thr) & ~ref["created"]).any()}
    assert {S_EDGE, 255} <= met                        # thresholds equal to a best score
    for thr, ref in zip(EDGES, refs):
        if thr < 0:
            assert ref["created"].all() and (ref["score"] == 0).any()
    kw = dict(match_threshold=list(EDGES), global_inhibition=[GIS[b % 5] for b in range(len(EDGES))])
    if entry == "frames":
        out = replay_ensemble(*crafted_recording(*EDGE_KEY), **kw)
    else:
        out = replay_ensemble_events(_stream(EDGE_KEY), **kw)
    for b, thr in enumerate(EDGES):
        _check(out, b, EDGE_KEY, thr, entry)


GRID_KEYS = ((20, 300), (21, 230), (22, 170))
B_GRID = 96


def _grid_agents():
    """Agent b replays recording b % 3 with threshold NONNEG[(b // 3) % 16]: agents b and b + 48 are replicas of one
    recording and threshold at different device rows, with different global inhibitions."""
    R = len(GRID_KEYS)
    rec = [b % R for b in range(B_GRID)]
    thr = [NONNEG[(b // R) % len(NONNEG)] for b in range(B_GRID)]
    return rec, thr, [GIS[b % 5] for b in range(B_GRID)]


def _check_grid(out, what):
    rec, thr, _ = _grid_agents()
    assert np.array_equal(out["length"], [GRID_KEYS[r][1] for r in rec])
    for b in range(B_GRID):
        _check(out, b, GRID_KEYS[rec[b]], thr[b], what)
    half = B_GRID // 2
    for k in ("score", "template", "created"):          # replicas: identical records
        assert np.array_equal(out[k][:half], out[k][half:]), (what, k)


@functools.lru_cache(maxsize=None)
def _grid_one_call():
    from pyratslam_b200.ros_ensemble import replay_ensemble
    rec, thr, gi = _grid_agents()
    recs = [crafted_recording(*k) for k in GRID_KEYS]
    return replay_ensemble([f for f, _ in recs], [o for _, o in recs], match_threshold=thr, global_inhibition=gi,
                           recording=rec)


@pytest.mark.gpu
def test_grid_stride_and_query_reloads():
    """96 agents of three recordings of different lengths, interleaved: the threshold-0 agents fill 10 groups of 32, so
    the (agent, group) items outnumber the sweep's 592 blocks and one block's items span agents, groups and recordings;
    the shorter recordings end while the others run on."""
    out = _grid_one_call()
    assert B_GRID * ((int(out["n_templates"].max()) + 31) // 32) > 592
    _check_grid(out, "one call")


@pytest.mark.gpu
def test_session_growth():
    """The same agents fed in uneven chunks from 32-template libraries that grow between feeds: the concatenated records
    equal the one-call replay's and the oracle's."""
    from pyratslam_b200.ros_ensemble import EnsembleSession
    rec, thr, gi = _grid_agents()
    recs = [crafted_recording(*k) for k in GRID_KEYS]
    cuts = [(0, 7, 40, 41, 130, 300), (0, 30, 31, 100, 230, 230), (0, 1, 90, 170, 170, 170)]
    s = EnsembleSession(n_recordings=len(GRID_KEYS), recording=rec, match_threshold=thr, global_inhibition=gi,
                        capacity=32)
    keys = ("score", "template", "created")
    got = {"score": np.full((B_GRID, 300), -1, np.int64), "template": np.full((B_GRID, 300), -1, np.int64),
           "created": np.zeros((B_GRID, 300), np.bool_)}
    pos = np.zeros(B_GRID, np.int64)
    caps = []
    try:
        for i in range(len(cuts[0]) - 1):
            o = s.feed([f[c[i]:c[i + 1]] for (f, _), c in zip(recs, cuts)],
                       [od[c[i]:c[i + 1]] for (_, od), c in zip(recs, cuts)])
            caps.append(s.capacity)
            for b in range(B_GRID):
                n = o["length"][b]
                assert (o["score"][b, n:] == -1).all()
                for k in keys:
                    got[k][b, pos[b]:pos[b] + n] = o[k][b, :n]
            pos += o["length"]
            if i == len(cuts[0]) - 2:
                got["agents"] = s.agents
        got["length"] = pos
        assert len(set(caps)) > 2, caps                # the libraries grew from 32, more than once
        one = _grid_one_call()
        for k in keys:
            assert np.array_equal(got[k], one[k]), k
        _check_grid(got, "session")
    finally:
        s.close()


@pytest.mark.gpu
def test_message_streams():
    """replay_ensemble_events on two streams of different lengths with runs of odometry between images and images with
    none before them: the scores per image, for agents of both recordings at every non-negative threshold."""
    from pyratslam_b200.ros_ensemble import replay_ensemble_events
    keys = ((30, 150), (31, 115))
    B = 2 * len(NONNEG)
    rec = [b % 2 for b in range(B)]
    thr = [NONNEG[b // 2] for b in range(B)]
    out = replay_ensemble_events([_stream(k, seed) for seed, k in enumerate(keys)], match_threshold=thr,
                                 global_inhibition=[GIS[b % 5] for b in range(B)], recording=rec)
    for b in range(B):
        _check(out, b, keys[rec[b]], thr[b], "events")
