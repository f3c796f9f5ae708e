"""Ensemble sessions: what feeding the agents in chunks costs against one replay_ensemble call, what it saves in device
memory, and a recording beyond the one-shot limit of 65535 frames.

Prints one JSON line with the GPU's name and power limit read in the same run:

* (a) chunk cost: agent-frames/s (B x frames / wall clock, setup included, median of --repeats) of one replay_ensemble
  call and of EnsembleSession fed 256, 1024 and 4096 frames at a time (starting at 32 templates, so the libraries grow
  during the feeds), alternated in one run, for one 1000-frame recording x 1024 settings and for 16 recordings x 16
  settings.  Whether every agent's records (template, created, arg-max) are identical between the one call and the
  256-frame feeds, with the resident pose-cell kernel forced on both sides.
* (b) memory: torch.cuda.max_memory_allocated of the one call and of a session fed 256 frames at a time, B = 1024,
  T = 10000 frames that revisit 200 places, so that the agents hold far fewer templates than frames.
* (c) one 100000-frame recording x 256 settings, generated and fed 4096 frames at a time (300 places, revisited).

    python bench_tools/ensemble_session.py [--repeats 3] > profiles/r6_ensemble_session.txt
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, os.path.join(ROOT, "bench_tools"))

from inject_replay import gpu_info  # noqa: E402
from multi_recording_replay import forced_path  # noqa: E402

ENERGY = 0.02
CHUNKS = (256, 1024, 4096)


def settings(S):
    thr = np.linspace(30000, 60000, 64)
    gi = np.linspace(0.05, 0.25, max(S // 64, 1))
    grid = [(t, g) for g in gi for t in thr][:S] if S >= 64 else [(t, g) for t, g in zip(np.linspace(30000, 60000, S),
                                                                                         np.linspace(0.05, 0.25, S))]
    return [t for t, _ in grid], [g for _, g in grid]


def odometry(rng, T):
    return np.stack([rng.uniform(0.1, 3, T), rng.uniform(-1, 1, T)], axis=1)


def recordings(R, T):
    from synth import synth_frames
    frames, odom = [], []
    for r in range(R):
        rng = np.random.default_rng(200 + r)
        frames.append(synth_frames(rng, T))
        odom.append(odometry(rng, T))
    return frames, odom


def one_call(frames, odom, S):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    thr, gi = settings(S)
    if len(frames) == 1:
        return replay_ensemble(frames[0], odom[0], match_threshold=thr, global_inhibition=gi, inject_energy=ENERGY)
    R = len(frames)
    return replay_ensemble(frames, odom, recording=np.repeat(np.arange(R), S), match_threshold=np.tile(thr, R),
                           global_inhibition=np.tile(gi, R), inject_energy=ENERGY)


def session(frames, odom, S, chunk):
    """A session fed ``chunk`` frames of every recording at a time; the records concatenated over the feeds."""
    from pyratslam_b200.ros_ensemble import EnsembleSession
    thr, gi = settings(S)
    R = len(frames)
    s = EnsembleSession(match_threshold=np.tile(thr, R), global_inhibition=np.tile(gi, R), inject_energy=ENERGY,
                        n_recordings=R, recording=np.repeat(np.arange(R), S))
    T = max(len(f) for f in frames)
    outs = []
    for t in range(0, T, chunk):
        if R == 1:
            outs.append(s.feed(frames[0][t:t + chunk], odom[0][t:t + chunk]))
        else:
            outs.append(s.feed([f[t:t + chunk] for f in frames], [o[t:t + chunk] for o in odom]))
    s.close()
    out = {k: np.concatenate([o[k] for o in outs], axis=1) for k in ("template", "created", "argmax")}
    out["capacity"] = s.capacity
    return out


def timed(fn, *args):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn(*args)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


def differing_agents(a, b):
    return [int(i) for i in np.nonzero([not all(np.array_equal(a[k][i], b[k][i]) for k in ("template", "created",
                                                                                          "argmax"))
                                        for i in range(len(a["template"]))])[0]]


def chunk_cost(frames, odom, S, repeats):
    B, T = len(frames) * S, max(len(f) for f in frames)
    walls = {"one_call": []}
    walls.update({"session_%d" % c: [] for c in CHUNKS})
    for _ in range(repeats):                 # alternated: one call, then each chunk size
        walls["one_call"].append(timed(one_call, frames, odom, S)[0])
        for c in CHUNKS:
            walls["session_%d" % c].append(timed(session, frames, odom, S, c)[0])
    res = {"agents": B, "frames": T}
    for k, w in walls.items():
        res[k + "_agent_frames_per_s"] = B * T / float(np.median(w))
        res[k + "_s"] = sorted(w)
    for c in CHUNKS:
        res["session_%d_over_one_call" % c] = res["session_%d_agent_frames_per_s" % c] / res["one_call_agent_frames_per_s"]
        # per-feed overhead: the extra wall clock over the one call, per feed
        feeds = -(-T // c)
        res["session_%d_extra_ms_per_feed" % c] = ((float(np.median(walls["session_%d" % c]))
                                                    - float(np.median(walls["one_call"]))) / feeds * 1e3)
    with forced_path("resident"):
        one = one_call(frames, odom, S)
        ses = session(frames, odom, S, CHUNKS[0])
    bad = differing_agents(one, ses)
    res["records_identical_resident_forced"] = not bad
    res["differing_agents_resident_forced"] = bad[:8]
    return res


def memory(repeats):
    import torch
    from synth import synth_frames
    B, T, K = 1024, 10000, 200
    rng = np.random.default_rng(7)
    base = synth_frames(rng, K)
    frames = base[np.arange(T) % K]
    odom = odometry(rng, T)
    res = {"agents": B, "frames": T, "places": K}
    for name, fn in (("one_call", lambda: one_call([frames], [odom], B)),
                     ("session_256", lambda: session([frames], [odom], B, 256))):
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base_bytes = torch.cuda.memory_allocated()
        wall, out = timed(fn)
        res[name + "_max_memory_allocated_bytes"] = torch.cuda.max_memory_allocated() - base_bytes
        res[name + "_s"] = wall
        if name == "session_256":
            res["session_capacity"] = out["capacity"]
        res[name + "_max_templates"] = int(out["created"].sum(axis=1).max())
        del out
    res["one_call_over_session_memory"] = (res["one_call_max_memory_allocated_bytes"]
                                           / res["session_256_max_memory_allocated_bytes"])
    return res


def long_recording():
    import torch
    from synth import synth_frames
    from pyratslam_b200.ros_ensemble import EnsembleSession
    S, T, K, chunk = 256, 100000, 300, 4096
    thr, gi = settings(S)
    rng = np.random.default_rng(11)
    base = synth_frames(rng, K)
    s = EnsembleSession(match_threshold=thr, global_inhibition=gi, inject_energy=ENERGY)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    feed_s = 0.0
    for t in range(0, T, chunk):
        n = min(chunk, T - t)
        fr, od = base[np.arange(t, t + n) % K], odometry(rng, n)
        t1 = time.perf_counter()
        s.feed(fr, od)
        feed_s += time.perf_counter() - t1
    wall = time.perf_counter() - t0
    res = {"agents": S, "frames": T, "places": K, "chunk": chunk, "wall_s_with_frame_generation": wall,
           "feed_s": feed_s, "agent_frames_per_s_in_feed": S * T / feed_s, "capacity": s.capacity,
           "n_templates_min": int(s.n_templates.min()), "n_templates_max": int(s.n_templates.max()),
           "frames_fed": int(s.frames_fed[0])}
    s.close()
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_session.py measures on the GPU; no CUDA device is visible")
    one, many = recordings(1, 1000), recordings(16, 1000)
    one_call([f[:20] for f in many[0][:2]], [o[:20] for o in many[1][:2]], 4)      # warm-up
    session([one[0][0][:40]], [one[1][0][:40]], 4, 16)
    res = {"a_1x1024": chunk_cost(one[0], one[1], 1024, a.repeats),
           "a_16x16": chunk_cost(many[0], many[1], 16, a.repeats)}
    del one, many
    res["b_memory"] = memory(a.repeats)
    res["c_100000_frames"] = long_recording()
    out = dict(gpu_info())
    out.update({"metric": "agent-frames/s (wall clock, setup included)", "inject_energy": ENERGY,
                "repeats": a.repeats, "results": res})
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
