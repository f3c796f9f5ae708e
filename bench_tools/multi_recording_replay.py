"""Multi-recording ensemble replay: R recordings x S settings as one replay_ensemble call against R sequential calls.

R in {1, 4, 16, 64} synthetic recordings of --frames frames each (synth_frames with default_rng(100 + r), odometry that
moves on every frame), S = 16 settings (match thresholds 30000..60000, global inhibitions 0.05..0.25, injection 0.02):
B = R x S agents.  Prints one JSON line with the GPU's name and power limit read in the same run:

* agent-frames/s of one call with ``recording=`` (B x frames / wall clock of replay_ensemble, setup included, median of
  --repeats runs) and of R sequential single-recording calls of S agents each, and their ratio -- both measured;
* whether every agent's records (template, created, arg-max) are identical between the two.  Checked with the
  resident pose-cell kernel forced on both sides, whose per-network arithmetic does not depend on B: with the automatic
  choice the one call (resident at B >= 256) and the 16-agent calls (cluster) sum the pose cells in a different order,
  and an arg-max near a tie can move by one cell; those differences are counted and reported as well;
* the cost of a mixed frame (some recording still or ended, so the pose-cell update saves and restores the networks
  of the others), at R = 16: (a) the recordings as above, no mixed frame; (b) the same frames with recording r still
  for 8 frames starting at frame 12 r, which makes 8 R frames mixed and leaves the sweep's work as it was;
  (c) recording r ending after frames x (1 - r / (2 R)), so that every frame after the first end is mixed.  The cost
  per mixed frame is (wall(b) - wall(a)) / mixed frames; (c) reports its agent-frames/s over the frames that exist.

    python bench_tools/multi_recording_replay.py [--frames 500] [--repeats 2] [--recordings 1,4,16,64]
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

S = 16
ENERGY = 0.02


def settings():
    return np.linspace(30000, 60000, S), np.linspace(0.05, 0.25, S)


def recordings(R, T):
    from synth import synth_frames
    frames, odom = [], []
    for r in range(R):
        rng = np.random.default_rng(100 + r)
        frames.append(synth_frames(rng, T))
        odom.append(np.stack([rng.uniform(0.1, 3, T), rng.uniform(-1, 1, T)], axis=1))
    return frames, odom


def one_call(frames, odom):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    R = len(frames)
    thr, gi = settings()
    return replay_ensemble(frames, odom, recording=np.repeat(np.arange(R), S), match_threshold=np.tile(thr, R),
                           global_inhibition=np.tile(gi, R), inject_energy=ENERGY)


def sequential(frames, odom):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    thr, gi = settings()
    return [replay_ensemble(f, o, match_threshold=thr, global_inhibition=gi, inject_energy=ENERGY)
            for f, o in zip(frames, odom)]


class forced_path:
    """Within the block every PoseCellEnsemble that replay_ensemble creates uses the given kernel family."""

    def __init__(self, path):
        self.path = path

    def __enter__(self):
        from pyratslam_b200 import ros_ensemble
        self.orig, path = ros_ensemble.PoseCellEnsemble, self.path

        class Forced(self.orig):
            def __init__(self, *a, **k):
                super().__init__(*a, **k)
                self.force_path(path)
        ros_ensemble.PoseCellEnsemble = Forced

    def __exit__(self, *exc):
        from pyratslam_b200 import ros_ensemble
        ros_ensemble.PoseCellEnsemble = self.orig


def differing(one, seq, R, T):
    """[(recording, setting, field, first frame)] where the one call's records differ from the sequential calls'."""
    bad = []
    for r in range(R):
        for s in range(S):
            for k in ("template", "created", "argmax"):
                a, w = one[k][r * S + s], seq[r][k][s]
                if not np.array_equal(a, w):
                    bad.append((r, s, k, int(np.argwhere((a != w).reshape(T, -1).any(axis=1))[0][0])))
    return bad


def timed(fn, *args):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn(*args)
    return time.perf_counter() - t0, out      # replay_ensemble returns after its last synchronisation


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=500)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--recordings", default="1,4,16,64")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("multi_recording_replay.py measures on the GPU; no CUDA device is visible")
    T = a.frames
    Rs = [int(r) for r in a.recordings.split(",")]
    frames, odom = recordings(max(Rs + [16]), T)

    one_call([f[:20] for f in frames[:2]], [o[:20] for o in odom[:2]])      # warm-up: module load, graph paths
    sequential([frames[0][:20]], [odom[0][:20]])
    res, checks = {}, {}
    for R in Rs:
        t_one, t_seq = [], []
        for _ in range(a.repeats):
            t, one = timed(one_call, frames[:R], odom[:R])
            t_one.append(t)
            t, seq = timed(sequential, frames[:R], odom[:R])
            t_seq.append(t)
        auto = differing(one, seq, R, T)
        del one, seq
        with forced_path("resident"):
            same = not differing(one_call(frames[:R], odom[:R]), sequential(frames[:R], odom[:R]), R, T)
        checks["R%d" % R] = {"identical_with_the_resident_kernel_on_both_sides": same,
                             "differing_agents_automatic_kernels": len({(r, s) for r, s, _, _ in auto}),
                             "differences_automatic_kernels": auto[:8]}
        assert same, R
        B = R * S
        one_fps, seq_fps = B * T / float(np.median(t_one)), B * T / float(np.median(t_seq))
        res["R%d" % R] = {"agents": B, "one_call_agent_frames_per_s": one_fps,
                          "sequential_agent_frames_per_s": seq_fps, "one_call_over_sequential": one_fps / seq_fps,
                          "one_call_s": sorted(t_one), "sequential_s": sorted(t_seq)}

    # mixed frames at R = 16
    R = 16
    fr, od = frames[:R], odom[:R]
    still = [o.copy() for o in od]
    n_mixed = 0
    for r in range(R):
        still[r][12 * r:12 * r + 8] = 0.0
    mixed = np.zeros(T, bool)
    for r in range(R):
        mixed[12 * r:12 * r + 8] = True
    n_mixed = int(mixed[:T].sum())
    ends = [int(T * (1 - r / (2 * R))) for r in range(R)]
    t_a, t_b, t_c = [], [], []
    for _ in range(a.repeats):
        t_a.append(timed(one_call, fr, od)[0])
        t_b.append(timed(one_call, fr, still)[0])
        t_c.append(timed(one_call, [f[:e] for f, e in zip(fr, ends)], [o[:e] for o, e in zip(od, ends)])[0])
    ta, tb, tc = (float(np.median(x)) for x in (t_a, t_b, t_c))
    mixed_c = T - min(ends)
    res["mixed_R16"] = {
        "agents": R * S,
        "a_no_mixed_s": sorted(t_a), "b_still_windows_s": sorted(t_b), "c_staggered_ends_s": sorted(t_c),
        "b_mixed_frames": n_mixed, "cost_per_mixed_frame_us": (tb - ta) / n_mixed * 1e6,
        "cost_per_mixed_frame_us_from_minima": (min(t_b) - min(t_a)) / n_mixed * 1e6,
        "per_frame_us_a": ta / T * 1e6,
        "c_mixed_frames": mixed_c, "c_agent_frames": S * sum(ends),
        "c_agent_frames_per_s": S * sum(ends) / tc, "a_agent_frames_per_s": R * S * T / ta}
    out = dict(gpu_info())
    out.update({"metric": "agent-frames/s (wall clock of replay_ensemble, setup included)", "frames": T,
                "settings_per_recording": S, "inject_energy": ENERGY, "repeats": a.repeats, "results": res,
                "record_checks": checks})
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
