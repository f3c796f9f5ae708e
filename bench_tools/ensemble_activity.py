"""Pose-cell activity capture of the ensemble replay (activity_threshold): what capturing every agent's cells above 0.002
at each frame costs, and what it returns.

Prints one JSON line with the GPU's name and power limit read in the same run:

* (a) rate: agent-frames/s (B x frames / wall clock, setup included, median of --repeats) of replay_ensemble on one
  recording of --frames synthetic frames with injection, at B = 16, 256 and 1024 settings, with the capture off, on
  with max_active_cells = 128 and on with max_active_cells = 0 (counts only), the three alternated in one run; the
  on/off ratios; whether the records are identical across the three; the mean and max active-cell count per agent
  and frame; and the bytes the capture returns per frame (int32 counts, int32 index + float32 value per kept cell).
* (b) device time per image tick of the capture node (k_ens_activity) and of the per-chunk pack (k_ens_activity_scan
  + k_ens_activity_gather), next to the library sweep's, from a separate torch.profiler run of --profile-frames frames
  at B = 1024 with max_active_cells = 128.

    python bench_tools/ensemble_activity.py [--frames 1000] [--repeats 3] > profiles/r12_ensemble_activity.txt
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

from ensemble_session import odometry, settings  # noqa: E402
from inject_replay import gpu_info  # noqa: E402

ENERGY = 0.02
THR = 0.002
AGENTS = (16, 256, 1024)
MODES = (("off", None, 128), ("on_k128", THR, 128), ("on_k0", THR, 0))


def recording(T, seed=400):
    from synth import synth_frames
    rng = np.random.default_rng(seed)
    frames = synth_frames(rng, T)
    for t in range(4, T, 3):
        frames[t] = frames[t - 1]
    return frames, odometry(rng, T)


def timed(fn):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def profile(frames, odom, B, table=None):
    """Device time per image tick of the capture and pack kernels and of the sweep (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity
    from pyratslam_b200.ros_ensemble import replay_ensemble
    thr, gi = settings(B)
    kw = dict(match_threshold=thr, global_inhibition=gi, inject_energy=ENERGY, activity_threshold=THR,
              max_active_cells=128)
    replay_ensemble(frames[:40], odom[:40], **kw)
    with torch.profiler.profile(activities=[ProfilerActivity.CUDA]) as prof:
        replay_ensemble(frames, odom, **kw)
        torch.cuda.synchronize()
    sums = {"capture": [0.0, 0], "pack": [0.0, 0], "sweep": [0.0, 0]}
    for ev in prof.events():
        name = ev.name
        dt = getattr(ev, "device_time_total", None)
        if dt is None:
            dt = ev.cuda_time_total
        if not dt:
            continue
        key = ("pack" if "k_ens_activity_scan" in name or "k_ens_activity_gather" in name else
               "capture" if "k_ens_activity" in name else
               "sweep" if "k_vt_sweep" in name else None)
        if key:
            sums[key][0] += dt
            sums[key][1] += 1
    if table:
        with open(table, "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))
    T = len(frames)
    return {k: {"us_per_tick": v[0] / T, "launches": v[1]} for k, v in sums.items()}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--profile-frames", type=int, default=300)
    ap.add_argument("--kernel-table", metavar="FILE", help="also write the profiler's kernel table to FILE")
    a = ap.parse_args(argv)
    import torch
    from pyratslam_b200.ros_ensemble import replay_ensemble
    torch.cuda.set_device(0)
    frames, odom = recording(a.frames)
    res = {}
    for B in AGENTS:
        thr, gi = settings(B)
        base = dict(match_threshold=thr, global_inhibition=gi, inject_energy=ENERGY)
        for _, t, k in MODES:                                                  # warm-up: module, graphs
            replay_ensemble(frames[:40], odom[:40], activity_threshold=t, max_active_cells=k, **base)
        secs = {m: [] for m, _, _ in MODES}
        outs = {}
        for _ in range(a.repeats):                                             # alternated
            for m, t, k in MODES:
                outs[m], s = timed(lambda: replay_ensemble(frames, odom, activity_threshold=t, max_active_cells=k,
                                                           **base))
                secs[m].append(s)
        row = {"agents": B, "frames": a.frames}
        for m, _, _ in MODES:
            row[m] = {"s": secs[m], "agent_frames_per_s": B * a.frames / float(np.median(secs[m]))}
        for m in ("on_k128", "on_k0"):
            row[m]["over_off"] = float(np.median(secs[m]) / np.median(secs["off"]))
        row["records_identical"] = all(np.array_equal(outs[m][key], outs["off"][key])
                                       for m in ("on_k128", "on_k0") for key in ("template", "created", "argmax"))
        cnt = outs["on_k128"]["activity_count"]
        kept = int(outs["on_k128"]["activity_ptr"][-1])
        row["active_cells"] = {"mean": float(cnt.mean()), "max": int(cnt.max()),
                               "entries_over_128": int((cnt > 128).sum())}
        row["bytes_per_frame"] = {"k128": (cnt.size * 4 + kept * 8) / a.frames, "k0": cnt.size * 4 / a.frames,
                                  "fixed_slots_k128": B * 128 * 8}
        res["B%d" % B] = row
    prof = profile(frames[:a.profile_frames], odom[:a.profile_frames], 1024, a.kernel_table)
    print(json.dumps(dict(gpu_info(), metric="agent-frames/s (wall clock, setup included)", inject_energy=ENERGY,
                          activity_threshold=THR, repeats=a.repeats, results=res,
                          device_time_B1024=prof)))


if __name__ == "__main__":
    main()
