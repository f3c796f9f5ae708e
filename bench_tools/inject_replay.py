"""Frame replay with and without the view-template -> pose-cell injection (ros_simulate.py:106-108), in every mode.

The bench's 1000-frame synthetic replay (synth_frames with default_rng(1), the same odometry as bench.py) is run with
inject_energy None and 0.02 by the reference-shaped calls (the host injects), fused_frame, the pipelined plans and the
native loop (prs_replay_run).  Before printing, the records of all modes are checked to be identical for each energy.
Prints one JSON line: frames/s per mode and energy (median of --repeats runs, modes alternated within a repeat, plus
the spread), with the GPU's name and power limit read in the same run.  The cost of the injection node is native with
injection against native without; the gain is every injected mode against the reference-shaped injected run.

    python bench_tools/inject_replay.py [--frames 1000] [--repeats 3] [--profile OUT.txt]

--profile: afterwards, a separate torch.profiler run of the native replay with injection writes its kernel table to
OUT.txt (the timed runs are not profiled).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

MODES = {"reference_shaped": {}, "fused": {"fused": True}, "pipelined": {"fused": True, "pipelined": True},
         "native": {"native": True}}
ENERGIES = (None, 0.02)
KEYS = ("template", "created", "argmax", "n_exp", "em_xy")


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        power, clock = (s.strip() for s in out[0].split(","))
    except Exception:  # noqa: BLE001 - reported as unknown, the timings do not depend on it
        power = clock = None
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--profile", default=None, help="write a torch.profiler kernel table of a native injected run here")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("inject_replay.py measures on the GPU; no CUDA device is visible")
    from synth import synth_frames
    from pyratslam_b200 import ros_simulate
    T = a.frames
    frames = synth_frames(np.random.default_rng(1), T)
    rng = np.random.default_rng(1)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)

    for energy in ENERGIES:     # warm-up: module load, lazy kernel attributes, graph capture paths
        for kw in MODES.values():
            ros_simulate.replay(frames[:20], odom[:20], inject_energy=energy, **kw)
    times = {(m, e): [] for m in MODES for e in ENERGIES}
    records = {}
    for _ in range(a.repeats):
        for energy in ENERGIES:
            for mode, kw in MODES.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rec = ros_simulate.replay(frames, odom, inject_energy=energy, **kw)
                times[(mode, energy)].append(time.perf_counter() - t0)   # replay() returns after its last sync
                records[(mode, energy)] = rec

    checks = {}
    for energy in ENERGIES:
        ref = records[("reference_shaped", energy)]
        for mode in MODES:
            rec = records[(mode, energy)]
            for k in KEYS:
                assert np.array_equal(rec[k], ref[k]), (mode, energy, k)
            assert rec["n_templates"] == ref["n_templates"], (mode, energy)
        checks[str(energy)] = "records identical in all %d modes (%d templates)" % (len(MODES), ref["n_templates"])

    fps = {}
    for (mode, energy), ts in times.items():
        med = float(np.median(ts))
        fps.setdefault("inject_%s" % energy, {})[mode] = {"frames_per_s": T / med, "min": T / max(ts), "max": T / min(ts)}
    inj, plain = fps["inject_0.02"], fps["inject_None"]
    out = dict(gpu_info())
    out.update({"metric": "end-to-end frames/s (wall clock, node construction included)", "frames": T,
                "repeats": a.repeats, "frames_per_s": fps, "record_checks": checks,
                "native_inject_over_native": inj["native"]["frames_per_s"] / plain["native"]["frames_per_s"],
                "injected_over_reference_shaped_injected": {
                    m: inj[m]["frames_per_s"] / inj["reference_shaped"]["frames_per_s"] for m in MODES}})
    print(json.dumps(out))

    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            ros_simulate.replay(frames[:200], odom[:200], native=True, inject_energy=0.02)
        os.makedirs(os.path.dirname(os.path.abspath(a.profile)), exist_ok=True)
        with open(a.profile, "w") as f:
            f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))


if __name__ == "__main__":
    main()
