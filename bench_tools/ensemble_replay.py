"""Ensemble replay (ros_ensemble.replay_ensemble): one recording through B agents against B single-agent replays.

The bench's 1000-frame synthetic replay (synth_frames with default_rng(1), the odometry of inject_replay.py) runs
through B in {1, 16, 64, 256, 1024} agents whose match thresholds (30000..60000) and global inhibitions (0.05..0.25,
BASELINE config 4) are spread over the agents, once without injection and once with inject_energy 0.02 for every
agent.  Prints one JSON line with the GPU's name and power limit read in the same run:

* agent-frames/s (B x frames / wall clock of replay_ensemble, warmed up, setup included; median of --repeats runs);
* the ratio to B x the measured frames/s of one single-agent ``replay(native=True)``: an extrapolation of running the
  agents one after another, not a measured B-agent run;
* a check, in the same run, that a sample of agents has the records of single-agent native replays with their
  parameters.

--profile OUT: afterwards, separate torch.profiler runs (one per B, with injection) write their kernel tables to OUT,
with the batched sweep's bytes/s: sum over frames and agents of the library size n_b x 1088 bytes (the packed
template's size) over the sweep kernel's total time.

    python bench_tools/ensemble_replay.py [--frames 1000] [--repeats 2] [--agents 1,16,64,256,1024] [--profile OUT]
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

ENERGIES = (None, 0.02)
TEMPLATE_BYTES = 1088           # one template of the packed library: 32 rows x 32 bytes + its row sums
HBM_BYTES_PER_S = 7.7e12        # one B200, NVIDIA's data sheet (HGX B200)


def params(B):
    return np.linspace(30000, 60000, B), np.linspace(0.05, 0.25, B)


def single(frames, odom, thr, gi, energy):
    """Records of one agent by the single-agent native replay (prs_replay_run), with its global inhibition."""
    from pyratslam_b200 import ros_simulate
    node = ros_simulate.RatslamRos(match_threshold=thr, inject_energy=energy)
    node.pcn.global_inhibition = gi
    res = node.replay_native(frames, odom)
    return res["template_index"].astype(np.int64), res["created"] != 0, res["argmax"]


def ensemble(frames, odom, B, energy, **kw):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    thr, gi = params(B)
    return replay_ensemble(frames, odom, match_threshold=thr, global_inhibition=gi, inject_energy=energy, **kw)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--agents", default="1,16,64,256,1024")
    ap.add_argument("--profile", default=None, help="write torch.profiler kernel tables and the sweep's bytes/s here")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_replay.py measures on the GPU; no CUDA device is visible")
    from synth import synth_frames
    from pyratslam_b200 import ros_simulate
    T = a.frames
    Bs = [int(b) for b in a.agents.split(",")]
    frames = synth_frames(np.random.default_rng(1), T)
    rng = np.random.default_rng(1)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)

    for energy in ENERGIES:     # warm-up: module load, lazy kernel attributes, graph capture paths
        ros_simulate.replay(frames[:20], odom[:20], native=True, inject_energy=energy)
        for B in Bs:
            ensemble(frames[:20], odom[:20], B, energy)
    single_t = {e: [] for e in ENERGIES}
    ens_t = {(B, e): [] for B in Bs for e in ENERGIES}
    outs = {}
    for _ in range(a.repeats):
        for energy in ENERGIES:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ros_simulate.replay(frames, odom, native=True, inject_energy=energy)
            single_t[energy].append(time.perf_counter() - t0)
            for B in Bs:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = ensemble(frames, odom, B, energy)
                ens_t[(B, energy)].append(time.perf_counter() - t0)     # replay_ensemble returns after its last sync
                outs[(B, energy)] = out
                del out

    checks = {}
    for (B, energy), out in outs.items():
        thr, gi = params(B)
        sample = sorted({0, B // 2, B - 1})
        for b in sample:
            tpl, created, flat = single(frames, odom, float(thr[b]), float(gi[b]), energy)
            assert np.array_equal(out["template"][b], tpl), (B, energy, b)
            assert np.array_equal(out["created"][b], created), (B, energy, b)
            X, Y, Th = 21, 21, 36
            amax = np.stack([flat // (Y * Th), (flat // Th) % Y, flat % Th], axis=1)
            assert np.array_equal(out["argmax"][b], amax), (B, energy, b)
        checks["B%d_inject_%s" % (B, energy)] = ("agents %s identical to single-agent native replays; templates "
                                                 "min/mean/max %d/%.0f/%d" % (sample, out["n_templates"].min(),
                                                                             out["n_templates"].mean(),
                                                                             out["n_templates"].max()))
    outs.clear()

    res = {}
    for energy in ENERGIES:
        s_fps = T / float(np.median(single_t[energy]))
        row = {"single_agent_native_frames_per_s": s_fps}
        for B in Bs:
            ts = ens_t[(B, energy)]
            afps = B * T / float(np.median(ts))
            row["B%d" % B] = {"agent_frames_per_s": afps, "min": B * T / max(ts), "max": B * T / min(ts),
                              "over_B_x_single_agent_native_extrapolated": afps / s_fps}
        res["inject_%s" % energy] = row
    out = dict(gpu_info())
    out.update({"metric": "agent-frames/s (wall clock of replay_ensemble, setup included)", "frames": T,
                "repeats": a.repeats, "results": res, "record_checks": checks})
    print(json.dumps(out), flush=True)

    if a.profile:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(os.path.dirname(os.path.abspath(a.profile)), exist_ok=True)
        with open(a.profile, "w") as f:
            for B in Bs:
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    o = ensemble(frames, odom, B, 0.02)
                # the library size each frame's sweep saw: the size after the frame minus its own append
                swept = int((np.cumsum(o["created"], axis=1) - o["created"]).sum())
                sweep_us = sum(e.device_time_total for e in prof.key_averages()
                               if e.key.startswith("k_vt_sweep_packed_ref_small"))
                bps = swept * TEMPLATE_BYTES / (sweep_us * 1e-6) if sweep_us else float("nan")
                f.write("# B = %d agents, %d frames, inject_energy 0.02: sweep of %d templates in all (%.3g GB), "
                        "k_vt_sweep_packed_ref_small %.3f ms in all -> %.3g GB/s (%.2f%% of %.1f TB/s HBM; the "
                        "libraries %s the 126 MB L2)\n"
                        % (B, T, swept, swept * TEMPLATE_BYTES / 1e9, sweep_us / 1e3, bps / 1e9,
                           100 * bps / HBM_BYTES_PER_S, HBM_BYTES_PER_S / 1e12,
                           "fit" if o["n_templates"].sum() * TEMPLATE_BYTES < 126e6 else "exceed"))
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=14))
                f.write("\n")
                del o


if __name__ == "__main__":
    main()
