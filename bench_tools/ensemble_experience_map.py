"""Ensemble experience maps: every agent's linked map built on the device against the host replay of the maps.

A 1000-frame recording in which loops close (tests/golden/em_records.py:loop_recording: periods of 40 synthetic frames
under random odometry, then 60 frames that cycle six fixed views while the twist stays just above the 0.001 gate) runs
through B in {1, 64, 256, 1024} agents with experience_links=True; the match thresholds (30000..60000) and global
inhibitions (0.05..0.25) are spread over the agents as in ensemble_replay.py.  Prints one JSON line with the GPU's name
and power limit read in the same run:

* the wall clock of replay_ensemble with experience_map=False and with "device" (warmed up, median of --repeats runs,
  run alternately);
* the map step on its own: ensemble_experience_maps(linked=True) on the replay's records, as wall clock (record upload,
  kernel and result download included, median of --repeats), as a share of the replay's wall clock without maps, and
  as the device time of its kernel (k_em_linked, torch.profiler, one run of its own afterwards; --profile OUT writes
  that run's table of kernels and copies per B);
* the host path (ros_ensemble._experience_maps, linked) measured at B = 1 and 64 and extrapolated linearly to
  B x 1000 frames, labelled as extrapolated;
* the loop closures and experiences per agent, and a check, in the same run, that sampled agents' device maps equal
  host ExperienceMap(linked=True) maps: structure exact, positions and link geometry within 1e-9.

    python bench_tools/ensemble_experience_map.py [--frames 1000] [--repeats 3] [--agents 1,64,256,1024] [--profile OUT]
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

SHAPE = (21, 21, 36)
HOST_AGENTS = (1, 64)


def params(B):
    return np.linspace(30000, 60000, B), np.linspace(0.05, 0.25, B)


def ensemble(frames, odom, B, experience_map):
    from pyratslam_b200.ros_ensemble import replay_ensemble
    thr, gi = params(B)
    return replay_ensemble(frames, odom, match_threshold=thr, global_inhibition=gi, experience_map=experience_map,
                           experience_links=True)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--agents", default="1,64,256,1024")
    ap.add_argument("--profile", default=None, help="write the map step's torch.profiler table per B here")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_experience_map.py measures on the GPU; no CUDA device is visible")
    from em_records import assert_same_map, host_maps, loop_recording
    from pyratslam_b200.experience_ensemble import ensemble_experience_maps, gate
    from pyratslam_b200.ros_ensemble import _experience_maps
    T = a.frames
    Bs = [int(b) for b in a.agents.split(",")]
    frames, odom = loop_recording(np.random.default_rng(1), T)
    moved, tw = gate(odom)

    for B in Bs:                # warm-up: module load, lazy kernel attributes, graph capture paths
        for em in (False, "device"):
            ensemble(frames[:20], odom[:20], B, em)
    replay_t = {(B, em): [] for B in Bs for em in (False, "device")}
    map_t = {B: [] for B in Bs}
    outs = {}
    for _ in range(a.repeats):
        for B in Bs:
            for em in (False, "device"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = ensemble(frames, odom, B, em)
                replay_t[(B, em)].append(time.perf_counter() - t0)      # replay_ensemble returns with host arrays
                if em == "device":
                    outs[B] = out
                del out
            o = outs[B]
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ensemble_experience_maps(o["template"], o["argmax"], odom, SHAPE, linked=True)
            map_t[B].append(time.perf_counter() - t0)

    host = {}
    for B in HOST_AGENTS:
        o = outs.get(B) or ensemble(frames, odom, B, "device")
        t0 = time.perf_counter()
        _experience_maps(o, moved, tw, SHAPE, True)
        host[B] = time.perf_counter() - t0

    checks = {}
    for B, o in outs.items():
        sample = sorted({0, B // 2, B - 1})
        maps, n_exp, exp_id, em_xy = host_maps(o["template"][sample], o["argmax"][sample], odom, SHAPE)
        for j, b in enumerate(sample):
            assert np.array_equal(o["n_exp"][b], n_exp[j]) and np.array_equal(o["exp_id"][b], exp_id[j]), (B, b)
            assert np.abs(o["em_xy"][b] - em_xy[j]).max() <= 1e-9, (B, b)
            assert_same_map(o["maps"].experience_map(b), maps[j], what=(B, b))
        closures, n_final = o["n_loop_closures"], o["n_exp"][:, -1]
        checks["B%d" % B] = ("agents %s equal host linked maps; loop closures min/mean/max %d/%.0f/%d, experiences "
                             "min/mean/max %d/%.0f/%d" % (sample, closures.min(), closures.mean(), closures.max(),
                                                          n_final.min(), n_final.mean(), n_final.max()))

    from torch.profiler import ProfilerActivity, profile
    kernel_ms, tables = {}, []
    for B, o in outs.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ensemble_experience_maps(o["template"], o["argmax"], odom, SHAPE, linked=True)
        kernel_ms[B] = sum(e.device_time_total for e in prof.key_averages() if "k_em_linked" in e.key) / 1e3
        tables.append("# B = %d agents, %d frames: ensemble_experience_maps(linked=True), k_em_linked %.3f ms\n%s\n"
                      % (B, T, kernel_ms[B], prof.key_averages().table(sort_by="cuda_time_total", row_limit=10)))

    per_af = {B: host[B] / (B * T) for B in host}
    res = {}
    for B in Bs:
        off, dev = float(np.median(replay_t[(B, False)])), float(np.median(replay_t[(B, "device")]))
        res["B%d" % B] = {
            "replay_s_experience_map_false": off, "replay_s_experience_map_device": dev,
            "device_map_share_of_replay": (dev - off) / off,
            "map_step_wall_s": float(np.median(map_t[B])), "map_step_share_of_replay": float(np.median(map_t[B])) / off,
            "map_step_kernel_ms": kernel_ms[B],
            "host_linked_map_s_extrapolated": per_af[max(per_af)] * B * T,
        }
    out = dict(gpu_info())
    out.update({"metric": "seconds (wall clock, median of repeats)", "frames": T, "repeats": a.repeats,
                "host_linked_map_us_per_agent_frame_measured": {"B%d" % B: v * 1e6 for B, v in per_af.items()},
                "results": res, "record_checks": checks})
    print(json.dumps(out), flush=True)
    if a.profile:
        os.makedirs(os.path.dirname(os.path.abspath(a.profile)), exist_ok=True)
        with open(a.profile, "w") as f:
            f.writelines(tables)


if __name__ == "__main__":
    main()
