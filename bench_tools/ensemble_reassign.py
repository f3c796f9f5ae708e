"""Ensemble sessions: what EnsembleSession.reassign costs at B = 1024 when half the agents become copies of the other
half, against the device's copy bandwidth and against one 256-frame feed of the same session.

A negative match threshold creates a template on every frame, so after F frames every agent holds F templates; the
reassign is measured at about 1000 and about 5000 templates per agent.  Per size, one JSON line: the device time of
the call between CUDA events on the current stream and its wall clock up to a device synchronise (median of
--repeats), the live bytes the copies move (per child: its parent's state slice, pc_work slots and count, library
groups of n templates and n locations), their rate, the same rate over the copy bandwidth of a 4 GiB device-to-device
torch copy measured in the same run, and the wall clock of the 256-frame feed that follows.  The first line holds the
GPU's name and power limit, read in the same run.  No linked maps: the library bytes dominate.

    python bench_tools/ensemble_reassign.py [--repeats 5] > profiles/r9_ensemble_reassign.txt
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

B = 1024
FEED = 256
GROUP_BYTES = 34816


def copy_bandwidth(torch, repeats):
    """Bytes per second of a 4 GiB device-to-device copy (each byte counted once), median over `repeats`."""
    src = torch.empty(4 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src)
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) / 1e3)
    del src, dst
    return float(4 << 30) / float(np.median(times))


def live_bytes(s, parents):
    """The bytes the copies of one reassign move, from the host's counts: per child its parent's live rows."""
    X, Y, Th = s.pose_size
    net = X * Y * Th * np.dtype(s._ens.np_dtype).itemsize
    total = 0
    for b, p in enumerate(parents):
        if p != b:
            n = int(s.n_templates[p])
            total += net + 24 + 4 + (n + 31) // 32 * GROUP_BYTES + 8 * n
    return total


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--sizes", default="1000,5000", help="templates per agent at which reassign is measured")
    a = ap.parse_args(argv)
    import torch
    from synth import synth_frames
    from pyratslam_b200.ros_ensemble import EnsembleSession, capacity_for
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_reassign.py measures on the GPU; no CUDA device")
    sizes = [int(v) for v in a.sizes.split(",")]
    T = sizes[-1] + FEED * len(sizes)
    rng = np.random.default_rng(17)
    frames = synth_frames(rng, T)
    odom = np.stack([rng.uniform(0.1, 3, T), rng.uniform(-1, 1, T)], axis=1)
    print(json.dumps(dict(gpu_info(), agents=B)), flush=True)
    bw = copy_bandwidth(torch, a.repeats)
    s = EnsembleSession(B, match_threshold=-1.0, global_inhibition=list(np.linspace(0.05, 0.25, B)),
                        inject_energy=0.02, capacity=capacity_for(T), active_set=2)
    parents = list(range(B // 2)) + list(range(B // 2))     # agents B/2.. become copies of agents 0..B/2-1
    t = 0
    for n in sizes:
        need = n - int(s.n_templates.max())
        s.feed(frames[t:t + need], odom[t:t + need])
        t += need
        assert (s.n_templates == n).all(), s.n_templates[:4]
        moved = live_bytes(s, parents)
        s.reassign(parents)                                  # warm-up: first launches of the copy kernels
        torch.cuda.synchronize()
        dev, wall = [], []
        for _ in range(a.repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            w0 = time.perf_counter()
            e0.record()
            s.reassign(parents)
            e1.record()
            torch.cuda.synchronize()
            wall.append(time.perf_counter() - w0)
            dev.append(e0.elapsed_time(e1) / 1e3)
        w0 = time.perf_counter()
        s.feed(frames[t:t + FEED], odom[t:t + FEED])
        torch.cuda.synchronize()
        feed_s = time.perf_counter() - w0
        t += FEED
        d, w = float(np.median(dev)), float(np.median(wall))
        print(json.dumps({"templates_per_agent": n, "moves": B // 2, "live_bytes": moved,
                          "reassign_device_ms": round(d * 1e3, 3), "reassign_wall_ms": round(w * 1e3, 3),
                          "reassign_GBps_device": round(moved / d / 1e9, 1),
                          "copy_bandwidth_GBps": round(bw / 1e9, 1), "share_of_copy_bandwidth": round(moved / d / bw, 3),
                          "feed_256_frames_wall_ms": round(feed_s * 1e3, 1),
                          "reassign_over_feed": round(w / feed_s, 4)}), flush=True)
    s.close()


if __name__ == "__main__":
    main()
