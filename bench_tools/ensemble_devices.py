"""Ensemble replay split over devices (replay_ensemble(devices=...), ShardedEnsembleSession): agent-frames/s at 1, 2, 4
and 8 devices, up to the devices visible.

The bench's synthetic frames (synth_frames, the odometry of ensemble_replay.py; recording r seeded with r + 1), 1000 per
recording, through:

* one recording x B = 1024 and 4096 agents (match thresholds 30000..60000, global inhibitions 0.05..0.25, spread);
* 16 recordings x 64 settings (B = 1024);

each at devices = None (one device, today's path), [0] (the sharded wrapper on one device: its overhead) and
list(range(n)) for n in 1, 2, 4, 8.  Agent-frames/s is B x frames over the wall clock of replay_ensemble, setup
included, warmed up; the device counts alternate inside each of --repeats rounds and the median is reported.  Then
one cross-device reassign at B = 1024: a session on two devices (two shards on device 0 when only one is visible) fed
200 frames, half the agents re-parented onto agents of the other shard, timed with CUDA events on device 0 around the
call (the call ends with a synchronise of every device) and with the host clock.  Prints the card's name and power
limit read in the same run, then one line per case.

    python bench_tools/ensemble_devices.py [--frames 1000] [--repeats 3] [--out FILE]
"""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, os.path.join(ROOT, "bench_tools"))

from inject_replay import gpu_info  # noqa: E402


def recording(seed, T):
    from synth import synth_frames
    frames = synth_frames(np.random.default_rng(seed), T)
    rng = np.random.default_rng(seed)
    return frames, np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)


def settings(B):
    return dict(match_threshold=np.linspace(30000, 60000, B), global_inhibition=np.linspace(0.05, 0.25, B))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the lines to this file")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("ensemble_devices.py measures on the GPU; no CUDA device is visible")
    from pyratslam_b200.ros_ensemble import ShardedEnsembleSession, replay_ensemble
    n_dev = torch.cuda.device_count()
    T = a.frames
    one = recording(1, T)
    many = [recording(r + 1, T) for r in range(16)]
    cases = {"1 recording x B=1024": (one[0], one[1], dict(settings(1024))),
             "1 recording x B=4096": (one[0], one[1], dict(settings(4096))),
             "16 recordings x 64 settings": ([f for f, _ in many], [o for _, o in many],
                                            dict(recording=np.repeat(np.arange(16), 64),
                                                 **{k: np.tile(v, 16) for k, v in settings(64).items()}))}
    counts = [n for n in (1, 2, 4, 8) if n <= n_dev]
    modes = [("devices=None", None), ("devices=[0]", [0])] + [("%d device(s)" % n, list(range(n))) for n in counts]
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    info = gpu_info()
    emit("# %s, power limit %s, max SM clock %s; %d device(s) visible; %d frames per recording, median of %d rounds, "
         "the modes alternated in each round" % (info["gpu"], info["power_limit"], info["max_sm_clock"], n_dev, T,
                                                 a.repeats))
    for name, (fr, od, kw) in cases.items():
        B = len(kw["match_threshold"])
        short = (fr[:20], od[:20]) if not isinstance(fr, list) else ([f[:20] for f in fr], [o[:20] for o in od])
        for _, devs in modes:       # warm-up: module load, graph capture, every device's context
            replay_ensemble(*short, devices=devs, **kw)
        times = {m: [] for m, _ in modes}
        for _ in range(a.repeats):
            for m, devs in modes:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = replay_ensemble(fr, od, devices=devs, **kw)       # returns after its last synchronise
                times[m].append(time.perf_counter() - t0)
                del out
        base = B * T / float(np.median(times["devices=None"]))
        for m, _ in modes:
            afps = B * T / float(np.median(times[m]))
            emit("%-28s %-14s %8.3f s  %.3g agent-frames/s  x%.2f of devices=None  (min %.3f s, max %.3f s)"
                 % (name, m, float(np.median(times[m])), afps, afps / base, min(times[m]), max(times[m])))

    B = 1024
    devs = [0, 1] if n_dev >= 2 else [0, 0]
    s = ShardedEnsembleSession(devs, B, **settings(B))
    s.feed(one[0][:200], one[1][:200])
    half = B // 2
    par = np.arange(B)
    par[:half] = np.arange(half, B)                   # agents 0..511 (shard 0) continue as agents 512..1023 (shard 1)
    s.reassign(np.arange(B))                          # warm-up of the call path
    torch.cuda.synchronize()
    with torch.cuda.device(0):
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        t0 = time.perf_counter()
        s.reassign(par)
        end.record()
        end.synchronize()
        wall = time.perf_counter() - t0
    s.close()
    emit("reassign across devices %s: %d of %d agents re-parented onto the other shard, %.0f templates each on average: "
         "%.3f ms (CUDA events on device 0), %.3f ms host clock" % (devs, half, B, float(s.n_templates.mean()),
                                                                   start.elapsed_time(end), wall * 1e3))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
