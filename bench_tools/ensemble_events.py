"""Message-stream ensemble replay (replay_ensemble_events): what replaying every odometry message costs.

Prints one JSON line with the GPU's name and power limit read in the same run:

* (a) rate: agent-messages/s (B x (odometry messages + images) / wall clock, setup included, median of --repeats) of
  replay_ensemble_events on one recording of 1000 images with 1, 3 and 5 gated odometry messages before each image,
  at B = 16, 256 and 1024 settings.
* (b) the odometry-only tick: (time at 5 messages per image - time at 1) / 4000, the marginal cost of one tick without
  an image, against a bare PoseCellEnsemble update of the same B networks (update_async over device odometry, CUDA
  events around 2000 updates after a warm-up), which is its floor.
* (c) where both paths apply, an alternating stream (one twist, one image): replay_ensemble_events against
  replay_ensemble on rosbag_io.events_to_arrays of the same stream, alternated in one run, and whether every agent's
  records (template, created, arg-max) are identical across the two.

    python bench_tools/ensemble_events.py [--repeats 3] > profiles/r7_ensemble_events.txt
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

from ensemble_session import settings  # noqa: E402
from inject_replay import gpu_info  # noqa: E402

ENERGY = 0.02
IMAGES = 1000
RATES = (1, 3, 5)
AGENTS = (16, 256, 1024)


def stream(per_image, T=IMAGES, seed=300):
    """T synthetic images (with revisits), each after ``per_image`` twists above the 0.001 gate."""
    from synth import synth_frames
    rng = np.random.default_rng(seed)
    frames = synth_frames(rng, T)
    ev, ns = [], 0
    for t in range(T):
        for _ in range(per_image):
            ns += 1000
            ev.append(("odom", (ns // 10 ** 9, ns % 10 ** 9), (float(rng.uniform(0.1, 3)), float(rng.uniform(-1, 1)))))
        ns += 1000
        ev.append(("image", (ns // 10 ** 9, ns % 10 ** 9), frames[t]))
    return ev


def timed(fn, repeats):
    import torch
    out, ts = None, []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return out, ts


def bare_update_s(B, n=2000):
    """Seconds per PoseCellEnsemble update of B networks (device odometry, no host synchronisation per update)."""
    import torch
    from pyratslam_b200.posecell_network import PoseCellEnsemble
    _, gi = settings(B)
    ens = PoseCellEnsemble((21, 21, 36), B, global_inhibition=np.array(gi), device=torch.device("cuda", 0))
    ens.inject(1, (10, 10, 18))
    rng = np.random.default_rng(7)
    od = torch.from_numpy(np.stack([rng.uniform(0.01, 0.3, B), rng.uniform(-0.1, 0.1, B)], axis=1)).cuda()
    for _ in range(50):
        ens.update_async(od)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        ens.update_async(od)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / n, ens.path


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--repeats", type=int, default=3)
    a = ap.parse_args(argv)
    import torch
    from pyratslam_b200 import rosbag_io as rb
    from pyratslam_b200.ros_ensemble import replay_ensemble, replay_ensemble_events
    torch.cuda.set_device(0)
    res = {}
    streams = {k: stream(k) for k in RATES}
    for B in AGENTS:
        thr, gi = settings(B)
        kw = dict(match_threshold=thr, global_inhibition=gi, inject_energy=ENERGY)
        replay_ensemble_events(stream(1, 40, seed=1), **kw)                     # warm-up: the plans' graphs, the module
        row = {"agents": B, "images": IMAGES}
        secs = {}
        for k in RATES:
            _, ts = timed(lambda: replay_ensemble_events(streams[k], **kw), a.repeats)
            secs[k] = float(np.median(ts))
            row["rate_%d" % k] = {"messages": IMAGES * (k + 1), "s": ts,
                                  "agent_messages_per_s": B * IMAGES * (k + 1) / secs[k]}
        tick = (secs[5] - secs[1]) / (4 * IMAGES)
        floor, path = bare_update_s(B)
        row["odometry_only_tick"] = {"marginal_s": tick, "bare_update_s": floor, "over_bare_update": tick / floor,
                                     "pose_cell_path": path}
        frames, odom, _ = rb.events_to_arrays(streams[1])
        ev_s, arr_s, ev_out, arr_out = [], [], None, None
        for _ in range(a.repeats):                                               # alternated
            ev_out, t = timed(lambda: replay_ensemble_events(streams[1], **kw), 1)
            ev_s += t
            arr_out, t = timed(lambda: replay_ensemble(frames, odom, **kw), 1)
            arr_s += t
        same = [b for b in range(B) if not all(np.array_equal(ev_out[k][b], arr_out[k][b])
                                               for k in ("template", "created", "argmax"))]
        row["alternating"] = {"events_s": ev_s, "arrays_s": arr_s,
                              "events_over_arrays": float(np.median(ev_s) / np.median(arr_s)),
                              "records_identical": not same, "differing_agents": same[:10]}
        res["B%d" % B] = row
    print(json.dumps(dict(gpu_info(), metric="agent-messages/s (wall clock, setup included)", inject_energy=ENERGY,
                          repeats=a.repeats, results=res)))


if __name__ == "__main__":
    main()
