#!/usr/bin/env python
"""Benchmark of the pose-cell / view-template hot path on B200.

  python bench.py --gpus N --steps K --warmup W            (torchrun for N > 1, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR     (writes the last timed step's outputs as .npy)

Headline workload (config.workload): BASELINE.json config 4 -- an ensemble of 4096 independent
reference-size (21, 21, 36) pose-cell networks IN TOTAL, float32, per-network global inhibition in
[0.05, 0.25] and per-network odometry, sharded by network over the N ranks (``scaling: "strong"``:
4096 / N networks per GPU, no collective).  A *step* is one PoseCellNetwork.update() of every network.
``value`` = cell-updates/s with odometry already on the device; ``e2e`` = the same through
``PoseCellEnsemble.update_submit / update_result`` with HOST odometry (pinned H2D in, arg-max D2H out).
Every rank keeps N replicas of its shard (260 MB of state per GPU at every N, more than the 126 MB L2)
and steps them in turn, so that every timed step streams its state from HBM at every N.

Before anything is timed every rank runs tests/multigpu_check.run_checks -- sharded library and sharded
ensemble against the oracle on the ranks of this very job -- and the line carries ``parity_nranks``.

Under ``extra_sharded``: BASELINE config 5, a 2^20-template library IN TOTAL split by contiguous ranges
(strong scaling; the weak-scaling variants of both configs are reported next to it).  At N = 1 the line also
carries, under ``extra``: the library sweeps, the single 256x256x72 network, float64 and 50x50x10 ensembles,
and the frame-by-frame replay (frames/s).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = (21, 21, 36)
N_CELLS = SHAPE[0] * SHAPE[1] * SHAPE[2]
B_TOTAL = 4096
REF_CORES = 16   # the reference arm uses at most this many host cores (per-core rate reported as well)
METRIC = "pose-cell cell-updates/s"
UNIT = "cell-updates/s"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(2)
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def kernel_source_sha():
    """sha256 over the sources of the headline kernel (what a committed ncu capture must have been taken from)."""
    import hashlib
    h = hashlib.sha256()
    for f in ("posecell_resident.cu",):
        h.update(open(os.path.join(ROOT, "pyratslam_b200", "csrc", f), "rb").read())
    return h.hexdigest()


def profiled_traffic():
    """DRAM bytes per launch of the headline kernel from the committed `ncu --set full` capture
    (profiles/r2_resident_traffic.json, written by bench_tools/ncu_traffic.py in the same gpurun as the capture).
    The record carries the sha256 of the kernel sources it was measured on; a mismatch returns (None, reason)."""
    path = os.path.join(ROOT, "profiles", "r2_resident_traffic.json")
    try:
        d = json.load(open(path))
    except Exception:
        return None, "no capture committed for this round"
    if d.get("kernel_source_sha256") != kernel_source_sha():
        return None, "profiles/r2_resident_traffic.json was captured on other kernel sources (stale)"
    return float(d["dram_bytes_per_launch"]), "profiles/r2_resident_traffic.json (%s, dram__bytes_read+write per launch)" % d.get("kernel", "?")


def ensemble_inputs(B, T, seed):
    rng = np.random.default_rng(seed)
    gis = np.linspace(0.05, 0.25, B)
    odom = np.stack([rng.uniform(0.0, 0.3, (T, B)), rng.uniform(-0.1, 0.1, (T, B))], axis=-1)
    return gis, odom


# --------------------------------------------------------------------------- CPU arms
def _oracle_worker(args):
    """One host core: its own persistent networks, W untimed + K timed updates of each."""
    from oracle import posecells as opc
    gis, odom, W, K = args
    nets = []
    for g in gis:
        n = opc.PoseCellNetwork(SHAPE, global_inhibition=float(g))
        n.inject(1.0, tuple(s // 2 for s in SHAPE))
        nets.append(n)
    for t in range(W):
        for b, n in enumerate(nets):
            n.update(odom[t, b])
    t0 = time.perf_counter()
    for t in range(W, W + K):
        for b, n in enumerate(nets):
            n.update(odom[t, b])
    return time.perf_counter() - t0


def cpu_baseline(budget_s=12.0):
    """The oracle (numpy/scipy port of the reference) on ONE host core, bounded sample."""
    from oracle import posecells as opc
    gis, odom = ensemble_inputs(4, 2, 3)
    t0 = time.perf_counter()
    opc.run_ensemble(SHAPE, gis, odom)                      # warm-up + calibration: 8 network-steps
    per = (time.perf_counter() - t0) / 8
    nets = max(4, min(64, int(budget_s / (per * 5))))
    gis, odom = ensemble_inputs(nets, 5, 3)
    t0 = time.perf_counter()
    opc.run_ensemble(SHAPE, gis, odom)
    dt = time.perf_counter() - t0
    return {"value": nets * 5 * N_CELLS / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d networks x 5 updates of the %dx%dx%d grid, numpy/scipy float64 oracle" % ((nets,) + SHAPE)}


def run_reference(args):
    """--impl reference: the oracle port on min(REF_CORES, available) host cores; each step = a bounded sample of
    networks.  The core count is pinned so that the number does not float with the box; the per-core rate is printed
    as well."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    avail = len(os.sched_getaffinity(0))
    cores = min(REF_CORES, avail)
    per_core = 4                                          # networks per core (about 50 ms of CPU per step)
    nets = cores * per_core
    W, K = args.warmup, args.steps
    gis, odom = ensemble_inputs(nets, W + K, 3)
    jobs = [(gis[c * per_core:(c + 1) * per_core], odom[:, c * per_core:(c + 1) * per_core], W, K) for c in range(cores)]
    with mp.get_context("fork").Pool(cores) as pool:
        dt = max(pool.map(_oracle_worker, jobs))          # slowest core bounds the step rate
    val = nets * args.steps * N_CELLS / dt
    sample = ("each step = one update of %d persistent networks (%d per core on %d of the box's %d cores) of the %dx%dx%d "
              "grid; numpy/scipy float64 oracle port of the reference (the Python-2/OpenCL reference cannot run here)"
              % ((nets, per_core, cores, avail) + SHAPE))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "ensemble of %d-cell pose-cell networks (BASELINE config 4), CPU sample" % N_CELLS,
                       "shape": list(SHAPE), "networks_per_step": nets},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "cores_available": avail,
                             "value_per_core": val / cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# --------------------------------------------------------------------------- GPU arm
def timed(torch, dist, world, fn, steps):
    """barrier + sync, run, sync + barrier; CUDA-event milliseconds, max over ranks."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(steps):
        fn(t)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    return ms


def extra_single_gpu(torch, peak, steps):
    """Secondary workloads, N = 1 only: library sweep, large grid, frame replay."""
    from pyratslam_b200 import PoseCellNetwork, _native as nat, ros_simulate
    out = {}
    # ---- BASELINE config 5: 2^20 uint8 templates (1 GiB), reference mode and circular mode
    n = 1 << 20
    g = torch.Generator(device="cuda").manual_seed(4)
    lib = torch.randint(0, 256, (n, 32, 32), dtype=torch.uint8, device="cuda", generator=g)
    qs = torch.randint(0, 256, (8, 32, 32), dtype=torch.uint8, device="cuda", generator=g)
    key = torch.zeros(1, dtype=torch.int64, device="cuda")
    L = nat.lib()
    packed = torch.zeros(int(L.prs_vt_packed_bytes(n)), dtype=torch.uint8, device="cuda")
    nat.check(L.prs_vt_pack_u8(lib.data_ptr(), n, packed.data_ptr(), 0, nat.stream_ptr()))
    scratch = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    for mode, name, offs in ((0, "ref", 15), (1, "circular", 32)):
        def sweep(t, mode=mode):   # the product path: bit-sliced library
            nat.check(L.prs_vt_sweep_packed_u8(packed.data_ptr(), n, qs[t % 8].data_ptr(), mode, 0, key.data_ptr(), None,
                                               scratch.data_ptr(), nat.stream_ptr()))

        def sweep_bytes(t, mode=mode):   # the byte-wise SWAR kernel on the row-major library, for comparison
            nat.check(L.prs_vt_sweep_u8(lib.data_ptr(), n, qs[t % 8].data_ptr(), mode, 0, key.data_ptr(), None,
                                        nat.stream_ptr()))
        k = max(5, min(steps, 20))
        timed(torch, None, 1, sweep, 3)
        ms = timed(torch, None, 1, sweep, k) / k
        timed(torch, None, 1, sweep_bytes, 2)
        ms_b = timed(torch, None, 1, sweep_bytes, 5) / 5
        gbs = n * 1024 / (ms * 1e-3) / 1e9
        out["vt_u8_" + name] = {"metric": "VT shift-compares/s", "value": n * offs / (ms * 1e-3), "templates_per_s": n / (ms * 1e-3),
                                "ms_per_query": ms, "library": "2^20 x 32x32 uint8, bit-sliced (1088 B/template, 1.06 GiB, > L2)",
                                "bytewise_kernel_ms_per_query": ms_b,
                                "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s",
                                             "frac": gbs / peak, "algorithmic_bytes_per_template": 1024}}
    del packed
    del lib
    # float32 profiles, 2^18 templates (1 GiB)
    nf = 1 << 18
    libf = torch.rand((nf, 32, 32), dtype=torch.float32, device="cuda", generator=g) * 255
    qf = torch.rand((32, 32), dtype=torch.float32, device="cuda", generator=g) * 255

    def sweepf(t):
        nat.check(nat.lib().prs_vt_sweep_f32(libf.data_ptr(), nf, qf.data_ptr(), 0, 0, key.data_ptr(), None, nat.stream_ptr()))
    timed(torch, None, 1, sweepf, 3)
    ms = timed(torch, None, 1, sweepf, 10) / 10
    gbs = nf * 4096 / (ms * 1e-3) / 1e9
    out["vt_f32_ref"] = {"metric": "VT shift-compares/s", "value": nf * 15 / (ms * 1e-3), "ms_per_query": ms,
                         "library": "2^18 x 32x32 float32 (1 GiB)",
                         "note": "read-only stream: can exceed the peak, which is a measured COPY (read + write) bandwidth",
                         "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak}}
    del libf
    # ---- BASELINE config 3: one 256x256x72 network
    shape = (256, 256, 72)
    net = PoseCellNetwork(shape)
    net.inject(1.0, (128, 128, 36))
    rng = np.random.default_rng(2)
    od = torch.from_numpy(np.stack([rng.uniform(0, 0.3, 64), rng.uniform(-0.05, 0.05, 64)], axis=1)).cuda()
    stepf = lambda t: net._ens.update_async(od[t % 64:t % 64 + 1])  # noqa: E731
    timed(torch, None, 1, stepf, 10)
    k = max(10, min(steps, 50))
    ms = timed(torch, None, 1, stepf, k) / k
    cells = shape[0] * shape[1] * shape[2]
    gbs = 8 * cells / (ms * 1e-3) / 1e9
    tf = cells * 98 / (ms * 1e-3) / 1e12
    out["large_grid_256x256x72"] = {"metric": METRIC, "value": cells / (ms * 1e-3), "ms_per_step": ms, "path": net.path,
                                    "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s",
                                                 "frac": gbs / peak, "algorithmic_bytes_per_cell_update": 8,
                                                 "fp32_issue": {"achieved_tfma_per_s": tf, "peak_tfma_per_s": 148 * 128 * 1.965e-3,
                                                                "frac": tf / (148 * 128 * 1.965e-3)}},
                                    "note": "the 18.9 MB state and its intermediates are L2-resident between the kernels "
                                            "of an update; L2 traffic per update is in profiles/"}
    del net
    # ---- the reference's own precision (float64, posecell_network.py:27,41) and simulate.py's grid (50x50x10) as
    #      ensembles larger than L2
    from pyratslam_b200 import PoseCellEnsemble
    for name, shp, B, dt, nbytes in (("ensemble_f64_21x21x36", SHAPE, 2048, np.float64, 8),
                                     ("ensemble_f32_50x50x10", (50, 50, 10), 2600, np.float32, 4)):
        cells = shp[0] * shp[1] * shp[2]
        gis = np.linspace(0.05, 0.25, B)
        e = PoseCellEnsemble(shp, B, global_inhibition=gis, dtype=dt)
        e.inject(1.0, tuple(v // 2 for v in shp))
        rng = np.random.default_rng(5)
        od = torch.from_numpy(np.stack([rng.uniform(0, 0.3, (16, B)), rng.uniform(-0.1, 0.1, (16, B))], axis=-1)).cuda()
        fn = lambda t: e.update_async(od[t % 16])  # noqa: E731
        timed(torch, None, 1, fn, 3)
        k = max(5, min(steps, 20))
        ms = timed(torch, None, 1, fn, k) / k
        gbs = 2 * nbytes * B * cells / (ms * 1e-3) / 1e9
        fma_peak = 148 * (128 if nbytes == 4 else 64) * 1.965e9 / 1e12
        tf = B * cells * 98 / (ms * 1e-3) / 1e12
        out[name] = {"metric": METRIC, "value": B * cells / (ms * 1e-3), "ms_per_step": ms, "networks": B, "path": e.path,
                     "state_mb": B * cells * nbytes / 1e6,
                     "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                                  "algorithmic_bytes_per_cell_update": 2 * nbytes,
                                  "fma_pipe": {"achieved_tfma_per_s": tf, "peak_tfma_per_s": fma_peak,
                                               "frac": tf / fma_peak,
                                               "pipe": "FP32 (128 FMA/clk/SM)" if nbytes == 4 else "FP64 (64 DFMA/clk/SM, measured)"}}}
        del e, od
    # ---- the sparsity-aware update (csrc/posecell_active.cu, opt-in).  SURVEY.md 8(d): the headline must not exploit
    #      the sparsity of the attractor state; a variant that does is reported separately -- here.  Same ensembles, same
    #      odometry as the dense rows above; the dense result of the same steps is the check.
    act_all = {}
    for name, shp, B, dt in (("4096x21x21x36_f32", SHAPE, B_TOTAL, np.float32), ("4096x21x21x36_f64", SHAPE, B_TOTAL, np.float64),
                             ("2600x50x50x10_f32", (50, 50, 10), 2600, np.float32), ("1x256x256x72_f32", (256, 256, 72), 1, np.float32)):
        cells = shp[0] * shp[1] * shp[2]
        nbytes = np.dtype(dt).itemsize
        gis, odom = ensemble_inputs(B, 64, 3)
        od = torch.from_numpy(odom).cuda()
        act, ref_state, ref_amax, nnz, dense_ms, dense_path = {}, None, None, 0, 0.0, ""
        for mode in (0, 1, 2):
            e = PoseCellEnsemble(shp, B, global_inhibition=gis, dtype=dt, active_set=mode)
            e.inject(1.0, tuple(v // 2 for v in shp))
            fn = lambda t: e.update_async(od[t % 64])  # noqa: E731
            timed(torch, None, 1, fn, 8)
            k = max(5, min(steps, 20))
            ms = timed(torch, None, 1, fn, k) / k
            st, am = e.state.clone(), e._argmax.clone()
            if mode == 0:
                ref_state, ref_amax, nnz, dense_ms, dense_path = st, am, int((st != 0).sum().item()), ms, e.path
                del e
                continue
            same = bool(torch.equal(am, ref_amax))
            rel = float((st - ref_state).abs().max().item() / ref_state.abs().max().item())
            # what this variant moves: mode 1 reads every cell once (the scan) and writes only the cells that change
            moved = (nbytes * B * cells if mode == 1 else 0) + 2 * nbytes * nnz
            act["scan_every_update" if mode == 1 else "list_carried_over"] = {
                "metric": METRIC, "value": B * cells / (ms * 1e-3), "ms_per_step": ms, "speedup_over_dense": dense_ms / ms,
                "argmax_identical_to_dense": same, "state_rel_diff_to_dense": rel,
                "bytes_moved_per_update": moved, "hbm_frac_of_bytes_moved": moved / (ms * 1e-3) / 1e9 / peak}
            assert same and rel <= (1e-4 if nbytes == 4 else 1e-11), (name, mode, same, rel)
            del e
        act_all[name] = dict(act, networks=B, non_zero_cells_per_network=nnz / B, dense_ms_per_step=dense_ms,
                             dense_path=dense_path)
        del od, ref_state, ref_amax
    out["active_set"] = dict(act_all, note="reported separately from the headline (SURVEY 8d): an update costs what the "
                                           "activity packet costs, not what the grid costs; exact for any state (networks "
                                           "the kernel flags are updated by the dense kernels in the same call, behind a "
                                           "conditional graph node)")
    # ---- BASELINE config 1: simulate.py's own scenario (50x50x10, 40 steps), every step through update()
    from pyratslam_b200 import simulate
    from oracle import drivers as odrv
    simulate.main(steps=40, verbose=False)
    t0 = time.perf_counter()
    for _ in range(5):
        trace = simulate.main(steps=40, verbose=False)
    dt_sim = (time.perf_counter() - t0) / 5
    t0 = time.perf_counter()
    ref_amax, _, _ = odrv.simulate_run()
    dt_cpu = time.perf_counter() - t0
    assert [tuple(t) for t in trace] == [tuple(t) for t in ref_amax.tolist()]
    out["simulate_50x50x10"] = {"metric": "pose-cell cell-updates/s", "value": 40 * 25000 / dt_sim,
                                "ms_per_step": dt_sim / 40 * 1e3, "cpu_oracle_ms_per_step": dt_cpu / 40 * 1e3,
                                "note": "simulate.py:36-58 loop incl. construction and one host sync per update(); "
                                        "arg-max trace identical to the oracle's"}
    # ---- BASELINE config 2: frame-by-frame replay (odometry update + template match per frame)
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    from synth import synth_frames
    T = 1000
    frames = synth_frames(np.random.default_rng(1), T)
    rng = np.random.default_rng(1)
    odom = np.stack([rng.uniform(0, 3, T), rng.uniform(-1, 1, T)], axis=1)
    ros_simulate.replay(frames[:20], odom[:20])
    t0 = time.perf_counter()
    rec = ros_simulate.replay(frames, odom)
    dt = time.perf_counter() - t0
    ros_simulate.replay(frames[:20], odom[:20], fused=True)
    t0 = time.perf_counter()
    rec_f = ros_simulate.replay(frames, odom, fused=True)
    dt_f = time.perf_counter() - t0
    assert np.array_equal(rec["template"], rec_f["template"]) and np.array_equal(rec["argmax"], rec_f["argmax"])
    ros_simulate.replay(frames[:20], odom[:20], fused=True, pipelined=True)
    t0 = time.perf_counter()
    rec_p = ros_simulate.replay(frames, odom, fused=True, pipelined=True)
    dt_p = time.perf_counter() - t0
    assert np.array_equal(rec["template"], rec_p["template"]) and np.array_equal(rec["argmax"], rec_p["argmax"])
    ros_simulate.replay(frames[:20], odom[:20], native=True)
    t0 = time.perf_counter()
    rec_n = ros_simulate.replay(frames, odom, native=True)
    dt_n = time.perf_counter() - t0
    assert np.array_equal(rec["template"], rec_n["template"]) and np.array_equal(rec["argmax"], rec_n["argmax"])
    assert np.array_equal(rec["created"], rec_n["created"]) and np.array_equal(rec["n_exp"], rec_n["n_exp"])
    assert np.array_equal(rec["em_xy"], rec_n["em_xy"])
    out["replay_21x21x36"] = {"metric": "end-to-end frames/s", "value": T / dt_n, "frames": T,
                              "templates_created": int(rec["n_templates"]),
                              "reference_shaped_calls_frames_per_s": T / dt,
                              "fused_frames_per_s": T / dt_f,
                              "pipelined_frames_per_s": T / dt_p,
                              "note": "host frames: 64 KiB H2D + pose-cell update + template match + 32 B D2H per frame, "
                                      "wall clock, node construction included; value = the loop on the C side of the ABI "
                                      "(prs_replay_run: two frame plans in flight, host bookkeeping replayed from the "
                                      "records); pipelined = two alternating frame plans driven from Python; "
                                      "fused = one CUDA-graph "
                                      "launch and one synchronisation per frame; reference_shaped = separate "
                                      "PoseCellNetwork.update / ViewTemplates.match calls; identical records"}
    return out


def extra_sharded_library(torch, dist, world, rank, peak, steps, n_total, label):
    """BASELINE config 5 across ranks: ``n_total`` uint8 templates split into contiguous global index ranges, one
    device-side MIN exchange of the packed key per query (csrc/sharded.cu over CUDA-IPC peer memory; the NCCL
    all-reduce path is timed next to it).  Planted templates make the answers known without a 10^6-template oracle
    sweep: a planted match in the first shard, and a pattern stored twice -- in the first and in the last shard --
    whose query must resolve to the LOWER index (numpy.argmin)."""
    from oracle import view_templates as ovt                      # checker only
    from pyratslam_b200 import ShardedViewTemplates, _native as nat
    from pyratslam_b200.sharding import shard_range
    lo, hi = shard_range(n_total, rank, world)
    n = hi - lo
    g = torch.Generator(device="cuda").manual_seed(40 + rank)
    lib = torch.randint(0, 256, (n, 32, 32), dtype=torch.uint8, device="cuda", generator=g)
    rp = np.random.default_rng(1234)
    P0, P1 = (rp.integers(0, 256, (32, 32), dtype=np.uint8) for _ in range(2))
    j0, jdup, j1 = 12345, 4242, n_total - 777
    for j, P in ((j0, P0), (jdup, P1), (j1, P1)):
        if lo <= j < hi:
            lib[j - lo] = torch.from_numpy(P).cuda()
    dark = lambda P: np.clip(P.astype(np.int16) - rp.integers(0, 4, P.shape), 0, 255).astype(np.uint8)  # noqa: E731
    q_np = [dark(P0), np.roll(dark(P1), 3, axis=0)] + [rp.integers(0, 256, (32, 32), dtype=np.uint8) for _ in range(6)]
    qs = torch.from_numpy(np.stack(q_np)).cuda()
    svt = ShardedViewTemplates(lib, lo, match_threshold=45000, mode="ref")
    del lib
    out = {"templates_total": n_total, "templates_per_gpu": n, "exchange": svt.exchange,
           "library": "%d x 32x32 uint8 in total, bit-sliced, %.0f MB per GPU (> L2)" % (n_total, n * 1088 / 1e6)}
    for mode, offs in (("ref", 15), ("circular", 32)):
        svt.mode = {"ref": nat.VT_MODE_REF, "circular": nat.VT_MODE_CIRCULAR}[mode]
        # parity inside the run: planted answers against the oracle's score of the planted template alone
        want0 = int(ovt.library_scores(P0[None], q_np[0], mode=mode)[0])
        want1 = int(ovt.library_scores(P1[None], q_np[1], mode=mode)[0])
        assert svt.match_key(qs[0]) == (want0, j0), (mode, svt.match_key(qs[0]), want0, j0)
        assert svt.match_key(qs[1]) == (want1, jdup), (mode, svt.match_key(qs[1]), want1, jdup)
        keys = svt.match_keys(qs)
        assert keys[:2] == [(want0, j0), (want1, jdup)] and keys == [svt.match_key(q) for q in qs]
        k = max(5, min(steps, 20))
        fn = lambda t: svt.match_key(qs[t % 8])  # noqa: E731
        timed(torch, dist, world, fn, 3)
        ms = timed(torch, dist, world, fn, k) / k
        fnb = lambda t: svt.match_keys(qs)  # noqa: E731
        timed(torch, dist, world, fnb, 2)
        kb = max(2, k // 4)
        ms_b = timed(torch, dist, world, fnb, kb) / (kb * len(qs))
        fns = lambda t: svt.local_sweep(qs[t % 8])  # noqa: E731      the shard's sweep alone, no exchange, no read-back
        timed(torch, dist, world, fns, 3)
        ms_s = timed(torch, dist, world, fns, k) / k
        def fnl(t):  # what a blocking query costs with NO exchange: the shard's sweep, then the host waits for it
            svt.local_sweep(qs[t % 8])
            torch.cuda.current_stream().synchronize()
        timed(torch, dist, world, fnl, 3)
        ms_l = timed(torch, dist, world, fnl, k) / k
        rec = {"metric": "VT shift-compares/s", "value": n_total * offs / (ms * 1e-3), "ms_per_query": ms,
               "local_sweep_only_ms": ms_s, "exchange_and_readback_ms": ms - ms_s,
               "blocking_local_query_ms": ms_l, "exchange_over_blocking_local_query_ms": ms - ms_l,
               "batched_8_queries": {"value": n_total * offs / (ms_b * 1e-3), "ms_per_query": ms_b},
               "roofline": {"bound": "hbm", "achieved": n * 1024 / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                            "frac": n * 1024 / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_template": 1024},
               "note": "value: ONE query per call (match_key): local sweep + device-side MIN over the ranks + 8-byte "
                       "result in pinned host memory + stream sync, every query; batched: 8 sweeps, one exchange; "
                       "local_sweep_only: back-to-back sweeps, no host wait (device time per sweep); blocking_local_query: "
                       "the same sweep with the host waiting for it and NO exchange -- what the sharding adds to a blocking "
                       "query is exchange_over_blocking_local_query_ms"}
        if world > 1 and svt.exchange == "fused":
            svt.set_exchange("nccl")
            assert svt.match_key(qs[0]) == (want0, j0)
            timed(torch, dist, world, fn, 3)
            rec["nccl_allreduce_ms_per_query"] = timed(torch, dist, world, fn, k) / k
            svt.set_exchange("fused")
        out["vt_u8_" + mode] = rec
    # create-or-match through the exchange: the random queries are novel, the planted ones match
    svt.mode = nat.VT_MODE_REF
    assert svt.match(qs[0]) == (j0, False) and svt.match(qs[1]) == (jdup, False)
    assert svt.match(qs[2]) == (n_total, True) and svt.match(qs[2]) == (n_total, False)
    out["parity"] = "planted match, cross-shard tie -> lowest index, novel -> created: checked against the oracle (%s)" % label
    svt.close()
    return out


def check_sampled_networks(ens, odom_dev, gis, rank):
    """Two networks of this rank's shard, three updates, against the oracle (arg-max bit-exact, state <= 1e-5)."""
    from oracle import posecells as opc                           # checker only
    import torch
    B = ens.n_networks
    pick = sorted({0, B - 1})
    before = ens.state[pick].clone()
    od = odom_dev[:3].cpu().numpy()
    got = []
    for t in range(3):
        ens.update_async(odom_dev[t])
        got.append(ens._unravel(ens._argmax[pick].cpu().numpy()))
    after = ens.state[pick].permute(0, 2, 3, 1).cpu().numpy().astype(np.float64)   # [th][x][y] -> [x][y][th]
    for i, b in enumerate(pick):
        ref = opc.PoseCellNetwork(SHAPE, global_inhibition=float(gis[b]))
        ref.posecells = before[i].permute(1, 2, 0).cpu().numpy().astype(np.float64)
        for t in range(3):
            assert tuple(ref.update(od[t, b])) == tuple(got[t][i]), (rank, b, t)
        err = np.abs(after[i] - ref.posecells).max() / max(ref.posecells.max(), 1e-30)
        assert err <= 1e-5, (rank, b, err)
    torch.cuda.synchronize()
    return len(pick)


def last_step_outputs(ens, n_sample=512):
    """What a caller of the timed update_async holds after the last timed step, as host arrays in float32 / float64:
    the arg-max cell (x, y, th), the total activity and the error flags of every network, and the whole state of a
    fixed, seeded sample of ``n_sample`` networks (``networks``) in the reference's [x][y][th] layout (32.5 MB of the 260 MB ensemble)."""
    import torch
    pick = np.sort(np.random.default_rng(0).choice(ens.n_networks, min(n_sample, ens.n_networks), replace=False))
    states = ens.state.index_select(0, torch.from_numpy(pick).to(ens.state.device)).permute(0, 2, 3, 1)
    return {"argmax": ens._unravel(ens._argmax.cpu().numpy()).astype(np.float64),
            "total": ens._total.cpu().numpy(), "err": ens._err.cpu().numpy().astype(np.float32),
            "networks": pick.astype(np.float64), "posecells": states.cpu().numpy()}


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import __graft_entry__ as ge
    ge.build()
    from pyratslam_b200 import PoseCellEnsemble
    from pyratslam_b200.sharding import shard_range
    peak, peak_src = measured_peaks()
    d = dist if world > 1 else None

    # ---- parity on the ranks of this job, before anything is timed
    parity = None
    if not args.no_parity:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import multigpu_check
        exch = multigpu_check.run_checks(rank, world)
        parity = {"parity_nranks": world, "exchange": exch,
                  "what": "tests/multigpu_check.run_checks: sharded 5003-template library (ref + circular + float32; ties, "
                          "appends) == numpy argmin of the oracle; sharded 64-network ensemble == oracle arg-max"}

    # ---- BASELINE config 4, strong scaling: 4096 networks in total, contiguous shards
    lo, hi = shard_range(B_TOTAL, rank, world)
    B = hi - lo
    R = world                                            # replicas of the shard: 260 MB of state per GPU at every N
    K, W = args.steps, max(args.warmup, 3)
    gis_all, odom_all = ensemble_inputs(B_TOTAL, 64, 3)
    gis, odom = gis_all[lo:hi], np.ascontiguousarray(odom_all[:, lo:hi])
    ens = [PoseCellEnsemble(SHAPE, B, global_inhibition=gis) for _ in range(R)]
    for e in ens:
        e.inject(1.0, tuple(s // 2 for s in SHAPE))
    od_dev = torch.from_numpy(odom).cuda()
    path = ens[0].path
    launches_per_step = 1 if path in ("resident", "pair") else 8
    if parity is not None:
        parity["sampled_networks_per_rank"] = check_sampled_networks(ens[0], od_dev, gis, rank)
    step_dev = lambda t: ens[t % R].update_async(od_dev[t % 64])  # noqa: E731
    step_hot = lambda t: ens[0].update_async(od_dev[t % 64])  # noqa: E731
    step_block = lambda t: ens[t % R].update(odom[t % 64])  # noqa: E731

    def step_host(t):
        # the public overlapped stepping API: every step copies its odometry in from pinned memory and its packed
        # result out, one step is kept in flight so that the copies hide behind the previous step's kernel
        ens[t % R].update_submit(odom[t % 64])
        if t > 0:
            ens[(t - 1) % R].update_result()
        if t == last_step[0]:  # the last step's result is read inside the timed region as well
            ens[t % R].update_result()

    def drain():
        for e in ens:
            while getattr(e, "_pipe_head", 0) > getattr(e, "_pipe_tail", 0):
                e.update_result()

    timed(torch, d, world, step_dev, W)
    # The timed steps start from the state these W steps leave, whatever number of batches the clock warm-up below
    # takes: with the same arguments they compute the same results from run to run
    start = [e.state.clone() for e in ens]
    # The GPU idled while the host ran the oracle checks: keep warming up (untimed) until two consecutive batches of K
    # steps agree within 1 % -- SM clocks at their boost level -- at most ten batches
    prev = None
    for _ in range(10):
        cur = timed(torch, d, world, step_dev, K)
        W += K
        if prev is not None and abs(cur - prev) <= 0.01 * prev:
            break
        prev = cur
    for e, s in zip(ens, start):
        e.state.copy_(s)
    del start
    with ClockSampler(local) as clk:
        ms = timed(torch, d, world, step_dev, K)
        last = last_step_outputs(ens[(K - 1) % R]) if args.dump_outputs else None
        # keep the sampler alive for at least a few samples on very short runs
        if ms < 400:
            timed(torch, d, world, step_dev, max(K, int(400 / max(ms / K, 1e-3))))
    clocks = clk.summary()
    value = B_TOTAL * N_CELLS * K / (ms * 1e-3)
    # end to end through the public API with host odometry
    last_step = [W - 1]
    timed(torch, d, world, step_host, W)
    drain()
    last_step[0] = K - 1
    ms_e2e = timed(torch, d, world, step_host, K)
    drain()
    e2e = B_TOTAL * N_CELLS * K / (ms_e2e * 1e-3)
    timed(torch, d, world, step_block, W)
    ms_blk = timed(torch, d, world, step_block, K)
    e2e_blk = B_TOTAL * N_CELLS * K / (ms_blk * 1e-3)
    alive = int(sum(int((e.state.amax(dim=(1, 2, 3)) > 0).sum().item()) for e in ens)) // R
    ms_hot = None
    weak = None
    if world > 1:
        timed(torch, d, world, step_hot, W)
        ms_hot = timed(torch, d, world, step_hot, K) / K
        del ens[1:]
        # weak-scaling variant of the same config (4096 networks PER GPU), reported as an extra
        gw, ow = ensemble_inputs(B_TOTAL, 64, 3 + rank)
        ew = PoseCellEnsemble(SHAPE, B_TOTAL, global_inhibition=gw)
        ew.inject(1.0, tuple(s // 2 for s in SHAPE))
        odw = torch.from_numpy(ow).cuda()
        stepw = lambda t: ew.update_async(odw[t % 64])  # noqa: E731
        timed(torch, d, world, stepw, W)
        msw = timed(torch, d, world, stepw, K) / K
        weak = {"value": world * B_TOTAL * N_CELLS / (msw * 1e-3), "ms_per_step": msw, "networks_per_gpu": B_TOTAL,
                "scaling": "weak"}
        del ew, odw

    line = None
    if rank == 0:
        alg_bytes = 2 * 4 * B * N_CELLS                  # read + write the float32 state once per update
        gbs = alg_bytes / (ms / K * 1e-3) / 1e9
        fma_per_cell = 98
        sm_mhz = clocks.get("sm_mhz") or 1965.0
        fp32_peak = 148 * 128 * sm_mhz * 1e6 / 1e12        # TFMA/s at the clock seen during the timed region
        tfma = B * N_CELLS * fma_per_cell / (ms / K * 1e-3) / 1e12
        traffic, traffic_src = profiled_traffic() if world == 1 else (None, "N > 1: shard sizes differ from the capture")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "ensemble of 4096 independent 21x21x36 pose-cell networks in total, sharded by "
                                   "network over the GPUs (BASELINE config 4)",
                       "shape": list(SHAPE), "networks_total": B_TOTAL, "networks_per_gpu": B, "path": path,
                       "l2": "every rank steps %d replica(s) of its shard in turn: %.0f MB of distinct state per GPU, more "
                             "than L2 (126 MB), so every timed step streams from HBM" % (R, R * B * N_CELLS * 4 / 1e6),
                       "parallelism": "networks sharded by rank, no collective",
                       "launches": "one kernel per step; consecutive steps of an ensemble overlap on the device per network "
                                   "(programmatic dependent launch + one sequence number per network, "
                                   "csrc/posecell_resident.cu; PRS_RESIDENT_PDL=0 serialises them: 0.3485 ms per step "
                                   "at N = 1, 0.0572 ms for 512 networks)"},
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / K, "h2d_bytes_per_step": B * 16,
                    "d2h_bytes_per_step": B * 16,
                    "api": "PoseCellEnsemble.update_submit / update_result (prs_pc_step_host_xyz_async): host odometry in "
                           "pinned memory -> step -> packed (x, y, th, err) per network in pinned host memory, every step, "
                           "one step in flight.  On the fused path the transfers are the kernel's own: it reads the "
                           "16 B of odometry per network from the pinned buffer over PCIe and writes the 16 B record "
                           "back (h2d / d2h_bytes_per_step), completion is a pinned word the host polls -- no copy "
                           "engine, no event between two updates, so that consecutive updates overlap "
                           "(PRS_HOST_ZERO_COPY=0 restores cudaMemcpyAsync on two copy streams).  The blocking call "
                           "(PoseCellEnsemble.update, host waits for every step) is blocking_call",
                    "blocking_call": {"value": e2e_blk, "ms_per_step": ms_blk / K,
                                      "api": "PoseCellEnsemble.update (prs_pc_step_host_xyz): same transfers, host waits "
                                             "for every step"}},
            "gpu_launches": K * launches_per_step,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                         "traffic": traffic, "peak_source": peak_src, "traffic_source": traffic_src,
                         "kernel": "k_pc_resident / k_pc_pair (one launch per step)" if launches_per_step == 1
                                   else "generic 8-kernel step (whole step timed)",
                         "algorithmic_bytes_per_cell_update": 8,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "binding_roof": "fp32 issue: 98 FMA per 8 B puts the FP32 pipe roof at 0.46 of the HBM roof",
                         "fp32_issue": {"fma_per_cell_update": fma_per_cell, "achieved_tfma_per_s": tfma,
                                        "peak_tfma_per_s": fp32_peak, "frac": tfma / fp32_peak}},
            "networks_alive": alive,
        }
        if parity is not None:
            line.update(parity)
        if ms_hot is not None:
            line["l2_resident_shard"] = {"ms_per_step": ms_hot, "value": B_TOTAL * N_CELLS / (ms_hot * 1e-3),
                                         "note": "the same step on ONE replica: the shard (%.0f MB) stays in L2 between "
                                                 "steps, which is what a user stepping this ensemble gets" % (B * N_CELLS * 4 / 1e6)}
        if weak is not None:
            line["extra_weak_ensemble"] = weak
        line["extra_sharded"] = None
        if world == 1:
            line["cpu_baseline"] = cpu_baseline()
            if not args.no_extra:
                line["extra"] = extra_single_gpu(torch, peak, K)
    del ens
    if not args.no_extra:
        shard = {"strong_2^20_total": extra_sharded_library(torch, d, world, rank, peak, K, 1 << 20,
                                                            "%d rank(s)" % world)}
        if world > 1:
            shard["weak_2^20_per_gpu"] = extra_sharded_library(torch, d, world, rank, peak, K, world << 20,
                                                                "%d rank(s), weak" % world)
        if rank == 0:
            line["extra_sharded"] = shard
    if rank == 0:
        emit(line)
    if last is not None:
        for name, a in last.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world > 1:
        dist.destroy_process_group()


_RESULT_OUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to fd 1
    when NCCL_DEBUG is set in the environment), so fd 1 is pointed at stderr for the rest of the run and the
    result line goes to a private duplicate of the original stdout."""
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr


def emit(line):
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads (profiling runs)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle checks (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the headline ensemble as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs:
        if args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1:
            ap.error("--dump-outputs writes the outputs of one GPU: use it with --impl ours --gpus 1")
        os.makedirs(args.dump_outputs, exist_ok=True)
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
