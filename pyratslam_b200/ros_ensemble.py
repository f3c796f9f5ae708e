"""One recording through B differently parameterised RatSLAM agents in one pass on the GPU.

Tuning RatSLAM offline means replaying one recording under many settings -- the match threshold, the global inhibition,
the view-template -> pose-cell injection energy -- and comparing the runs.  ``replay_ensemble`` runs all of them at
once: agent ``b`` is the ROS loop of ``ros_simulate.replay(native=True, match_threshold=..., inject_energy=...)`` with
``pcn.global_inhibition`` set to its own value, and it has its own pose-cell network, view-template library and
experience map.  The frames and the odometry are shared, so a frame is one CUDA graph for the whole ensemble
(``prs_ens_replay_run``, csrc/view_templates.cu): one pose-cell update of all B networks, one query, one sweep over
every agent's library, then the per-agent create-or-match decision and injection.

Tuning on several recordings keeps the settings from fitting one route: with ``frames`` and ``odom`` given as lists of
R recordings, agent ``b`` replays recording ``recording[b]`` (``prs_ens_multi_replay_run``), still in one graph per
frame.

    python -m pyratslam_b200.ros_ensemble BAG [BAG ...] --match-threshold 30000,45000,60000 --global-inhibition 0.1,0.2
"""
from __future__ import annotations

import ctypes
import itertools
import math
import numbers

import numpy as np
import torch

from . import _native as nat
from . import experience_ensemble as xens
from .experience_map import ExperienceMap
from .kernels import PC_GLOBAL_INHIB
from .posecell_network import PoseCellEnsemble, _as_np_dtype
from .ros_simulate import IM_SIZE, MATCH_THRESHOLD, POSE_SIZE, X_RANGE, X_STEP, Y_RANGE, Y_STEP, RatslamRos

MAX_CAPACITY = 1 << 16          # templates per agent the frame's library sweep takes (kSmallLibrary)


def _real(v):
    return isinstance(v, (numbers.Real, np.number)) and not isinstance(v, (bool, np.bool_))


def agent_parameters(n_agents=None, match_threshold=MATCH_THRESHOLD, global_inhibition=PC_GLOBAL_INHIB,
                     inject_energy=None):
    """Broadcast the per-agent parameters to B agents and validate them (no CUDA involved).

    Each parameter is a scalar or a length-B sequence; B is ``n_agents`` or the length of the sequences.  Returns
    ``(B, thresholds uint32[B], gi float64[B], energies list of float-or-None)``; the thresholds are clamped the way the
    single-agent frame plans clamp them.  ``ValueError`` for disagreeing lengths, non-finite thresholds or inhibitions,
    and energies that are negative or not finite."""
    params = {"match_threshold": match_threshold, "global_inhibition": global_inhibition, "inject_energy": inject_energy}
    seqs = {}
    for k, v in params.items():
        if v is None or _real(v):
            continue
        try:
            seqs[k] = list(v)
        except TypeError:
            raise ValueError("%s must be a scalar or a sequence, got %r" % (k, v)) from None
    B = None if n_agents is None else int(n_agents)
    if B is not None and B < 1:
        raise ValueError("n_agents must be >= 1, got %r" % (n_agents,))
    for k, v in seqs.items():
        if B is None:
            B = len(v)
        if len(v) != B or B == 0:
            raise ValueError("%s has %d values for %d agents" % (k, len(v), B))
    B = 1 if B is None else B
    out = {k: seqs[k] if k in seqs else [v] * B for k, v in params.items()}
    thr = []
    for v in out["match_threshold"]:
        if not _real(v) or not math.isfinite(float(v)):
            raise ValueError("match_threshold must be finite numbers, got %r" % (v,))
        thr.append(int(min(max(math.floor(v), 0), 0xFFFFFFFF)))    # as RatslamRos._fused_plan
    gi = []
    for v in out["global_inhibition"]:
        if not _real(v) or not math.isfinite(float(v)):
            raise ValueError("global_inhibition must be finite numbers, got %r" % (v,))
        gi.append(float(v))
    energies = []
    for v in out["inject_energy"]:
        if v is not None and (not _real(v) or not math.isfinite(float(v)) or float(v) < 0):
            raise ValueError("inject_energy must be None or a finite energy >= 0 (the injection runs on the device), "
                             "got %r" % (v,))
        energies.append(None if v is None else float(v))
    return B, np.array(thr, dtype=np.uint32), np.array(gi, dtype=np.float64), energies


def capacity_for(T):
    """Templates per agent for a T-frame replay: one frame appends at most one template, whole groups of 32."""
    return (int(T) + 1 + 31) // 32 * 32


def agent_recordings(recording, B, n_recordings):
    """int64 [B]: the recording each agent replays, from ``recording`` = one index or a length-B sequence of indices into
    the ``n_recordings`` recordings (no CUDA involved).  ``ValueError`` for a length other than B and for anything that is
    not an integer in [0, n_recordings)."""
    if isinstance(recording, (numbers.Integral, np.integer)) and not isinstance(recording, (bool, np.bool_)):
        rec = [recording] * B
    else:
        try:
            rec = list(recording)
        except TypeError:
            raise ValueError("recording must be an index or a sequence of indices, got %r" % (recording,)) from None
        if len(rec) != B:
            raise ValueError("recording has %d values for %d agents" % (len(rec), B))
    for r in rec:
        if (not isinstance(r, (numbers.Integral, np.integer)) or isinstance(r, (bool, np.bool_))
                or not 0 <= int(r) < n_recordings):
            raise ValueError("recording must be indices in [0, %d), got %r" % (n_recordings, r))
    return np.array(rec, dtype=np.int64)


def _recording_count(recording):
    """The agent count a sequence ``recording`` implies, None for a scalar."""
    if recording is None or isinstance(recording, (numbers.Number, np.number, str, bytes)):
        return None
    try:
        return len(recording)
    except TypeError:
        return None


def _multi_chunk(R, frame_bytes):
    """Frames per recording in one device chunk (prs_ens_multi_scratch_bytes): 256 MiB over R recordings, in [1, 256]."""
    return int(min(max((256 << 20) // (R * frame_bytes), 1), 256))


def _unravel(flat, shape):
    X, Y, Th = shape
    flat = np.asarray(flat, dtype=np.int64)
    return np.stack([flat // (Y * Th), (flat // Th) % Y, flat % Th], axis=-1)


class EnsembleAgents:
    """What every agent holds after the replay: its library, the template locations and its pose cells."""

    def __init__(self, ens, libs, loc, n_templates, shape):
        self._ens, self._libs, self._loc = ens, libs, loc
        self.n_templates = n_templates
        self.shape = shape

    def __len__(self):
        return len(self.n_templates)

    @property
    def path(self):
        """The pose-cell kernel family that updated the ensemble (``PoseCellEnsemble.path``)."""
        return self._ens.path

    @property
    def state(self):
        """The device tensor ``[B, Th, X, Y]`` of every agent's pose cells (theta-major)."""
        return self._ens.state

    def templates(self, b):
        """uint8 ``[n_b, 32, 32]``: agent b's templates as ``ViewTemplate.template`` holds them."""
        n = int(self.n_templates[b])
        out = torch.empty((n, 32, 32), dtype=torch.uint8, device=self._libs.device)
        with torch.cuda.device(self._libs.device):
            for i in range(n):
                nat.check(nat.lib().prs_vt_unpack_u8(self._libs[b].data_ptr(), i, out[i].data_ptr(), nat.stream_ptr()),
                          "prs_vt_unpack_u8")
            return out.cpu().numpy()

    def locations(self, b):
        """int64 ``[n_b, 3]``: the pose cell each of agent b's templates was created at (``ViewTemplate.location``)."""
        return _unravel(self._loc[b, :int(self.n_templates[b])].cpu().numpy(), self.shape)

    def posecells(self, b):
        """Agent b's pose cells, float64 ``[X, Y, Th]`` (the reference's layout)."""
        return self._ens.state[b].permute(1, 2, 0).cpu().numpy().astype(np.float64)


def replay_ensemble(frames, odom, n_agents=None, match_threshold=MATCH_THRESHOLD, global_inhibition=PC_GLOBAL_INHIB,
                    inject_energy=None, pose_size=POSE_SIZE, dtype=np.float32, active_set=0, experience_map=False,
                    experience_links=False, mode="ref", recording=0):
    """Replay ``frames[T,256,256]`` (uint8) and ``odom[T,2]`` = (linear.x, angular.z) through B agents.

    ``match_threshold``, ``global_inhibition`` and ``inject_energy`` (None = no injection, else a finite energy >= 0)
    are scalars or length-B sequences.  Every agent starts as ``RatslamRos`` does: energy 1 at the grid's midpoint,
    an empty library.  Returns a dict with ``template [B,T]``, ``created [B,T]``, ``argmax [B,T,3]`` (the cell each
    match was made with), ``n_templates [B]`` and ``agents`` (``EnsembleAgents``); with ``experience_map=True`` also
    ``n_exp [B,T]`` and ``em_xy [B,T,2]``, replayed on the host from the records as ``RatslamRos.replay_native`` does
    (O(B*T) Python, off by default).  A pose-cell error raises what ``replay(native=True)`` raises (``KeyError((5, 5))``
    for the reference's LUT hole, ``ValueError`` for an oversize shift) for the first offending frame, which the shared
    odometry makes the same frame for every agent.

    ``experience_map="device"`` builds the maps with ``experience_ensemble``: with ``experience_links=True`` every
    agent's linked map on the device, next to ``n_exp`` and ``em_xy`` also ``exp_id [B,T]`` (the current experience),
    ``n_loop_closures [B]`` and ``maps`` (``EnsembleExperienceMaps``); without links the shared dead reckoning once
    (``maps`` None).  Any other value than False, True or "device" raises ``ValueError``.

    Several recordings: ``frames`` and ``odom`` are lists of R arrays ``[T_r,256,256]`` uint8 and ``[T_r,2]``, and
    ``recording`` (an index or a length-B sequence, broadcast like the parameters) names the one each agent replays.
    Agent b's outputs equal those of ``replay_ensemble`` on its own recording, or ``replay(native=True)``; the arrays are
    ``[B, T_max]`` with ``length [B]`` (the agent's recording's frame count), and past an agent's length ``template`` and
    ``argmax`` are -1, ``created`` False, ``n_exp`` and ``exp_id`` -1 and ``em_xy`` NaN.  A pose-cell error raises what
    the native replay of that recording raises, for the earliest frame and, within it, the lowest agent.  With single
    arrays ``recording`` can only be 0."""
    if not (isinstance(experience_map, (bool, np.bool_))
            or (isinstance(experience_map, str) and experience_map == "device")):
        raise ValueError("experience_map must be False, True or 'device', got %r" % (experience_map,))
    B, thr, gi, energies = agent_parameters(n_agents if n_agents is not None else _recording_count(recording),
                                            match_threshold, global_inhibition, inject_energy)
    if mode != "ref":
        raise ValueError("replay_ensemble supports the reference matching mode only, got mode=%r" % (mode,))
    if isinstance(frames, (list, tuple)) and (len(frames) == 0 or np.ndim(frames[0]) == 3):
        return _replay_recordings(frames, odom, agent_recordings(recording, B, max(len(frames), 1)), thr, gi, energies,
                                  pose_size, dtype, active_set, experience_map, experience_links)
    agent_recordings(recording, B, 1)
    frames = np.asarray(frames)
    odom = np.asarray(odom, dtype=np.float64)
    T = len(frames)
    if frames.dtype != np.uint8 or frames.ndim != 3 or tuple(frames.shape[1:]) != IM_SIZE or odom.shape != (T, 2):
        raise ValueError("replay_ensemble: frames must be uint8 [T,%d,%d] and odom [T,2], got %s %r and %r"
                         % (IM_SIZE[0], IM_SIZE[1], frames.dtype, frames.shape, odom.shape))
    pose_size = tuple(int(s) for s in pose_size)
    np_dtype = _as_np_dtype(dtype)
    cap = capacity_for(T)
    if cap > MAX_CAPACITY:
        raise ValueError("replay_ensemble: %d frames need %d templates per agent; the library sweep takes at most %d"
                         % (T, cap, MAX_CAPACITY))
    frames = np.ascontiguousarray(frames)
    lib_bytes = (cap // 32) * 34816
    need = B * (lib_bytes + cap * 8 + int(np.prod(pose_size)) * np.dtype(np_dtype).itemsize + 64)
    if experience_map == "device" and experience_links:
        need += xens.work_bytes(B, T, cap) + xens.record_bytes(B, T)
    nat.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    free, _ = torch.cuda.mem_get_info(dev)
    if need > free:
        raise ValueError("replay_ensemble: %d agents x %d templates need %.2f GB of device memory, %.2f GB are free"
                         % (B, cap, need / 1e9, free / 1e9))

    ens = PoseCellEnsemble(pose_size, B, global_inhibition=gi, dtype=np_dtype, device=dev, active_set=active_set)
    midpoint = tuple(math.floor(s / 2) for s in pose_size)
    ens.inject(1, midpoint)                                             # RatslamRos.__init__
    L = nat.lib()
    assert int(L.prs_vt_packed_bytes(cap)) == lib_bytes
    libs = torch.zeros((B, lib_bytes), dtype=torch.uint8, device=dev)
    loc = torch.full((B, cap), -1, dtype=torch.int64, device=dev)
    n_dev = torch.zeros(B, dtype=torch.int32, device=dev)
    thr_dev = torch.from_numpy(thr.view(np.int32)).to(dev)
    injecting = any(e is not None for e in energies)
    energy_dev = torch.tensor([-1.0 if e is None else e for e in energies], dtype=torch.float64, device=dev)
    pc_work = torch.zeros(3 * B, dtype=torch.int64, device=dev)
    scratch = torch.empty(int(L.prs_ens_scratch_bytes(B, IM_SIZE[0], IM_SIZE[1])), dtype=torch.uint8, device=dev)
    res = np.zeros((T, B), dtype=RatslamRos._RESULT_DTYPE)
    stream = torch.cuda.Stream(device=dev)
    plan = ctypes.c_void_p()
    with torch.cuda.device(dev):
        nat.check(L.prs_pc_argmax(ens._h, ens.state.data_ptr(), pc_work.data_ptr(), nat.stream_ptr()), "prs_pc_argmax")
        torch.cuda.current_stream(dev).synchronize()
        nat.check(L.prs_ens_create(
            ens._h, ens.state.data_ptr(), ens._gi.data_ptr(), pc_work.data_ptr(), libs.data_ptr(), cap, n_dev.data_ptr(),
            thr_dev.data_ptr(), energy_dev.data_ptr() if injecting else None, loc.data_ptr(), nat.VT_MODE_REF,
            IM_SIZE[0], IM_SIZE[1], Y_RANGE[0], Y_RANGE[1], Y_STEP, X_RANGE[0], X_RANGE[1], X_STEP, scratch.data_ptr(),
            ctypes.byref(plan)), "prs_ens_create")
        try:
            moved, tw = xens.gate(odom)
            nat.check(L.prs_ens_replay_run(plan, frames.ctypes.data, tw.ctypes.data, moved.ctypes.data, T,
                                           res.ctypes.data, ctypes.c_void_p(stream.cuda_stream)), "prs_ens_replay_run")
        finally:
            L.prs_ens_destroy(plan)
    bad = np.nonzero((((res["pc_err"] & ~nat.ERR_INJECT_LOC) != 0) & (moved[:, None] != 0)).any(axis=1))[0]
    if len(bad):
        stop = int(bad[0])
        ens._raise_on_err(np.asarray(res["pc_err"][stop] & ~nat.ERR_INJECT_LOC, dtype=np.int32))
    n_templates = res["n_templates"][-1].astype(np.int64) if T else np.zeros(B, np.int64)
    out = {"template": res["template_index"].T.astype(np.int64), "created": res["created"].T != 0,
           "argmax": _unravel(res["argmax"].T, pose_size), "n_templates": n_templates,
           "agents": EnsembleAgents(ens, libs, loc, n_templates, pose_size)}
    if experience_map == "device":
        out.update(xens._maps(res["template_index"], np.ascontiguousarray(res["argmax"]), moved, tw, pose_size,
                              experience_links, 1.0, 0.5, dev))
    elif experience_map:
        out["n_exp"], out["em_xy"] = _experience_maps(out, moved, tw, pose_size, experience_links)
    return out


def _experience_maps(out, moved, tw, pose_size, linked, rec_of=None):
    """Each agent's experience map replayed from its records (``RatslamRos.replay_native``'s bookkeeping); with
    ``rec_of``, ``moved [T,R]`` and ``tw [T,R,2]`` hold every recording's odometry and agent b follows ``rec_of[b]``."""
    B, T = out["template"].shape
    n_exp = np.zeros((B, T), np.int64)
    em_xy = np.zeros((B, T, 2))
    for b in range(B):
        em = ExperienceMap(linked=linked, pc_dims=pose_size)
        tpl, amax = out["template"][b], out["argmax"][b]
        mv, tws = (moved, tw) if rec_of is None else (moved[:, rec_of[b]], tw[:, rec_of[b]])
        for t in range(T):
            if mv[t]:
                vt = int(tpl[t - 1]) if t > 0 else None
                em.update(float(tws[t, 0]), float(tws[t, 1]), tuple(int(c) for c in amax[t]), vt if linked else None)
            n_exp[b, t] = len(em.experiences)
            if em.current_exp is not None:
                em_xy[b, t] = em.get_current_point()
    return n_exp, em_xy


def _replay_recordings(frames, odom, rec_of, thr, gi, energies, pose_size, dtype, active_set, experience_map,
                       experience_links):
    """replay_ensemble over R recordings: agent b replays ``frames[rec_of[b]]``, ``odom[rec_of[b]]``."""
    R = len(frames)
    if not isinstance(odom, (list, tuple)) or len(odom) != R or R == 0:
        raise ValueError("replay_ensemble: frames and odom must be lists of the same, non-zero number of recordings, "
                         "got %d and %s" % (R, len(odom) if isinstance(odom, (list, tuple)) else type(odom).__name__))
    fr, od = [], []
    for r in range(R):
        f, o = np.asarray(frames[r]), np.asarray(odom[r], dtype=np.float64)
        if f.dtype != np.uint8 or f.ndim != 3 or tuple(f.shape[1:]) != IM_SIZE or o.shape != (len(f), 2):
            raise ValueError("replay_ensemble: recording %d: frames must be uint8 [T,%d,%d] and odom [T,2], got %s %r "
                             "and %r" % (r, IM_SIZE[0], IM_SIZE[1], f.dtype, f.shape, o.shape))
        fr.append(np.ascontiguousarray(f))
        od.append(o)
    B = len(rec_of)
    lengths = np.array([len(f) for f in fr], dtype=np.int32)
    T = int(lengths.max())
    pose_size = tuple(int(s) for s in pose_size)
    np_dtype = _as_np_dtype(dtype)
    cap = capacity_for(T)
    if cap > MAX_CAPACITY:
        raise ValueError("replay_ensemble: %d frames need %d templates per agent; the library sweep takes at most %d"
                         % (T, cap, MAX_CAPACITY))
    lib_bytes = (cap // 32) * 34816
    net_bytes = int(np.prod(pose_size)) * np.dtype(np_dtype).itemsize
    frame_bytes = IM_SIZE[0] * IM_SIZE[1]
    # per agent: library, locations, network, its snapshot and the records; plus one chunk of every recording's frames
    need = B * (lib_bytes + cap * 8 + 2 * net_bytes + 64) + R * _multi_chunk(R, frame_bytes) * frame_bytes
    if experience_map == "device" and experience_links:
        need += xens.work_bytes(B, T, cap) + xens.record_bytes(B, T)
    nat.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    free, _ = torch.cuda.mem_get_info(dev)
    if need > free:
        raise ValueError("replay_ensemble: %d agents x %d templates need %.2f GB of device memory, %.2f GB are free"
                         % (B, cap, need / 1e9, free / 1e9))

    # the agents of one recording get contiguous indices on the device (the sweep reloads a query per recording change)
    order = np.argsort(rec_of, kind="stable")
    inv = np.argsort(order)
    ens = PoseCellEnsemble(pose_size, B, global_inhibition=gi[order], dtype=np_dtype, device=dev, active_set=active_set)
    ens.inject(1, tuple(math.floor(s / 2) for s in pose_size))         # RatslamRos.__init__
    L = nat.lib()
    assert int(L.prs_vt_packed_bytes(cap)) == lib_bytes
    libs = torch.zeros((B, lib_bytes), dtype=torch.uint8, device=dev)
    loc = torch.full((B, cap), -1, dtype=torch.int64, device=dev)
    n_dev = torch.zeros(B, dtype=torch.int32, device=dev)
    thr_dev = torch.from_numpy(thr[order].view(np.int32)).to(dev)
    injecting = any(e is not None for e in energies)
    energy_dev = torch.tensor([-1.0 if energies[i] is None else energies[i] for i in order], dtype=torch.float64,
                              device=dev)
    rec_dev = torch.from_numpy(rec_of[order].astype(np.int32)).to(dev)
    pc_work = torch.zeros(3 * B, dtype=torch.int64, device=dev)
    scratch = torch.empty(int(L.prs_ens_scratch_bytes(B, IM_SIZE[0], IM_SIZE[1])), dtype=torch.uint8, device=dev)
    moved = np.zeros((T, R), np.uint8)             # past a recording's end: not moved
    tw = np.zeros((T, R, 2))
    for r in range(R):
        moved[:lengths[r], r], tw[:lengths[r], r] = xens.gate(od[r])
    res = np.zeros((T, B), dtype=RatslamRos._RESULT_DTYPE)
    stream = torch.cuda.Stream(device=dev)
    plan = ctypes.c_void_p()
    frame_ptrs = (ctypes.c_void_p * R)(*[f.ctypes.data if len(f) else None for f in fr])
    with torch.cuda.device(dev):
        nat.check(L.prs_pc_argmax(ens._h, ens.state.data_ptr(), pc_work.data_ptr(), nat.stream_ptr()), "prs_pc_argmax")
        torch.cuda.current_stream(dev).synchronize()
        nat.check(L.prs_ens_create(
            ens._h, ens.state.data_ptr(), ens._gi.data_ptr(), pc_work.data_ptr(), libs.data_ptr(), cap, n_dev.data_ptr(),
            thr_dev.data_ptr(), energy_dev.data_ptr() if injecting else None, loc.data_ptr(), nat.VT_MODE_REF,
            IM_SIZE[0], IM_SIZE[1], Y_RANGE[0], Y_RANGE[1], Y_STEP, X_RANGE[0], X_RANGE[1], X_STEP, scratch.data_ptr(),
            ctypes.byref(plan)), "prs_ens_create")
        try:
            mscratch = torch.empty(int(L.prs_ens_multi_scratch_bytes(plan, R)), dtype=torch.uint8, device=dev)
            nat.check(L.prs_ens_set_recordings(plan, R, rec_dev.data_ptr(), mscratch.data_ptr()),
                      "prs_ens_set_recordings")
            nat.check(L.prs_ens_multi_replay_run(plan, frame_ptrs, tw.ctypes.data, moved.ctypes.data, lengths.ctypes.data,
                                                 T, res.ctypes.data, ctypes.c_void_p(stream.cuda_stream)),
                      "prs_ens_multi_replay_run")
        finally:
            L.prs_ens_destroy(plan)
        # back to the caller's agent order
        inv_d = torch.from_numpy(inv).to(dev)
        ens.state.copy_(ens.state[inv_d])
        ens.global_inhibition = gi
        nat.check(L.prs_pc_invalidate_active(ens._h, nat.stream_ptr()), "prs_pc_invalidate_active")
        libs, loc = libs[inv_d], loc[inv_d]
    res = np.ascontiguousarray(res[:, inv])
    agent_moved = moved[:, rec_of]                  # [T, B]
    bad = ((res["pc_err"] & ~nat.ERR_INJECT_LOC) != 0) & (agent_moved != 0)
    if bad.any():
        t, b = np.argwhere(bad)[0]                  # frame-major: the earliest frame, then the lowest agent
        ens._raise_on_err(np.array([res["pc_err"][t, b] & ~nat.ERR_INJECT_LOC], dtype=np.int32))
    length = lengths[rec_of].astype(np.int64)
    past = np.arange(T)[None, :] >= length[:, None]  # [B, T]
    n_templates = res["n_templates"][-1].astype(np.int64) if T else np.zeros(B, np.int64)
    argmax = _unravel(res["argmax"].T, pose_size)
    argmax[past] = -1
    out = {"template": res["template_index"].T.astype(np.int64), "created": res["created"].T != 0, "argmax": argmax,
           "n_templates": n_templates, "length": length,
           "agents": EnsembleAgents(ens, libs, loc, n_templates, pose_size)}
    if experience_map == "device":
        out.update(xens._maps(res["template_index"], np.ascontiguousarray(res["argmax"]), moved, tw, pose_size,
                              experience_links, 1.0, 0.5, dev, rec_of=rec_of))
    elif experience_map:
        out["n_exp"], out["em_xy"] = _experience_maps(out, moved, tw, pose_size, experience_links, rec_of)
    if experience_map:
        for k in ("n_exp", "exp_id"):
            if k in out:
                out[k][past] = -1
        out["em_xy"][past] = np.nan
    return out


def _list(text, parse):
    return [parse(v.strip()) for v in text.split(",") if v.strip()]


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="Replay ROS1 bags through an ensemble of RatSLAM agents: the cross product "
                                             "of the bags and the given parameter lists, one agent per combination")
    ap.add_argument("bag", nargs="+")
    ap.add_argument("--match-threshold", default=str(MATCH_THRESHOLD), metavar="T1,T2,...")
    ap.add_argument("--global-inhibition", default="0.2", metavar="G1,G2,...")
    ap.add_argument("--inject-energy", default="none", metavar="E1,E2,...",
                    help="energies injected at the matched template's pose cell; 'none' = no injection")
    ap.add_argument("--experience-links", action="store_true",
                    help="build every agent's linked experience map on the device and print its experience and "
                         "loop-closure counts")
    ap.add_argument("--image-topic", default="navbot/camera/image")
    ap.add_argument("--odom-topic", default="navbot/odom")
    a = ap.parse_args(argv)
    from . import rosbag_io as rb
    thr = _list(a.match_threshold, float)
    gis = _list(a.global_inhibition, float)
    ens = _list(a.inject_energy, lambda s: None if s.lower() == "none" else float(s))
    combos = list(itertools.product(thr, gis, ens))
    recs = [rb.events_to_arrays(rb.read_events(bag, image_topic=a.image_topic, odom_topic=a.odom_topic))[:2]
            for bag in a.bag]
    several = len(a.bag) > 1
    agents = list(itertools.product(range(len(a.bag)), combos))     # bag-major
    kw = dict(n_agents=len(agents), match_threshold=[c[0] for _, c in agents],
              global_inhibition=[c[1] for _, c in agents], inject_energy=[c[2] for _, c in agents],
              experience_map="device" if a.experience_links else False, experience_links=a.experience_links)
    if several:
        out = replay_ensemble([f for f, _ in recs], [o for _, o in recs], recording=[r for r, _ in agents], **kw)
    else:
        out = replay_ensemble(recs[0][0], recs[0][1], **kw)
    for b, (r, (t, g, e)) in enumerate(agents):
        T = len(recs[r][0])
        last = tuple(int(c) for c in out["argmax"][b, T - 1]) if T else None
        line = ("agent %d  match_threshold %g  global_inhibition %g  inject_energy %s:  templates %d  created %d/%d  "
                "final arg-max %s" % (b, t, g, "none" if e is None else "%g" % e, out["n_templates"][b],
                                      int(out["created"][b].sum()), T, last))
        if several:
            line = "bag %s  %s" % (a.bag[r], line)
        if a.experience_links:
            line += "  experiences %d  loop closures %d" % (out["maps"].n_experiences[b], out["n_loop_closures"][b])
        print(line)


if __name__ == "__main__":
    main()
