"""One recording through B differently parameterised RatSLAM agents in one pass on the GPU.

Tuning RatSLAM offline means replaying one recording under many settings -- the match threshold, the global inhibition,
the view-template -> pose-cell injection energy -- and comparing the runs.  ``replay_ensemble`` runs all of them at
once: agent ``b`` is the ROS loop of ``ros_simulate.replay(native=True, match_threshold=..., inject_energy=...)`` with
``pcn.global_inhibition`` set to its own value, and it has its own pose-cell network, view-template library and
experience map.  Tuning on several recordings keeps the settings from fitting one route: with ``frames`` and ``odom``
given as lists of R recordings, agent ``b`` replays recording ``recording[b]``.  ``replay_ensemble_events`` replays
message streams instead, every odometry message its own pose-cell update, as the node does.

Every form runs as ticks (``prs_ens_run``, csrc/view_templates.cu): a tick is an optional twist and an optional image
per recording, and a frame is a tick with an image.  A tick is one CUDA graph for the whole ensemble: one pose-cell
update of all B networks, one query per recording, one sweep over every agent's library, then the per-agent
create-or-match decision and injection.

``EnsembleSession`` keeps the agents on the device between calls and feeds them recordings in pieces: bags streamed
in chunks, recordings longer than 65535 frames, or a second run of a route continuing the maps of the first.

``ShardedEnsembleSession`` splits the agents over several GPUs (``devices=`` of the replays, ``--devices``).

    python -m pyratslam_b200.ros_ensemble BAG [BAG ...] --match-threshold 30000,45000,60000 --global-inhibition 0.1,0.2
"""
from __future__ import annotations

import ctypes
import itertools
import math
import numbers
import threading

import numpy as np
import torch

from . import _native as nat
from . import experience_ensemble as xens
from .experience_map import ExperienceMap
from .kernels import PC_GLOBAL_INHIB
from .posecell_network import PoseCellEnsemble, _as_np_dtype
from .ros_simulate import (IM_SIZE, MATCH_THRESHOLD, ODOM_FREQ, POSE_SIZE, X_RANGE, X_STEP, Y_RANGE, Y_STEP,
                           RatslamRos, key_scores)

MAX_CAPACITY = 1 << 16          # templates per agent the frame's library sweep takes (kSmallLibrary)


class _Keep:
    """The value of an omitted ``EnsembleSession.reassign`` setting: each agent keeps its parent's.  (``None`` is a
    setting: no injection.)"""

    def __repr__(self):
        return "KEEP"


KEEP = _Keep()


def _real(v):
    return isinstance(v, (numbers.Real, np.number)) and not isinstance(v, (bool, np.bool_))


def agent_parameters(n_agents=None, match_threshold=MATCH_THRESHOLD, global_inhibition=PC_GLOBAL_INHIB,
                     inject_energy=None):
    """Broadcast the per-agent parameters to B agents and validate them (no CUDA involved).

    Each parameter is a scalar or a length-B sequence; B is ``n_agents`` or the length of the sequences.  Returns
    ``(B, thresholds float64[B], gi float64[B], energies list of float-or-None)``; a threshold is the caller's number, as
    ``ViewTemplates`` compares it: a frame creates a template when its best score is strictly above it, so a negative
    threshold creates on every frame.  ``ValueError`` for disagreeing lengths, non-finite thresholds or inhibitions, and
    energies that are negative or not finite."""
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
        thr.append(float(v))
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
    return B, np.array(thr, dtype=np.float64), np.array(gi, dtype=np.float64), energies


def reassign_parameters(parents, rec_of, match_threshold, global_inhibition, inject_energy, new_threshold=KEEP,
                        new_inhibition=KEEP, new_energy=KEEP):
    """``EnsembleSession.reassign``'s arguments validated (no CUDA involved): ``parents`` against the agents'
    recordings ``rec_of [B]``, and the children's settings -- each the parent's setting of the current
    ``match_threshold``, ``global_inhibition`` and ``inject_energy`` (caller order), or the ``new_*`` value where it is
    not ``KEEP``, broadcast and validated by ``agent_parameters``.  Returns ``(parents int64 [B], thresholds,
    inhibitions, energies)``; ``ValueError`` for a wrong length, a parent that is not an integer in [0, B) or replays
    another recording than its child, and refused settings."""
    B = len(rec_of)
    if isinstance(parents, (str, bytes)):
        raise ValueError("parents must be a sequence of %d agent indices, got %r" % (B, parents))
    try:
        par = list(parents)
    except TypeError:
        raise ValueError("parents must be a sequence of %d agent indices, got %r" % (B, parents)) from None
    if len(par) != B:
        raise ValueError("parents has %d values for %d agents" % (len(par), B))
    for p in par:
        if (not isinstance(p, (numbers.Integral, np.integer)) or isinstance(p, (bool, np.bool_))
                or not 0 <= int(p) < B):
            raise ValueError("parents must be agent indices in [0, %d), got %r" % (B, p))
    par = np.array(par, dtype=np.int64)
    rec_of = np.asarray(rec_of)
    cross = np.nonzero(rec_of[par] != rec_of)[0]
    if len(cross):
        b = int(cross[0])
        raise ValueError("agent %d replays recording %d, its parent %d recording %d: an agent continues from its own "
                         "recording's position" % (b, rec_of[b], par[b], rec_of[par[b]]))
    pick = lambda new, own: own if new is KEEP else new                   # noqa: E731
    _, thr, gi, energies = agent_parameters(B, pick(new_threshold, np.asarray(match_threshold)[par]),
                                            pick(new_inhibition, np.asarray(global_inhibition)[par]),
                                            pick(new_energy, [inject_energy[p] for p in par]))
    return par, thr, gi, energies


def activity_parameters(activity_threshold=None, max_active_cells=128, pose_size=POSE_SIZE):
    """The pose-cell activity capture's settings validated (no CUDA involved): ``activity_threshold`` None (no capture)
    or a finite real number, ``max_active_cells`` an integer in [0, X*Y*Th] (0: counts only).  Returns ``(threshold
    float or None, max_cells int)``; ``ValueError`` otherwise."""
    if activity_threshold is not None and (not _real(activity_threshold)
                                           or not math.isfinite(float(activity_threshold))):
        raise ValueError("activity_threshold must be None or a finite number, got %r" % (activity_threshold,))
    n = int(np.prod([int(s) for s in pose_size]))
    if (not isinstance(max_active_cells, (numbers.Integral, np.integer)) or isinstance(max_active_cells, (bool, np.bool_))
            or not 0 <= int(max_active_cells) <= n):
        raise ValueError("max_active_cells must be an integer in [0, %d], got %r" % (n, max_active_cells))
    return (None if activity_threshold is None else float(activity_threshold)), int(max_active_cells)


def activity_entry(result, b, i):
    """Agent b's activity at image i of a result with the capture on: ``(index int64 [k,3], value float64 [k])``, the
    captured cells (x, y, th) in C order and their values, as ``PoseCellNetwork.active_cells`` returns them.  k is
    ``min(activity_count[b, i], max_active_cells)``, 0 past the agent's length."""
    n = result["activity_count"].shape[1]
    if not 0 <= b < result["activity_count"].shape[0] or not 0 <= i < n:
        raise IndexError("activity_entry: (%r, %r) outside the result's [%d, %d]"
                         % (b, i, result["activity_count"].shape[0], n))
    lo, hi = result["activity_ptr"][b * n + i], result["activity_ptr"][b * n + i + 1]
    return result["activity_cell"][lo:hi], result["activity_value"][lo:hi]


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


def _ens_chunk(R, frame_bytes):
    """Ticks per recording in one device chunk (prs_ens_scratch_bytes): 256 MiB of images over R recordings, in
    [1, 256]."""
    return int(min(max((256 << 20) // (R * frame_bytes), 1), 256))


def _unravel(flat, shape):
    X, Y, Th = shape
    flat = np.asarray(flat, dtype=np.int64)
    return np.stack([flat // (Y * Th), (flat // Th) % Y, flat % Th], axis=-1)


class EnsembleAgents:
    """What every agent holds after the replay: its library, the template locations and its pose cells."""

    def __init__(self, ens, libs, loc, n_templates, shape, rows=None):
        self._ens, self._libs, self._loc = ens, libs, loc
        self._rows = rows           # the ensemble's row of each agent, when it holds them in another order
        self.n_templates = n_templates
        self.shape = shape

    def __len__(self):
        return len(self.n_templates)

    def _row(self, b):
        return b if self._rows is None else int(self._rows[b])

    @property
    def path(self):
        """The pose-cell kernel family that updated the ensemble (``PoseCellEnsemble.path``)."""
        return self._ens.path

    @property
    def state(self):
        """The device tensor ``[B, Th, X, Y]`` of every agent's pose cells (theta-major)."""
        if self._rows is None:
            return self._ens.state
        return self._ens.state[torch.from_numpy(np.asarray(self._rows)).to(self._ens.state.device)]

    def templates(self, b):
        """uint8 ``[n_b, 32, 32]``: agent b's templates as ``ViewTemplate.template`` holds them."""
        n = int(self.n_templates[b])
        lib = self._libs[self._row(b)]
        out = torch.empty((n, 32, 32), dtype=torch.uint8, device=self._libs.device)
        with torch.cuda.device(self._libs.device):
            for i in range(n):
                nat.check(nat.lib().prs_vt_unpack_u8(lib.data_ptr(), i, out[i].data_ptr(), nat.stream_ptr()),
                          "prs_vt_unpack_u8")
            return out.cpu().numpy()

    def locations(self, b):
        """int64 ``[n_b, 3]``: the pose cell each of agent b's templates was created at (``ViewTemplate.location``)."""
        return _unravel(self._loc[self._row(b), :int(self.n_templates[b])].cpu().numpy(), self.shape)

    def posecells(self, b):
        """Agent b's pose cells, float64 ``[X, Y, Th]`` (the reference's layout)."""
        return self._ens.state[self._row(b)].permute(1, 2, 0).cpu().numpy().astype(np.float64)


def grow_capacity(capacity, n_max, t):
    """A session's library growth rule (no CUDA involved): ``(capacity', frames)`` before t more frames when the
    fullest library holds ``n_max`` templates.  capacity' is ``capacity`` while n_max + t fits it, else
    ``min(65536, max(2 * capacity, capacity_for(n_max + t)))``: doubling keeps the growths O(log) per session.  A frame
    appends at most one template, so ``frames = min(t, capacity' - n_max)`` of them fit; fewer than t only at 65536,
    where the rest goes in later sub-runs, and 0 when a library is full."""
    cap = int(capacity)
    if n_max + t > cap:
        cap = min(MAX_CAPACITY, max(2 * cap, capacity_for(n_max + t)))
    return cap, max(min(int(t), cap - int(n_max)), 0)


def _grow_rows(rows, need):
    """Experience-map workspace rows for ``need``: unchanged while they suffice, else doubled (at least ``need``)."""
    return rows if need <= rows else max(2 * rows, need)


def feed_inputs(frames, odom, n_recordings):
    """Validate one feed of a session of ``n_recordings`` recordings (no CUDA involved): with one recording ``frames``
    uint8 [t,256,256] and ``odom`` [t,2]; with R > 1 lists of R such arrays, of any lengths (0 allowed).  Returns lists
    of R contiguous uint8 frame arrays and R float64 odometry arrays; ``ValueError`` otherwise."""
    R = int(n_recordings)
    if R == 1:
        if isinstance(frames, (list, tuple)) or isinstance(odom, (list, tuple)):
            raise ValueError("EnsembleSession.feed: a session of one recording takes arrays, not lists")
        frames, odom = [frames], [odom]
    elif (not isinstance(frames, (list, tuple)) or not isinstance(odom, (list, tuple)) or len(frames) != R
          or len(odom) != R):
        raise ValueError("EnsembleSession.feed: a session of %d recordings takes lists of %d frame and %d odometry "
                         "arrays" % (R, R, R))
    fr, od = [], []
    for r in range(R):
        f = np.asarray(frames[r])
        try:
            o = np.asarray(odom[r], dtype=np.float64)
        except (TypeError, ValueError):
            raise ValueError("EnsembleSession.feed: recording %d: odometry must be numbers" % r) from None
        if f.dtype != np.uint8 or f.ndim != 3 or tuple(f.shape[1:]) != IM_SIZE or o.shape != (len(f), 2):
            raise ValueError("EnsembleSession.feed: recording %d: frames must be uint8 [t,%d,%d] and odom [t,2], got %s "
                             "%r and %r" % (r, IM_SIZE[0], IM_SIZE[1], f.dtype, f.shape, o.shape))
        fr.append(np.ascontiguousarray(f))
        od.append(o)
    return fr, od


def _frame_ticks(frames, odom):
    """Recordings of paired frames and twists as tick streams (``event_ticks``'s form): every tick has an image."""
    return [(np.ascontiguousarray(f), o, xens.gate(o)[0], np.ones(len(f), np.bool_)) for f, o in zip(frames, odom)]


def _is_event(x):
    return isinstance(x, (tuple, list)) and len(x) == 3 and isinstance(x[0], str)


def event_ticks(events):
    """Compact one message stream (``rosbag_io.read_events``) into ticks of (optional gated twist, optional image),
    odometry before image, as ``ros_simulate.replay_events(fused=True)`` folds it (no CUDA involved): an odometry message
    directly followed by an image shares that image's tick, odometry the 0.001 gate drops makes no tick, an image with
    no twist before it is an image-only tick and any other odometry an odometry-only tick.  Returns ``(frames uint8
    [I,256,256], odom float64 [K,2], moved uint8 [K], image bool [K])``: the stream's images in order, and per tick the
    (linear.x, angular.z) twist (0 where it does not move), the gate and whether it has an image.  ``ValueError`` for
    anything that is not such a stream."""
    if isinstance(events, (str, bytes)) or not hasattr(events, "__iter__"):
        raise ValueError("a message stream is a sequence of (kind, stamp, payload) events, got %r" % (events,))
    events = list(events)
    frames, odom, moved, image = [], [], [], []
    i, n = 0, len(events)
    while i < n:
        ev = events[i]
        if not _is_event(ev):
            raise ValueError("event %d is not a (kind, stamp, payload) tuple: %r" % (i, ev))
        kind, _, payload = ev
        if kind == "odom":
            try:
                x, z = float(payload[0]), float(payload[1])
            except (TypeError, ValueError, IndexError):
                raise ValueError("event %d: odometry must be a (linear.x, angular.z) pair, got %r" % (i, payload)) from None
            mv = abs(x) > 0.001 or abs(z) > 0.001                                  # ros_simulate.py:128
            paired = i + 1 < n and _is_event(events[i + 1]) and events[i + 1][0] == "image"
            if mv or paired:
                odom.append((x, z) if mv else (0.0, 0.0))
                moved.append(mv)
                image.append(paired)
                if paired:
                    i += 1
                    frames.append(events[i][2])
            i += 1
            continue
        if kind != "image":
            raise ValueError("event %d: unknown event kind %r" % (i, kind))
        odom.append((0.0, 0.0))
        moved.append(False)
        image.append(True)
        frames.append(payload)
        i += 1
    for j, f in enumerate(frames):
        f = np.asarray(f)
        if f.dtype != np.uint8 or f.shape != IM_SIZE:
            raise ValueError("image %d of the stream must be uint8 %r, got %s %r" % (j, IM_SIZE, f.dtype, f.shape))
        frames[j] = f
    fr = np.stack(frames) if frames else np.zeros((0,) + IM_SIZE, np.uint8)
    return (fr, np.asarray(odom, dtype=np.float64).reshape(-1, 2), np.asarray(moved, dtype=np.uint8),
            np.asarray(image, dtype=np.bool_))


def event_streams(events, n_recordings):
    """One feed of message streams for a session of ``n_recordings`` recordings: a stream for R = 1, a list of R streams
    otherwise.  Returns the R compacted streams (``event_ticks``); ``ValueError`` for anything else."""
    R = int(n_recordings)
    if R == 1:
        return [event_ticks(events)]
    if (isinstance(events, (str, bytes)) or not isinstance(events, (list, tuple)) or len(events) != R
            or any(_is_event(s) for s in events)):
        raise ValueError("EnsembleSession.feed_events: a session of %d recordings takes a list of %d message streams"
                         % (R, R))
    return [event_ticks(s) for s in events]


def _session_arguments(n_agents, match_threshold, global_inhibition, inject_energy, pose_size, dtype, experience_map,
                       n_recordings, recording, capacity, activity_threshold, max_active_cells):
    """``EnsembleSession``'s arguments validated and broadcast (no CUDA involved): ``(B, R, thresholds, inhibitions,
    energies, rec_of, capacity, pose_size, activity threshold, max cells, numpy dtype)``; ``ValueError`` otherwise."""
    if isinstance(experience_map, (bool, np.bool_)) and experience_map:
        raise ValueError("EnsembleSession: experience_map=True replays the maps on the host from whole recordings; "
                         "a session builds them on the device (experience_map='device')")
    if not (isinstance(experience_map, (bool, np.bool_))
            or (isinstance(experience_map, str) and experience_map == "device")):
        raise ValueError("experience_map must be False or 'device', got %r" % (experience_map,))
    if (not isinstance(n_recordings, (numbers.Integral, np.integer)) or isinstance(n_recordings, (bool, np.bool_))
            or n_recordings < 1):
        raise ValueError("n_recordings must be an integer >= 1, got %r" % (n_recordings,))
    R = int(n_recordings)
    B, thr, gi, energies = agent_parameters(n_agents if n_agents is not None else _recording_count(recording),
                                            match_threshold, global_inhibition, inject_energy)
    rec_of = agent_recordings(recording, B, R)
    cap = 32 if capacity is None else capacity
    if not _real(cap) or not 1 <= cap <= MAX_CAPACITY or cap != int(cap):
        raise ValueError("capacity must be an integer in [1, %d], got %r" % (MAX_CAPACITY, capacity))
    cap = (int(cap) + 31) // 32 * 32
    pose_size = tuple(int(s) for s in pose_size)
    act_thr, act_k = activity_parameters(activity_threshold, max_active_cells, pose_size)
    np_dtype = _as_np_dtype(dtype)
    return B, R, thr, gi, energies, rec_of, cap, pose_size, act_thr, act_k, np_dtype


def _full_library(agent, n, unit, frame):
    return ValueError("EnsembleSession: agent %d holds %d templates, the most the library sweep takes, and %s %d of its "
                      "recording remains" % (agent, n, unit, frame))


class EnsembleSession:
    """B RatSLAM agents that stay on the device between calls: ``feed`` replays the next frames of every recording.

    The parameters are those of ``replay_ensemble`` and are validated and broadcast the same way; ``n_recordings`` R
    and ``recording`` (an index or a length-B sequence) say which recording each agent replays, ``capacity`` is the
    initial templates per agent (default 32, rounded up to whole groups of 32).  ``experience_map`` is False or
    "device"; the host replay (True) needs whole recordings and is refused.

    ``feed(frames, odom)`` takes uint8 [t,256,256] and [t,2] (R = 1) or lists of R such arrays of any lengths, 0
    allowed, and continues each recording where the previous feed left it.  It returns what ``replay_ensemble``'s
    several-recordings form returns for the fed frames: ``template``, ``created``, ``score``, ``argmax`` ``[B, t_max]``,
    ``length [B]`` (the agent's recording's frames in this feed, -1 / False past it), ``n_templates [B]``, and with
    ``experience_map="device"`` ``n_exp``, ``exp_id``, ``em_xy`` and ``n_loop_closures``.  Template and experience ids
    are global to the session: concatenating agent b's first ``length[b]`` columns over the feeds gives what
    ``replay_ensemble`` returns on the concatenation of its recording's feeds.  The libraries grow when a feed could
    overfill them (``grow_capacity``), so a session replays any number of frames while no agent holds more than 65536
    templates.  A pose-cell error raises what ``replay_ensemble`` raises and closes the session; a closed session's
    ``feed`` raises ``RuntimeError``.

    ``activity_threshold`` (None: off) captures every agent's pose-cell activity at each image on the device: the
    cells above the threshold in the state the match was made with (after the image's update, before its injection),
    the first ``max_active_cells`` of them in C order, and their true count.  The result then also holds
    ``activity_count [B, i_max]`` (-1 past the length), ``activity_ptr [B * i_max + 1]`` (row pointers over the (agent,
    image) pairs, row-major), ``activity_cell int64 [n, 3]`` and ``activity_value float64 [n]``; ``activity_entry``
    returns one entry.  Concatenating agent b's entries over the feeds gives the one-call activity."""

    def __init__(self, n_agents=None, match_threshold=MATCH_THRESHOLD, global_inhibition=PC_GLOBAL_INHIB,
                 inject_energy=None, pose_size=POSE_SIZE, dtype=np.float32, active_set=0, experience_map=False,
                 experience_links=False, n_recordings=1, recording=0, capacity=None, activity_threshold=None,
                 max_active_cells=128):
        self._plan, self._ens, self._work = None, None, None
        self._closed = True
        # the error a feed raised, where it names a tick and an agent: (tick of the feed, agent, and for a full library
        # the (templates, unit, frame) of its message)
        self._fault = None
        B, R, thr, gi, energies, rec_of, cap, pose_size, act_thr, act_k, np_dtype = _session_arguments(
            n_agents, match_threshold, global_inhibition, inject_energy, pose_size, dtype, experience_map, n_recordings,
            recording, capacity, activity_threshold, max_active_cells)
        nat.require_cuda()
        dev = torch.device("cuda", torch.cuda.current_device())
        self.B, self.R, self.pose_size, self.capacity = B, R, pose_size, cap
        self._act_thr, self._act_k, self._act_buf = act_thr, act_k, None    # the capture's settings and buffer
        self._cells = None
        self._np_dtype = np_dtype
        self._thr, self._gi, self._energies = thr, gi, list(energies)     # the settings in force, caller order
        self._dev, self._rec_of = dev, rec_of
        self._map = isinstance(experience_map, str)
        self._linked = self._map and bool(experience_links)
        # the agents of one recording get contiguous indices on the device (the sweep reloads a query per recording
        # change); _order[d] is the agent at device row d, _rows[b] the device row of agent b
        self._order = np.argsort(rec_of, kind="stable")
        self._rows = np.argsort(self._order)
        self._ens = ens = PoseCellEnsemble(pose_size, B, global_inhibition=gi[self._order], dtype=np_dtype, device=dev,
                                           active_set=active_set)
        ens.inject(1, tuple(math.floor(s / 2) for s in pose_size))         # RatslamRos.__init__
        L = nat.lib()
        self._libs = torch.zeros((B, int(L.prs_vt_packed_bytes(cap))), dtype=torch.uint8, device=dev)
        self._loc = torch.full((B, cap), -1, dtype=torch.int64, device=dev)
        self._n_dev = torch.zeros(B, dtype=torch.int32, device=dev)
        self._thr_dev = torch.from_numpy(thr[self._order]).to(dev)
        injecting = any(e is not None for e in energies)
        self._energy_dev = torch.tensor([-1.0 if energies[i] is None else energies[i] for i in self._order],
                                        dtype=torch.float64, device=dev) if injecting else None
        self._rec_dev = torch.from_numpy(rec_of[self._order].astype(np.int32)).to(dev)
        self._pc_work = torch.zeros(3 * B, dtype=torch.int64, device=dev)
        self._scratch = torch.empty(int(L.prs_ens_scratch_bytes(ens._h, R, IM_SIZE[0], IM_SIZE[1])), dtype=torch.uint8,
                                    device=dev)
        self._stream = torch.cuda.Stream(device=dev)
        self.frames_fed = np.zeros(R, np.int64)
        self._n = np.zeros(B, np.int64)                       # templates per device row
        self._prev_tpl = np.full(B, -1, np.int32)             # per device row: the template of its last frame
        self._dr = [(0, (0, 0, 0))] * R                       # per recording: the dead reckoning's (n_exp, accum)
        self._counts = np.zeros((4, B), np.int64)             # per device row: the linked map's counts
        self._counts[2] = -1
        with torch.cuda.device(dev):
            nat.check(L.prs_pc_argmax(ens._h, ens.state.data_ptr(), self._pc_work.data_ptr(), nat.stream_ptr()),
                      "prs_pc_argmax")
            torch.cuda.current_stream(dev).synchronize()
            self._create_plan()
            self._closed = False
            if self._linked:
                self._E, self._N = cap, cap
                self._work = torch.empty(int(L.prs_em_session_bytes(B, self._E, self._N)), dtype=torch.uint8,
                                         device=dev)
                nat.check(L.prs_em_session_init(B, self._E, self._N, self._work.data_ptr(), nat.stream_ptr()),
                          "prs_em_session_init")

    # ------------------------------------------------------------------ the plan and its growth
    def _create_plan(self):
        L = nat.lib()
        plan = ctypes.c_void_p()
        e = self._ens
        nat.check(L.prs_ens_create(
            e._h, e.state.data_ptr(), e._gi.data_ptr(), self._pc_work.data_ptr(), self._libs.data_ptr(), self.capacity,
            self._n_dev.data_ptr(), self._thr_dev.data_ptr(),
            None if self._energy_dev is None else self._energy_dev.data_ptr(), self._loc.data_ptr(), self.R,
            self._rec_dev.data_ptr(), nat.VT_MODE_REF, IM_SIZE[0], IM_SIZE[1], Y_RANGE[0], Y_RANGE[1], Y_STEP,
            X_RANGE[0], X_RANGE[1], X_STEP, self._scratch.data_ptr(), ctypes.byref(plan)), "prs_ens_create")
        self._plan = plan
        self._room = self.capacity - int(self._n.max())
        self._chunk = int(L.prs_ens_chunk(plan))
        if self._act_thr is not None:
            # every plan of the session captures (a growth or an injection change makes the plan again); the buffer
            # depends on B, the chunk and the dtype only, so it is made once
            if self._act_buf is None:
                self._act_buf = torch.empty(int(L.prs_ens_activity_bytes(plan, self._act_k)), dtype=torch.uint8,
                                            device=self._dev)
            nat.check(L.prs_ens_set_activity(plan, self._act_thr, self._act_k, self._act_buf.data_ptr()),
                      "prs_ens_set_activity")

    def _grow(self, cap):
        """Libraries of ``cap`` templates: a larger library is the old one with groups appended, so each agent's row is
        copied as a prefix; the plan is made again on the new buffers (its graphs are captured again)."""
        L = nat.lib()
        libs = torch.zeros((self.B, int(L.prs_vt_packed_bytes(cap))), dtype=torch.uint8, device=self._dev)
        libs[:, :self._libs.shape[1]].copy_(self._libs)
        loc = torch.full((self.B, cap), -1, dtype=torch.int64, device=self._dev)
        loc[:, :self.capacity].copy_(self._loc)
        torch.cuda.current_stream(self._dev).synchronize()
        L.prs_ens_destroy(self._plan)
        self._plan = None
        self._libs, self._loc, self.capacity = libs, loc, cap
        self._create_plan()

    def _grow_maps(self, E, N):
        L = nat.lib()
        work = torch.empty(int(L.prs_em_session_bytes(self.B, E, N)), dtype=torch.uint8, device=self._dev)
        nat.check(L.prs_em_session_grow(self.B, self._E, self._N, E, N, self._work.data_ptr(), work.data_ptr(),
                                        nat.stream_ptr()), "prs_em_session_grow")
        self._work, self._E, self._N = work, E, N

    # ------------------------------------------------------------------ reassigning agents
    def reassign(self, parents, match_threshold=KEEP, global_inhibition=KEEP, inject_energy=KEEP):
        """Make agent b an exact copy of agent ``parents[b]`` as it was before the call, then give the agents new
        settings; call it between feeds.  The next feed continues every agent from the current frame.

        ``parents`` is a length-B sequence of agent indices in the caller's order; ``parents[b] == b`` leaves agent b
        as it is, and any mapping is valid (many children of one parent, swaps, cycles).  A copy is everything a later
        feed reads: the pose cells and their cached arg-max, the library, the template locations, the template of the
        last image (the map tag of ``feed_events``), the linked map with its loop closures, and the parent's settings.
        A setting given replaces the copied one for every agent; it is a scalar or a length-B sequence, broadcast and
        validated as ``agent_parameters`` does, and ``inject_energy=None`` turns injection off.  ``KEEP`` (the
        default) keeps the copied settings.  ``ValueError`` before any CUDA call for a wrong length, a non-integer or
        out-of-range parent, a parent that replays another recording than its child, or refused settings;
        ``RuntimeError`` on a closed session.  The copies run as kernels over the live bytes of the device rows; an
        error there closes the session, as in ``feed``."""
        if self._closed:
            raise RuntimeError("EnsembleSession: the session is closed")
        B = self.B
        par, thr, gi, energies = reassign_parameters(parents, self._rec_of, self._thr, self._gi, self._energies,
                                                     match_threshold, global_inhibition, inject_energy)
        moves = np.nonzero(par != np.arange(B))[0]
        try:
            self._reassign(par, moves, thr, gi, energies)
        except BaseException:
            self.close()
            raise

    def _reassign(self, par, moves, thr, gi, energies):
        L = nat.lib()
        with torch.cuda.device(self._dev):
            if len(moves):
                dst = np.ascontiguousarray(self._rows[moves], dtype=np.int32)
                src = np.ascontiguousarray(self._rows[par[moves]], dtype=np.int32)
                self._copy_rows(L, dst, src)
            self._thr, self._gi = thr, gi
            self._thr_dev.copy_(torch.from_numpy(thr[self._order]))
            self._ens.global_inhibition = gi[self._order]
            was_injecting = self._energy_dev is not None
            self._energies = energies
            injecting = any(e is not None for e in energies)
            e_rows = torch.tensor([-1.0 if energies[i] is None else energies[i] for i in self._order],
                                  dtype=torch.float64)
            if injecting and was_injecting:
                self._energy_dev.copy_(e_rows)
            self._stream.wait_stream(torch.cuda.current_stream(self._dev))
            if injecting != was_injecting:
                # the plan has an injection node exactly when some agent injects: made again, as _grow makes it
                self._energy_dev = e_rows.to(self._dev) if injecting else None
                torch.cuda.current_stream(self._dev).synchronize()
                L.prs_ens_destroy(self._plan)
                self._plan = None
                self._create_plan()

    def _copy_rows(self, L, dst, src):
        """Device rows ``dst[m]`` <- ``src[m]`` in the plan's buffers and the map workspace, and the host's copies of
        their counts and last templates."""
        n = len(dst)
        stream = nat.stream_ptr()
        n_tpl = np.ascontiguousarray(self._n, dtype=np.int32)
        args = (n, dst.ctypes.data, src.ctypes.data)
        stage = torch.empty(int(L.prs_ens_copy_stage_bytes(self._plan, *args, n_tpl.ctypes.data)), dtype=torch.uint8,
                            device=self._dev)
        nat.check(L.prs_ens_copy_agents(self._plan, *args, n_tpl.ctypes.data, stage.data_ptr(), stage.numel(), stream),
                  "prs_ens_copy_agents")
        if self._linked:
            n_rows = np.ascontiguousarray(self._counts[:2].max(axis=0), dtype=np.int32)
            em_stage = torch.empty(int(L.prs_em_session_copy_stage_bytes(self.B, self._E, self._N, *args,
                                                                         n_rows.ctypes.data)),
                                   dtype=torch.uint8, device=self._dev)
            nat.check(L.prs_em_session_copy_agents(self.B, self._E, self._N, self._work.data_ptr(), *args,
                                                   n_rows.ctypes.data, em_stage.data_ptr(), em_stage.numel(), stream),
                      "prs_em_session_copy_agents")
            self._counts[:, dst] = self._counts[:, src]
        self._n[dst] = self._n[src]
        self._prev_tpl[dst] = self._prev_tpl[src]
        self._ens._state_gen += 1

    # ------------------------------------------------------------------ agents carried to another session
    def _export_agents(self, agents):
        """Stages of agents ``agents`` (caller order, repeats allowed) as they are now, on the session's device:
        ``(plan stage, map stage or None, host state)`` for ``_import_agents`` of another session (prs_ens_export_agents,
        prs_em_session_export_agents).  Asynchronous on the current stream."""
        L = nat.lib()
        rows = np.ascontiguousarray(self._rows[agents], dtype=np.int32)
        n, stream = len(rows), nat.stream_ptr()
        n_tpl = np.ascontiguousarray(self._n, dtype=np.int32)
        stage = torch.empty(int(L.prs_ens_export_stage_bytes(self._plan, n, rows.ctypes.data, n_tpl.ctypes.data)),
                            dtype=torch.uint8, device=self._dev)
        nat.check(L.prs_ens_export_agents(self._plan, n, rows.ctypes.data, n_tpl.ctypes.data, stage.data_ptr(),
                                          stage.numel(), stream), "prs_ens_export_agents")
        em_stage = None
        if self._linked:
            n_rows = np.ascontiguousarray(self._counts[:2].max(axis=0), dtype=np.int32)
            em_stage = torch.empty(int(L.prs_em_session_export_stage_bytes(self.B, self._E, self._N, n, rows.ctypes.data,
                                                                           n_rows.ctypes.data)),
                                   dtype=torch.uint8, device=self._dev)
            nat.check(L.prs_em_session_export_agents(self.B, self._E, self._N, self._work.data_ptr(), n,
                                                     rows.ctypes.data, n_rows.ctypes.data, em_stage.data_ptr(),
                                                     em_stage.numel(), stream), "prs_em_session_export_agents")
        host = {"n": self._n[rows].copy(), "prev_tpl": self._prev_tpl[rows].copy(),
                "counts": self._counts[:, rows].copy(), "N": self._N if self._linked else 0}
        return stage, em_stage, host

    def _fit_agents(self, host):
        """Grow the libraries and the map workspace to take the exported agents ``host`` describes."""
        need = max(int(host["n"].max()), int(host["N"]))
        cap, _ = grow_capacity(self.capacity, need, 0)
        if cap != self.capacity:
            self._grow(cap)
        if self._linked:
            E = _grow_rows(self._E, int(host["counts"][:2].max()))
            N = self.capacity if self._N < host["N"] else self._N
            if E != self._E or N != self._N:
                self._grow_maps(E, N)

    def _import_agents(self, agents, stage, em_stage, host):
        """Agents ``agents`` (caller order, distinct) become the exported ones, from stages on this session's device
        (prs_ens_import_agents, prs_em_session_import_agents); ``_fit_agents`` ran before.  On the current stream."""
        L = nat.lib()
        rows = np.ascontiguousarray(self._rows[agents], dtype=np.int32)
        n, stream = len(rows), nat.stream_ptr()
        nat.check(L.prs_ens_import_agents(self._plan, n, rows.ctypes.data, stage.data_ptr(), stage.numel(), stream),
                  "prs_ens_import_agents")
        if self._linked:
            nat.check(L.prs_em_session_import_agents(self.B, self._E, self._N, self._work.data_ptr(), n,
                                                     rows.ctypes.data, em_stage.data_ptr(), em_stage.numel(), stream),
                      "prs_em_session_import_agents")
            self._counts[:, rows] = host["counts"]
        self._n[rows] = host["n"]
        self._prev_tpl[rows] = host["prev_tpl"]
        self._ens._state_gen += 1
        self._stream.wait_stream(torch.cuda.current_stream(self._dev))

    @property
    def match_threshold(self):
        """float64 [B]: every agent's match threshold in force, in the caller's order."""
        return self._thr.copy()

    @property
    def global_inhibition(self):
        """float64 [B]: every agent's global inhibition in force, in the caller's order."""
        return self._gi.copy()

    @property
    def inject_energy(self):
        """list of B energies (None = no injection) in force, in the caller's order."""
        return list(self._energies)

    # ------------------------------------------------------------------ feeding
    def feed(self, frames, odom):
        """Replay the next frames of every recording; see the class documentation for the inputs and the result."""
        if self._closed:
            raise RuntimeError("EnsembleSession: the session is closed")
        fr, od = feed_inputs(frames, odom, self.R)
        return self._feed_ticks(_frame_ticks(fr, od), "frame")

    def feed_events(self, events):
        """Replay the next messages of every recording the way the node's message loop does
        (``ros_simulate.replay_events``): one pose-cell update and one experience-map update per gated odometry message,
        one match per image.  ``events`` is a message stream (``rosbag_io.read_events``, or a piece of ``iter_events``)
        for R = 1 and a list of R streams otherwise, any of them empty; a piece may end anywhere, inside a run of
        odometry too.  The streams are compacted into ticks (``event_ticks``).  Returns per image: ``template``, ``created``, ``score``, ``argmax`` ``[B, i_max]``,
        ``length [B]`` (the images of the agent's recording in this feed; -1 / False past it), ``n_templates [B]``, and
        with ``experience_map="device"`` ``n_exp``, ``exp_id``, ``em_xy`` at each image (-1 / NaN past the length) and
        ``n_loop_closures``.  ``feed`` and ``feed_events`` continue the same agents, libraries and maps.  With the
        activity capture on, its entries are per image too: the state each image's match was made with; odometry-only
        ticks capture nothing (there is no per-update capture of message streams)."""
        if self._closed:
            raise RuntimeError("EnsembleSession: the session is closed")
        return self._feed_ticks(event_streams(events, self.R), "image")

    def _feed_ticks(self, streams, unit="image"):
        """The feed of R tick streams (``event_ticks``'s form) with the result of ``feed_events``: per image, ``unit``
        ("frame" or "image") naming one in the error of a full library."""
        R, B = self.R, self.B
        n_ticks = np.array([len(st[2]) for st in streams], dtype=np.int64)
        n_img = np.array([len(st[0]) for st in streams], dtype=np.int64)
        K = int(n_ticks.max())
        moved = np.zeros((K, R), np.uint8)             # past a recording's ticks: no update, no image
        tw = np.zeros((K, R, 2))
        img = np.zeros((K, R), np.bool_)
        for r, (_, od, mv, im) in enumerate(streams):
            moved[:n_ticks[r], r] = mv
            tw[:n_ticks[r], r] = od / float(ODOM_FREQ)                 # the twist given to update(), as xens.gate
            img[:n_ticks[r], r] = im
        gate = np.ascontiguousarray(img.astype(np.uint8) | (moved << 1))
        img_tick = img.any(axis=1)
        res = np.empty((K, B), dtype=RatslamRos._RESULT_DTYPE)    # device rows; every tick's records are written
        rec_rows = self._rec_of[self._order]                        # per device row: its recording
        if self._linked:
            n_exp = np.zeros((K, B), np.int32)
            exp_id = np.zeros((K, B), np.int32)
            em_xy = np.zeros((K, B, 2))
        first = np.zeros(R, np.int64)                  # per recording: its first image of the sub-run
        if self._act_thr is not None:                  # per tick and device row the count, and the packed cells
            act_counts, act_cells = np.full((K, B), -1, np.int32), []
        try:
            with torch.cuda.device(self._dev):
                k0 = 0
                while k0 < K:
                    left = int(img_tick[k0:].sum())
                    cap, run = grow_capacity(self.capacity, int(self._n.max()), left)
                    if run == 0 and left:
                        d = int(np.argmax(self._n))
                        frame = int(self.frames_fed[rec_rows[d]] + first[rec_rows[d]])
                        self._fault = (k0, int(self._order[d]), (int(self._n[d]), unit, frame))
                        raise _full_library(self._order[d], self._n[d], unit, frame)
                    if cap != self.capacity:
                        self._grow(cap)
                    # ticks [k0, k1) hold `run` ticks with images; the last sub-run takes the trailing odometry
                    k1 = K if run >= left else k0 + int(np.nonzero(img_tick[k0:])[0][run])
                    if self._room < min(run, left):
                        nat.check(nat.lib().prs_ens_refresh_room(self._plan, ctypes.c_void_p(self._stream.cuda_stream)),
                                  "prs_ens_refresh_room")
                        self._room = self.capacity - int(self._n.max())
                    sub = slice(k0, k1)
                    sub_img = img[sub].sum(axis=0)
                    self._run(streams, first, sub_img, tw[sub], moved[sub], gate[sub], res[sub],
                              None if self._act_thr is None else (act_counts[sub], act_cells), k0)
                    self._room -= int(img_tick[sub].sum())
                    self._n = res["n_templates"][k1 - 1].astype(np.int64)
                    if self._linked:
                        self._maps(res[sub], self._event_tags(res[sub], img[sub][:, rec_rows]),
                                   int(moved[sub].sum(axis=0).max()), tw[sub], moved[sub], n_exp[sub], exp_id[sub],
                                   em_xy[sub])
                    first += sub_img
                    k0 = k1
        except BaseException:
            self.close()
            raise
        self.frames_fed += n_img
        length = n_img[self._rec_of]
        i_max = int(n_img.max())
        # built in device rows, where each recording's agents are one slice, and put in the caller's order at the end
        out = {"template": np.full((B, i_max), -1, np.int64), "created": np.zeros((B, i_max), np.bool_),
               "score": np.full((B, i_max), -1, np.int64), "argmax": np.full((B, i_max, 3), -1, np.int64)}
        if self._map:
            out["n_exp"] = np.full((B, i_max), -1, np.int64)
            out["exp_id"] = np.full((B, i_max), -1, np.int64)
            out["em_xy"] = np.full((B, i_max, 2), np.nan)
        for r in range(R):
            d = slice(*np.searchsorted(rec_rows, [r, r + 1]))
            ticks = np.nonzero(img[:, r])[0]
            m = len(ticks)
            at = slice(0, m) if m == 0 or ticks[-1] == m - 1 else ticks    # a frame feed's images: the first m ticks
            sel = res[at, d]
            out["template"][d, :m] = sel["template_index"].T
            out["created"][d, :m] = sel["created"].T != 0
            out["score"][d, :m] = key_scores(sel["key"].T)
            out["argmax"][d, :m] = _unravel(sel["argmax"].T, self.pose_size)
            if self._linked:
                out["n_exp"][d, :m] = n_exp[at, d].T
                out["exp_id"][d, :m] = exp_id[at, d].T
                out["em_xy"][d, :m] = em_xy[at, d].transpose(1, 0, 2)
            if self._map:
                n_r, xy_r = self._dead_reckoning(r, moved[:, r], tw[:, r], n_ticks[r])
                if not self._linked:
                    out["n_exp"][d, :m] = n_r[ticks]
                    out["exp_id"][d, :m] = n_r[ticks] - 1
                    out["em_xy"][d, :m] = xy_r[ticks]
        if not (self._order == np.arange(B)).all():
            out = {k: v[self._rows] for k, v in out.items()}
        out["n_templates"], out["length"] = self.n_templates, length
        if self._map:
            out["n_loop_closures"] = self.n_loop_closures
        if self._act_thr is not None:
            out.update(self._activity(act_counts, act_cells, img, i_max))
        return out

    def _activity(self, counts, cells, img, i_max):
        """The activity keys of one feed in the caller's order, from ``counts [K,B]`` (per tick and device row) and
        the packed cells of its runs (tick-major, then device row), selected per recording as the records are."""
        B, k_max = self.B, self._act_k
        kept = np.clip(counts, 0, k_max).astype(np.int64)
        start = (np.cumsum(kept.ravel()) - kept.ravel()).reshape(kept.shape)     # first packed cell of each entry
        idx = np.concatenate([c[0] for c in cells] + [np.zeros(0, np.int32)])
        val = np.concatenate([c[1] for c in cells] + [np.zeros(0, self._np_dtype)])
        count = np.full((B, i_max), -1, np.int64)
        src = np.zeros((B, i_max), np.int64)
        for r in range(self.R):
            ticks = np.nonzero(img[:, r])[0]
            agents = np.nonzero(self._rec_of == r)[0]
            d = self._rows[agents]
            count[agents, :len(ticks)] = counts[ticks][:, d].T
            src[agents, :len(ticks)] = start[ticks][:, d].T
        n = np.clip(count, 0, k_max).ravel()
        ptr = np.zeros(B * i_max + 1, np.int64)
        np.cumsum(n, out=ptr[1:])
        g = np.repeat(src.ravel() - ptr[:-1], n) + np.arange(ptr[-1])
        if self._cells is None:         # flat C-order index -> (x, y, th): one row gather per cell instead of divisions
            self._cells = _unravel(np.arange(int(np.prod(self.pose_size))), self.pose_size)
        return {"activity_count": count, "activity_ptr": ptr, "activity_cell": self._cells[idx[g]],
                "activity_value": val[g].astype(np.float64)}

    def _run(self, streams, first, sub_img, tw, moved, gate, res, act=None, k0=0):
        """One sub-run of ticks through ``prs_ens_run``; with the activity capture, ``act`` = (counts [T,B], list of
        packed cells) receives it, one device chunk of ticks per run.  A pose-cell error raises what the native replay
        raises, for the earliest tick: with one recording, with the bits of every agent at it (they share the
        odometry), else for the lowest agent at it."""
        L = nat.lib()
        fb = IM_SIZE[0] * IM_SIZE[1]
        stream = ctypes.c_void_p(self._stream.cuda_stream)
        T = len(gate)
        step = max(T if act is None else self._chunk, 1)         # the capture packs the ticks of one chunk per run
        at = np.array(first, dtype=np.int64)
        for a in range(0, T, step):
            z = min(a + step, T)
            n_img = sub_img if step == T else (gate[a:z] & 1).sum(axis=0).astype(np.int64)
            ptrs = (ctypes.c_void_p * self.R)(*[streams[r][0].ctypes.data + int(at[r]) * fb if n_img[r] else None
                                                for r in range(self.R)])
            tw_p, n_images = np.ascontiguousarray(tw[a:z]), np.ascontiguousarray(n_img, dtype=np.int32)
            gate_p = np.ascontiguousarray(gate[a:z])
            nat.check(L.prs_ens_run(self._plan, ptrs, tw_p.ctypes.data, gate_p.ctypes.data, n_images.ctypes.data,
                                    z - a, res[a:z].ctypes.data, stream), "prs_ens_run")
            if act is not None:
                counts = np.empty((z - a, self.B), np.int32)
                total = ctypes.c_longlong(0)
                nat.check(L.prs_ens_activity_pack(self._plan, counts.ctypes.data, ctypes.byref(total), stream),
                          "prs_ens_activity_pack")
                idx, val = np.empty(total.value, np.int32), np.empty(total.value, self._np_dtype)
                nat.check(L.prs_ens_activity_copy(self._plan, total.value, idx.ctypes.data, val.ctypes.data, stream),
                          "prs_ens_activity_copy")
                act[0][a:z] = counts
                act[1].append((idx, val))
            at += n_img
        err = res["pc_err"] & ~nat.ERR_INJECT_LOC                            # device rows
        bad = (err != 0) & (moved[:, self._rec_of[self._order]] != 0)
        if not bad.any():
            return
        t = int(np.nonzero(bad.any(axis=1))[0][0])
        self._fault = (k0 + t, int(self._order[np.nonzero(bad[t])[0]].min()), None)    # the feed's tick k0 + t
        if self.R == 1:
            self._ens._raise_on_err(err[t].astype(np.int32))
        d = self._rows[np.nonzero(bad[t, self._rows])[0][0]]
        self._ens._raise_on_err(err[t, d:d + 1].astype(np.int32))

    def _event_tags(self, res, img):
        """``tag [K,B]`` of one sub-run of ticks (device rows): the template of the agent's most recent image before
        each tick (``RatslamRos._em_update``'s ``published_index[-1]``), carried across sub-runs and feeds."""
        K, B = res.shape
        last = np.where(img, np.arange(K)[:, None], -1)
        np.maximum.accumulate(last, axis=0, out=last)
        filled = np.where(last >= 0, res["template_index"][np.maximum(last, 0), np.arange(B)[None, :]],
                          self._prev_tpl[None, :]).astype(np.int32)
        tag = np.empty((K, B), np.int32)
        tag[0] = self._prev_tpl
        tag[1:] = filled[:-1]
        if K:
            self._prev_tpl = filled[-1].copy()
        return tag

    def _maps(self, res, tag, updates, tw, moved, n_exp, exp_id, em_xy):
        """The linked maps continued over one sub-run's records (device rows): ``tag [T,B]`` is the view each step's
        experience is tagged with, ``updates`` bounds the moved steps of any agent (one experience and one link each)."""
        L = nat.lib()
        T, B = res.shape
        E = _grow_rows(self._E, int(self._counts[:2].max()) + int(updates))
        if E != self._E or self.capacity != self._N:
            self._grow_maps(E, self.capacity)
        X, Y, Th = self.pose_size
        dev = self._dev
        flat_d = torch.from_numpy(np.ascontiguousarray(res["argmax"])).to(dev)
        tag_d = torch.from_numpy(tag).to(dev)
        tw_d = torch.from_numpy(np.ascontiguousarray(tw)).to(dev)
        moved_d = torch.from_numpy(np.ascontiguousarray(moved)).to(dev)
        n_d = torch.empty((T, B), dtype=torch.int32, device=dev)
        id_d = torch.empty((T, B), dtype=torch.int32, device=dev)
        xy_d = torch.empty((T, B, 2), dtype=torch.float64, device=dev)
        nat.check(L.prs_em_linked_resume_run(B, T, self._E, self._N, flat_d.data_ptr(), tag_d.data_ptr(), self.R,
                                             tw_d.data_ptr(), moved_d.data_ptr(),
                                             self._rec_dev.data_ptr() if self.R > 1 else None, X, Y, Th, 1.0,
                                             self._work.data_ptr(), n_d.data_ptr(), id_d.data_ptr(), xy_d.data_ptr(),
                                             nat.stream_ptr()), "prs_em_linked_resume_run")
        lay, end = xens._work_layout(B, self._E, self._N)
        if int(self._work[end:end + 4].view(torch.int32).item()):
            raise RuntimeError("EnsembleSession: the experience-map workspace (%d rows, %d template heads) was too small"
                               % (self._E, self._N))
        o = lay["counts"][0]
        self._counts = self._work[o:o + 16 * B].view(torch.int32).view(4, B).cpu().numpy().astype(np.int64)
        n_exp[:] = n_d.cpu().numpy()
        exp_id[:] = id_d.cpu().numpy()
        em_xy[:] = xy_d.cpu().numpy()

    def _dead_reckoning(self, r, moved, tw, length):
        """Recording r's unlinked map continued over its frames of this feed: ``(n_exp [T], em_xy [T,2])``."""
        n, xy, accum = xens.dead_reckoning(moved, tw, start=self._dr[r])
        if length:
            self._dr[r] = (int(n[length - 1]), accum)
        return n, xy

    # ------------------------------------------------------------------ what the agents hold
    @property
    def n_templates(self):
        """int64 [B]: templates in each agent's library."""
        return self._n[self._rows].copy()

    @property
    def n_experiences(self):
        """int64 [B]: experiences in each agent's map so far (0 without ``experience_map``)."""
        if self._linked:
            return self._counts[0][self._rows].copy()
        if self._map:
            return np.array([self._dr[r][0] for r in self._rec_of], dtype=np.int64)
        return np.zeros(self.B, np.int64)

    @property
    def n_loop_closures(self):
        """int64 [B]: loop closures of each agent's linked map (0 without one)."""
        return self._counts[3][self._rows].copy() if self._linked else np.zeros(self.B, np.int64)

    @property
    def agents(self):
        """``EnsembleAgents``, in the caller's agent order (the libraries as they are now)."""
        if self._ens is None:
            raise RuntimeError("EnsembleSession: the session is closed")
        identity = bool((self._order == np.arange(self.B)).all())
        return EnsembleAgents(self._ens, self._libs, self._loc, self.n_templates, self.pose_size,
                              None if identity else self._rows)

    @property
    def maps(self):
        """``EnsembleExperienceMaps`` of the linked device maps, in the caller's agent order; None without them."""
        if not self._linked or self._work is None:
            return None
        return xens.EnsembleExperienceMaps(self._work, self.B, self._E, self._N, None, None, self.pose_size, 1.0, 0.5,
                                           rec_of=self._rec_of, accum={r: dr[1] for r, dr in enumerate(self._dr)},
                                           cols=self._rows)

    def close(self):
        """Destroy the frame plan; a closed session's ``feed`` raises ``RuntimeError``.  What ``agents`` and ``maps``
        returned before stays readable."""
        if self._plan is not None:
            nat.lib().prs_ens_destroy(self._plan)
            self._plan = None
        self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _device_list(devices):
    """``devices`` validated as a non-empty sequence of CUDA device indices (no CUDA involved): a list of ints."""
    if isinstance(devices, (str, bytes)) or not hasattr(devices, "__iter__"):
        raise ValueError("devices must be a non-empty sequence of CUDA device indices, got %r" % (devices,))
    devs = list(devices)
    if not devs:
        raise ValueError("devices must be a non-empty sequence of CUDA device indices, got %r" % (devices,))
    for d in devs:
        if not isinstance(d, (numbers.Integral, np.integer)) or isinstance(d, (bool, np.bool_)) or int(d) < 0:
            raise ValueError("devices must be CUDA device indices, got %r" % (d,))
    return [int(d) for d in devs]


def _check_devices(devs):
    """``ValueError`` for a device index this process cannot see (after ``nat.require_cuda``)."""
    n = torch.cuda.device_count()
    for d in devs:
        if d >= n:
            raise ValueError("devices: cuda:%d does not exist, %d device(s) are visible" % (d, n))


def shard_agents(rec_of, devices):
    """Split B agents over ``devices`` (no CUDA involved beyond the range check): ``rec_of`` is each agent's recording
    in the caller's order, ``devices`` a non-empty sequence of CUDA device indices, repeats allowed (two shards on one
    device).  The agents sorted by recording (stable) -- the device-row order of ``EnsembleSession`` -- are cut into
    ``len(devices)`` contiguous pieces whose sizes differ by at most one, so a shard holds few recordings and one
    recording may span two shards.  Returns per shard ``(agents, recordings)``: its agents' caller-order indices in that
    order (int64) and the global recordings it holds, increasing (int64); shard-local recording i is
    ``recordings[i]``.

    The split balances agent counts only.  An agent's cost grows with its recording's length and its library's size,
    so shards of long recordings or large libraries take longer, and a feed lasts as long as its slowest shard.

    ``ValueError`` for an empty ``devices``, an entry that is not an integer (bools included), more shards than agents
    and, once CUDA is up, a device index outside ``torch.cuda.device_count()``."""
    devs = _device_list(devices)
    rec_of = np.asarray(rec_of, dtype=np.int64)
    if len(devs) > len(rec_of):
        raise ValueError("devices: %d shards for %d agents; a shard holds at least one agent" % (len(devs), len(rec_of)))
    nat.require_cuda()
    _check_devices(devs)
    return _split(rec_of, len(devs))


def _split(rec_of, n):
    """``shard_agents``'s pieces of ``rec_of`` for n shards (pure)."""
    order = np.argsort(rec_of, kind="stable")
    return [(a, np.unique(rec_of[a])) for a in np.array_split(order, n)]


def _shard_index(shards, B):
    """Per agent: its shard and its index within the shard."""
    shard_of, local_of = np.empty(B, np.int64), np.empty(B, np.int64)
    for i, (a, _) in enumerate(shards):
        shard_of[a], local_of[a] = i, np.arange(len(a))
    return shard_of, local_of


def plan_agent_moves(parents, shards):
    """``ShardedEnsembleSession.reassign``'s moves (no CUDA involved): ``parents`` int [B] (validated) over the
    ``shards`` of ``shard_agents``.  Returns ``(local, cross)``: ``local[s] = (dst, src)``, shard s's in-shard moves as
    local agent indices, and ``cross``, one ``(s, t, src, dst)`` per pair of shards with moves from s to t, the parents'
    local indices in s and the children's in t, children in increasing caller order.  Applied in three steps -- export
    every cross parent from the state before the call, run each shard's in-shard copies, import -- every child ends as
    its parent was before the call."""
    par = np.asarray(parents, dtype=np.int64)
    B = len(par)
    shard_of, local_of = _shard_index(shards, B)
    moved = np.nonzero(par != np.arange(B))[0]
    src_shard, dst_shard = shard_of[par[moved]], shard_of[moved]
    local = []
    for s in range(len(shards)):
        m = moved[(src_shard == s) & (dst_shard == s)]
        local.append((local_of[m], local_of[par[m]]))
    cross = []
    for s in range(len(shards)):
        for t in range(len(shards)):
            m = moved[(src_shard == s) & (dst_shard == t)] if s != t else moved[:0]
            if len(m):
                cross.append((s, t, local_of[par[m]], local_of[m]))
    return local, cross


class ShardedAgents:
    """``EnsembleAgents`` of a sharded session: every accessor goes to the agent's shard and its index there."""

    def __init__(self, parts, shard_of, local_of, n_templates, shape):
        self._parts, self._shard_of, self._local_of = parts, shard_of, local_of
        self.n_templates = n_templates
        self.shape = shape

    def __len__(self):
        return len(self.n_templates)

    def _at(self, b):
        b = int(b)
        return self._parts[self._shard_of[b]], int(self._local_of[b])

    @property
    def path(self):
        """The pose-cell kernel family of each shard (``PoseCellEnsemble.path``)."""
        return [p.path for p in self._parts]

    @property
    def state(self):
        """The device tensor ``[B, Th, X, Y]`` of every agent's pose cells, for one shard only."""
        if len(self._parts) > 1:
            raise RuntimeError("ShardedAgents.state: the pose cells live on %d shards; read each agent's with "
                               "posecells(b)" % len(self._parts))
        st = self._parts[0].state
        return st[torch.from_numpy(self._local_of).to(st.device)]

    def templates(self, b):
        p, j = self._at(b)
        return p.templates(j)

    def locations(self, b):
        p, j = self._at(b)
        return p.locations(j)

    def posecells(self, b):
        p, j = self._at(b)
        return p.posecells(j)


class ShardedMaps:
    """``EnsembleExperienceMaps`` of a sharded session: per-agent arrays in the caller's order, every accessor going to
    the agent's shard."""

    def __init__(self, parts, shards, shard_of, local_of):
        self._parts, self._shard_of, self._local_of = parts, shard_of, local_of
        B = len(shard_of)
        for k in ("n_experiences", "n_links", "current", "n_loop_closures"):
            v = np.zeros(B, np.int64)
            for (a, _), p in zip(shards, parts):
                v[a] = getattr(p, k)
            setattr(self, k, v)
        self.pose_size = parts[0].pose_size

    def __len__(self):
        return len(self.n_experiences)

    def _at(self, b):
        b = int(b)
        return self._parts[self._shard_of[b]], int(self._local_of[b])

    def experiences(self, b):
        p, j = self._at(b)
        return p.experiences(j)

    def links(self, b):
        p, j = self._at(b)
        return p.links(j)

    def experience_map(self, b):
        p, j = self._at(b)
        return p.experience_map(j)


_FILL = {"template": -1, "created": False, "score": -1, "argmax": -1, "n_exp": -1, "exp_id": -1, "em_xy": np.nan,
         "activity_count": -1}


class ShardedEnsembleSession:
    """``EnsembleSession`` with its agents split over several CUDA devices: ``devices`` (a sequence of device indices,
    repeats allowed) comes first, the other arguments, the methods and the results are ``EnsembleSession``'s.

    ``shard_agents`` cuts the agents, sorted by recording, into one contiguous piece per entry of ``devices``; each
    piece is a plain ``EnsembleSession`` on its device, holding its agents' settings and the recordings they replay.
    A feed runs every shard's ticks in its own host thread (the native runs release the GIL, so the devices overlap)
    and joins them before it returns; the results are merged into the caller's agent order and equal one device's key
    by key, the per-image arrays padded as one device pads them.  An error in any shard closes every shard and raises
    what one device raises, for the earliest tick and, within it, the lowest agent.

    ``reassign`` takes parents anywhere: a child whose parent lives on another shard receives it through a stage
    exported from the parent's device before any shard changes, copied across with one peer copy and imported after
    the shards' own copies (``plan_agent_moves``)."""

    def __init__(self, devices, n_agents=None, match_threshold=MATCH_THRESHOLD, global_inhibition=PC_GLOBAL_INHIB,
                 inject_energy=None, pose_size=POSE_SIZE, dtype=np.float32, active_set=0, experience_map=False,
                 experience_links=False, n_recordings=1, recording=0, capacity=None, activity_threshold=None,
                 max_active_cells=128):
        self._shards, self._closed = [], True
        devs = _device_list(devices)
        B, R, thr, gi, energies, rec_of, cap, pose_size, act_thr, act_k, np_dtype = _session_arguments(
            n_agents, match_threshold, global_inhibition, inject_energy, pose_size, dtype, experience_map, n_recordings,
            recording, capacity, activity_threshold, max_active_cells)
        if len(devs) > B:
            raise ValueError("devices: %d shards for %d agents; a shard holds at least one agent" % (len(devs), B))
        nat.require_cuda()
        _check_devices(devs)
        self.B, self.R, self.pose_size = B, R, pose_size
        self._devs, self._rec_of = devs, rec_of
        self._thr, self._gi, self._energies = thr, gi, list(energies)
        self._map = isinstance(experience_map, str)
        self._linked = self._map and bool(experience_links)
        self._act = act_thr is not None
        self._split = _split(rec_of, len(devs))
        self._shard_of, self._local_of = _shard_index(self._split, B)
        self.frames_fed = np.zeros(R, np.int64)
        try:
            for d, (a, recs) in zip(devs, self._split):
                with torch.cuda.device(d):
                    self._shards.append(EnsembleSession(
                        len(a), thr[a], gi[a], [energies[i] for i in a], pose_size, np_dtype, active_set,
                        experience_map, experience_links, len(recs), np.searchsorted(recs, rec_of[a]), cap, act_thr,
                        act_k))
        except BaseException:
            self.close()
            raise
        self._closed = False

    # ------------------------------------------------------------------ running on every shard
    def _each(self, fn):
        """``fn(i, shard)`` for every shard in its own thread under its device; the threads are joined before it
        returns.  Returns the results; if any shard raised, closes every shard and raises (``_first_error``)."""
        n = len(self._shards)
        results, errors = [None] * n, [None] * n

        def work(i):
            try:
                with torch.cuda.device(self._devs[i]):
                    results[i] = fn(i, self._shards[i])
            except BaseException as e:                  # noqa: B902 -- re-raised on the calling thread
                errors[i] = e

        threads = [threading.Thread(target=work, args=(i,)) for i in range(n)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if any(e is not None for e in errors):
            self.close()
            raise self._first_error(errors)
        return results

    def _first_error(self, errors):
        """The error one device raises: the faults that name a tick and an agent (pose-cell errors, a full library) go
        by (tick, caller agent); a full library's text names the caller's agent."""
        named = [(sh._fault[0], int(self._split[i][0][sh._fault[1]]), i) for i, sh in enumerate(self._shards)
                 if errors[i] is not None and sh._fault is not None]
        if not named:
            return next(e for e in errors if e is not None)
        _, b, i = min(named)
        detail = self._shards[i]._fault[2]
        return errors[i] if detail is None else _full_library(b, *detail)

    def _check_open(self):
        if self._closed:
            raise RuntimeError("EnsembleSession: the session is closed")

    # ------------------------------------------------------------------ feeding
    def feed(self, frames, odom):
        """``EnsembleSession.feed`` over every shard."""
        self._check_open()
        fr, od = feed_inputs(frames, odom, self.R)
        return self._feed_ticks(_frame_ticks(fr, od), "frame")

    def feed_events(self, events):
        """``EnsembleSession.feed_events`` over every shard."""
        self._check_open()
        return self._feed_ticks(event_streams(events, self.R), "image")

    def _feed_ticks(self, streams, unit="image"):
        for sh in self._shards:
            sh._fault = None
        parts = self._each(lambda i, sh: sh._feed_ticks([streams[r] for r in self._split[i][1]], unit))
        n_img = np.array([len(st[0]) for st in streams], dtype=np.int64)
        self.frames_fed += n_img
        return self._merge(parts, int(n_img.max()))

    def _merge(self, parts, i_max):
        """The shards' results in the caller's order: per-image arrays [B, i_max] padded as one device pads them,
        per-agent arrays scattered, and the activity capture's CSR rebuilt over the merged agents."""
        B = self.B
        out = {}
        for k, v in parts[0].items():
            if k.startswith("activity_") and k != "activity_count":
                continue
            if k in _FILL:
                out[k] = np.full((B, i_max) + v.shape[2:], _FILL[k], v.dtype)
                for (a, _), p in zip(self._split, parts):
                    out[k][a, :p[k].shape[1]] = p[k]
            else:
                out[k] = np.zeros(B, v.dtype)
                for (a, _), p in zip(self._split, parts):
                    out[k][a] = p[k]
        if self._act:
            # agent b's entries are one slice of its shard's packed cells (its row of the shard's [B_s, i_s] entries)
            slices = [None] * B
            for (a, _), p in zip(self._split, parts):
                i_s = p["activity_count"].shape[1]
                ptr = p["activity_ptr"]
                for j, b in enumerate(a):
                    slices[b] = (p, ptr[j * i_s], ptr[(j + 1) * i_s])
            n = np.clip(out["activity_count"], 0, None)
            kept = np.minimum(n, self._shards[0]._act_k).ravel()
            ptr = np.zeros(B * i_max + 1, np.int64)
            np.cumsum(kept, out=ptr[1:])
            out["activity_ptr"] = ptr
            out["activity_cell"] = np.concatenate([p["activity_cell"][lo:hi] for p, lo, hi in slices]
                                                  + [np.zeros((0, 3), np.int64)])
            out["activity_value"] = np.concatenate([p["activity_value"][lo:hi] for p, lo, hi in slices]
                                                   + [np.zeros(0)])
        return out

    # ------------------------------------------------------------------ reassigning agents
    def reassign(self, parents, match_threshold=KEEP, global_inhibition=KEEP, inject_energy=KEEP):
        """``EnsembleSession.reassign`` with parents on any shard; ``ValueError`` before any CUDA call for what one
        device refuses.  Every setting is resolved per agent first (KEEP: the parent's, wherever it lives).  Then
        (``plan_agent_moves``): 1. every parent of a child on another shard is exported from the state as it was
        before the call; 2. each shard runs its own copies and takes its settings; 3. each destination grows to fit
        its incoming parents, receives the stages (one peer copy, ordered after the export with an event) and imports
        them.  An error closes every shard."""
        self._check_open()
        par, thr, gi, energies = reassign_parameters(parents, self._rec_of, self._thr, self._gi, self._energies,
                                                     match_threshold, global_inhibition, inject_energy)
        try:
            self._reassign(par, thr, gi, energies)
        except BaseException:
            self.close()
            raise

    def _reassign(self, par, thr, gi, energies):
        local, cross = plan_agent_moves(par, self._split)
        staged = []
        for s, t, src, dst in cross:                   # 1. every cross parent as it is before the call
            with torch.cuda.device(self._devs[s]):
                stage, em_stage, host = self._shards[s]._export_agents(src)
                done = torch.cuda.Event()
                done.record(torch.cuda.current_stream())
            staged.append((s, t, dst, stage, em_stage, host, done))

        for i, sh in enumerate(self._shards):          # 2. each shard's own copies and settings
            a = self._split[i][0]
            p = np.arange(len(a))
            p[local[i][0]] = local[i][1]
            with torch.cuda.device(self._devs[i]):
                sh._reassign(p, local[i][0], thr[a], gi[a], [energies[b] for b in a])
        for s, t, dst, stage, em_stage, host, done in staged:     # 3. grow, copy across, import
            sh, d = self._shards[t], self._devs[t]
            with torch.cuda.device(d):
                sh._fit_agents(host)
                cur = torch.cuda.current_stream()
                cur.wait_event(done)
                there = [self._to_device(x, d, self._devs[s], cur) for x in (stage, em_stage)]
                sh._import_agents(dst, there[0], there[1], host)
        for d in sorted(set(self._devs)):
            torch.cuda.synchronize(d)
        self._thr, self._gi, self._energies = thr, gi, list(energies)

    @staticmethod
    def _to_device(stage, dst_dev, src_dev, stream):
        """The stage on ``dst_dev``: one prs_stage_copy (a peer copy between devices) on ``stream``."""
        if stage is None:
            return None
        out = torch.empty_like(stage, device=torch.device("cuda", dst_dev))
        nat.check(nat.lib().prs_stage_copy(out.data_ptr(), dst_dev, stage.data_ptr(), src_dev, stage.numel(),
                                           ctypes.c_void_p(stream.cuda_stream)), "prs_stage_copy")
        return out

    # ------------------------------------------------------------------ what the agents hold
    def _gather(self, name):
        self._require_shards()
        v = np.zeros(self.B, np.int64)
        for (a, _), sh in zip(self._split, self._shards):
            v[a] = getattr(sh, name)
        return v

    def _require_shards(self):
        if len(self._shards) != len(self._devs):
            raise RuntimeError("EnsembleSession: the session is closed")

    @property
    def match_threshold(self):
        """float64 [B]: every agent's match threshold in force, in the caller's order."""
        return self._thr.copy()

    @property
    def global_inhibition(self):
        """float64 [B]: every agent's global inhibition in force, in the caller's order."""
        return self._gi.copy()

    @property
    def inject_energy(self):
        """list of B energies (None = no injection) in force, in the caller's order."""
        return list(self._energies)

    @property
    def n_templates(self):
        """int64 [B]: templates in each agent's library."""
        return self._gather("n_templates")

    @property
    def n_experiences(self):
        """int64 [B]: experiences in each agent's map so far (0 without ``experience_map``)."""
        return self._gather("n_experiences")

    @property
    def n_loop_closures(self):
        """int64 [B]: loop closures of each agent's linked map (0 without one)."""
        return self._gather("n_loop_closures")

    @property
    def agents(self):
        """``ShardedAgents``, in the caller's agent order (the libraries as they are now)."""
        self._require_shards()
        if any(sh._ens is None for sh in self._shards):
            raise RuntimeError("EnsembleSession: the session is closed")
        return ShardedAgents([sh.agents for sh in self._shards], self._shard_of, self._local_of, self.n_templates,
                             self.pose_size)

    @property
    def maps(self):
        """``ShardedMaps`` of the linked device maps, in the caller's agent order; None without them."""
        self._require_shards()
        parts = [sh.maps for sh in self._shards]
        if any(p is None for p in parts):
            return None
        return ShardedMaps(parts, self._split, self._shard_of, self._local_of)

    def close(self):
        """Close every shard; a closed session's ``feed`` raises ``RuntimeError``.  What ``agents`` and ``maps``
        returned before stays readable."""
        for sh in self._shards:
            sh.close()
        self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def replay_ensemble(frames, odom, n_agents=None, match_threshold=MATCH_THRESHOLD, global_inhibition=PC_GLOBAL_INHIB,
                    inject_energy=None, pose_size=POSE_SIZE, dtype=np.float32, active_set=0, experience_map=False,
                    experience_links=False, mode="ref", recording=0, activity_threshold=None, max_active_cells=128,
                    devices=None):
    """Replay ``frames[T,256,256]`` (uint8) and ``odom[T,2]`` = (linear.x, angular.z) through B agents.

    ``match_threshold``, ``global_inhibition`` and ``inject_energy`` (None = no injection, else a finite energy >= 0)
    are scalars or length-B sequences.  Every agent starts as ``RatslamRos`` does: energy 1 at the grid's midpoint,
    an empty library.  Returns a dict with ``template [B,T]``, ``created [B,T]``, ``score [B,T]`` (int64: the best score
    each match was made with, -1 where nothing was compared -- an empty library, past the agent's ``length``),
    ``argmax [B,T,3]`` (the cell each match was made with), ``n_templates [B]`` and ``agents`` (``EnsembleAgents``); with
    ``experience_map=True`` also ``n_exp [B,T]`` and ``em_xy [B,T,2]``, replayed on the host from the records as
    ``RatslamRos.replay_native`` does (O(B*T) Python, off by default).  A pose-cell error raises what
    ``replay(native=True)`` raises (``KeyError((5, 5))`` for the reference's LUT hole, ``ValueError`` for an oversize
    shift) for the first offending frame, which the shared odometry makes the same frame for every agent.

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
    arrays ``recording`` can only be 0.

    ``activity_threshold`` (None: off, else a finite number) captures every agent's pose-cell activity at each frame
    on the device, from the state the frame's match was made with -- after its update, before its injection, the state
    ``argmax`` describes: the cells with a value above the threshold (compared in double, 0.002 is what the viewers
    draw) in C order [x][y][th], at most ``max_active_cells`` of them (an integer in [0, X*Y*Th], 0 for counts only;
    the first ones, as ``PoseCellNetwork.active_cells(max_cells=...)`` keeps), and their true count.  The result then
    holds ``activity_count [B, T]`` (-1 past the agent's length), ``activity_ptr [B * T + 1]`` (row pointers over the
    (agent, frame) pairs, row-major), ``activity_cell int64 [n, 3]`` and ``activity_value float64 [n]``;
    ``activity_entry(out, b, t)`` returns one entry as ``(index, value)``.  Off by default; off, nothing changes.

    This is one ``EnsembleSession`` fed once, with libraries reserved for every frame up front; a session fed in
    pieces replays recordings that do not fit in host memory, or longer than 65535 frames.

    ``devices`` (None: the current device) is a sequence of CUDA device indices to split the agents over: one
    ``ShardedEnsembleSession`` fed once, with the same result; ``agents`` and ``maps`` are then its ``ShardedAgents``
    and ``ShardedMaps``."""
    if not (isinstance(experience_map, (bool, np.bool_))
            or (isinstance(experience_map, str) and experience_map == "device")):
        raise ValueError("experience_map must be False, True or 'device', got %r" % (experience_map,))
    devices = None if devices is None else _device_list(devices)
    several = isinstance(frames, (list, tuple)) and (len(frames) == 0 or np.ndim(frames[0]) == 3)
    if several:
        R = len(frames)
        if not isinstance(odom, (list, tuple)) or len(odom) != R or R == 0:
            raise ValueError("replay_ensemble: frames and odom must be lists of the same, non-zero number of "
                             "recordings, got %d and %s"
                             % (R, len(odom) if isinstance(odom, (list, tuple)) else type(odom).__name__))
        fr, od = [], []
        for r in range(R):
            f, o = np.asarray(frames[r]), np.asarray(odom[r], dtype=np.float64)
            if f.dtype != np.uint8 or f.ndim != 3 or tuple(f.shape[1:]) != IM_SIZE or o.shape != (len(f), 2):
                raise ValueError("replay_ensemble: recording %d: frames must be uint8 [T,%d,%d] and odom [T,2], got %s "
                                 "%r and %r" % (r, IM_SIZE[0], IM_SIZE[1], f.dtype, f.shape, o.shape))
            fr.append(f)
            od.append(o)
    else:
        f, o = np.asarray(frames), np.asarray(odom, dtype=np.float64)
        if f.dtype != np.uint8 or f.ndim != 3 or tuple(f.shape[1:]) != IM_SIZE or o.shape != (len(f), 2):
            raise ValueError("replay_ensemble: frames must be uint8 [T,%d,%d] and odom [T,2], got %s %r and %r"
                             % (IM_SIZE[0], IM_SIZE[1], f.dtype, f.shape, o.shape))
        fr, od = [f], [o]
    R = len(fr)
    T = max(len(f) for f in fr)
    if capacity_for(T) > MAX_CAPACITY:
        raise ValueError("replay_ensemble: %d frames need %d templates per agent; the library sweep takes at most %d"
                         % (T, capacity_for(T), MAX_CAPACITY))
    out, rec_of = _replay_once("replay_ensemble", _frame_ticks(fr, od), n_agents, recording, match_threshold,
                               global_inhibition, inject_energy, pose_size, dtype, active_set,
                               "device" if experience_map == "device" else False, experience_links, mode,
                               activity_threshold, max_active_cells, devices)
    if isinstance(experience_map, (bool, np.bool_)) and experience_map:
        moved, tw = np.zeros((T, R), np.uint8), np.zeros((T, R, 2))
        for r in range(R):
            moved[:len(fr[r]), r], tw[:len(fr[r]), r] = xens.gate(od[r])
        pose_size = tuple(int(s) for s in pose_size)
        if several:
            out["n_exp"], out["em_xy"] = _experience_maps(out, moved, tw, pose_size, experience_links, rec_of)
            past = np.arange(T)[None, :] >= out["length"][:, None]
            out["n_exp"][past] = -1
            out["em_xy"][past] = np.nan
        else:
            out["n_exp"], out["em_xy"] = _experience_maps(out, moved[:, 0], tw[:, 0], pose_size, experience_links)
    if not several:
        del out["length"]
    return out


def replay_ensemble_events(events, n_agents=None, match_threshold=MATCH_THRESHOLD, global_inhibition=PC_GLOBAL_INHIB,
                           inject_energy=None, pose_size=POSE_SIZE, dtype=np.float32, active_set=0, experience_map=False,
                           experience_links=False, mode="ref", recording=0, activity_threshold=None,
                           max_active_cells=128, devices=None):
    """``replay_ensemble`` over message streams (``rosbag_io.read_events``) instead of paired frames and twists: agent b
    is the node's message loop, ``ros_simulate.replay_events(events, match_threshold=..., inject_energy=...,
    experience_links=...)`` with ``pcn.global_inhibition`` set to its own value, so every gated odometry message is its
    own pose-cell update and experience-map update.  ``events`` is one stream, or a list of R streams with
    ``recording`` naming each agent's.  The parameters and their validation are ``replay_ensemble``'s;
    ``experience_map`` is False or "device" (the host maps, True, are refused).  Returns what
    ``EnsembleSession.feed_events`` returns -- per image ``template``, ``created``, ``score``, ``argmax``
    ``[B, i_max]`` and ``length [B]``, the maps' ``n_exp``, ``exp_id``, ``em_xy`` and ``n_loop_closures`` -- plus
    ``agents`` and, with ``experience_map="device"``, ``maps``.  On a stream in which odometry and images alternate it equals
    ``replay_ensemble`` on ``rosbag_io.events_to_arrays(events)[:2]``.  The activity capture (``activity_threshold``,
    ``max_active_cells``) is ``replay_ensemble``'s, per image: odometry-only ticks capture nothing (there is no
    per-update capture of message streams).  This is one ``EnsembleSession`` fed once; ``devices`` splits the agents
    over several devices as ``replay_ensemble``'s does."""
    if not (isinstance(experience_map, (bool, np.bool_)) and not experience_map
            or (isinstance(experience_map, str) and experience_map == "device")):
        raise ValueError("replay_ensemble_events: experience_map must be False or 'device' (the host maps need the "
                         "paired frames of replay_ensemble), got %r" % (experience_map,))
    devices = None if devices is None else _device_list(devices)
    several = (isinstance(events, (list, tuple)) and len(events) > 0 and not _is_event(events[0]))
    streams = [event_ticks(st) for st in events] if several else [event_ticks(events)]
    return _replay_once("replay_ensemble_events", streams, n_agents, recording, match_threshold, global_inhibition,
                        inject_energy, pose_size, dtype, active_set, experience_map, experience_links, mode,
                        activity_threshold, max_active_cells, devices)[0]


def _replay_once(who, streams, n_agents, recording, match_threshold, global_inhibition, inject_energy, pose_size,
                 dtype, active_set, experience_map, experience_links, mode, activity_threshold=None, max_active_cells=128,
                 devices=None):
    """``replay_ensemble`` and ``replay_ensemble_events`` after their inputs are validated: the agents' parameters and
    recordings are broadcast and validated and the device memory is checked before any other CUDA call, then one
    ``EnsembleSession`` with libraries for every image is fed the R tick streams once -- a ``ShardedEnsembleSession``
    over ``devices`` when given, with the memory checked per physical device.  Returns the feed's result with
    ``agents`` (and ``maps`` for ``experience_map="device"``), and the agents' recordings."""
    B, thr, gi, energies = agent_parameters(n_agents if n_agents is not None else _recording_count(recording),
                                            match_threshold, global_inhibition, inject_energy)
    if mode != "ref":
        raise ValueError("%s supports the reference matching mode only, got mode=%r" % (who, mode))
    R = len(streams)
    rec_of = agent_recordings(recording, B, R)
    pose_size = tuple(int(s) for s in pose_size)
    act_thr, act_k = activity_parameters(activity_threshold, max_active_cells, pose_size)
    np_dtype = _as_np_dtype(dtype)
    K = max(len(st[2]) for st in streams)
    img = np.zeros((K, R), np.bool_)
    for r, st in enumerate(streams):
        img[:len(st[3]), r] = st[3]
    cap = min(capacity_for(int(img.any(axis=1).sum())), MAX_CAPACITY)
    linked = experience_map == "device" and experience_links
    if devices is not None:
        if len(devices) > B:
            raise ValueError("devices: %d shards for %d agents; a shard holds at least one agent" % (len(devices), B))
        nat.require_cuda()
        _check_devices(devices)
        need = {}
        for d, (a, recs) in zip(devices, _split(rec_of, len(devices))):
            need[d] = need.get(d, 0) + _session_bytes(len(a), len(recs), cap, K, pose_size, np_dtype, linked,
                                                      None if act_thr is None else act_k)
        for d in sorted(need):
            free, _ = torch.cuda.mem_get_info(torch.device("cuda", d))
            if need[d] > free:
                raise ValueError("%s: the agents on cuda:%d need %.2f GB of device memory (%d templates each), "
                                 "%.2f GB are free" % (who, d, need[d] / 1e9, cap, free / 1e9))
        session = ShardedEnsembleSession(devices, B, thr, gi, energies, pose_size, np_dtype, active_set, experience_map,
                                         experience_links, R, rec_of, cap, act_thr, act_k)
        try:
            out = session._feed_ticks(streams)
            out["agents"] = session.agents
            if experience_map == "device":
                out["maps"] = session.maps
        finally:
            session.close()
        return out, rec_of
    need = _session_bytes(B, R, cap, K, pose_size, np_dtype, linked, None if act_thr is None else act_k)
    nat.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device())
    free, _ = torch.cuda.mem_get_info(dev)
    if need > free:
        raise ValueError("%s: %d agents x %d templates need %.2f GB of device memory, %.2f GB are free"
                         % (who, B, cap, need / 1e9, free / 1e9))
    session = EnsembleSession(B, thr, gi, energies, pose_size, np_dtype, active_set, experience_map, experience_links,
                              R, rec_of, cap, act_thr, act_k)
    try:
        out = session._feed_ticks(streams)
        out["agents"] = session.agents
        if experience_map == "device":
            out["maps"] = session.maps
    finally:
        session.close()
    return out, rec_of


def _session_bytes(B, R, cap, K, pose_size, np_dtype, linked, act_k):
    """Device bytes an ``EnsembleSession`` of B agents and R recordings allocates for a replay of K ticks with
    libraries of ``cap`` templates (``act_k`` None: no activity capture)."""
    # per agent its library, template locations, network, the network's snapshot of a mixed tick (R > 1 only), a chunk
    # of records and a few scalars; one chunk of every recording's images
    frame_bytes = IM_SIZE[0] * IM_SIZE[1]
    chunk = _ens_chunk(R, frame_bytes)
    net_bytes = int(np.prod(pose_size)) * np.dtype(np_dtype).itemsize
    need = (B * ((cap // 32) * 34816 + cap * 8 + (2 if R > 1 else 1) * net_bytes + chunk * 32 + 128)
            + R * chunk * frame_bytes)
    if linked:
        need += xens.work_bytes(B, K, cap) + xens.record_bytes(B, K)
    if act_k is not None:       # the capture's counts, slots and packed cells of one chunk (prs_ens_activity_bytes)
        rows = chunk * B
        need += rows * 4 + 2 * rows * act_k * (4 + np.dtype(np_dtype).itemsize) + (rows + 1) * 8 + 6 * 256
    return need


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


def _list(text, parse):
    return [parse(v.strip()) for v in text.split(",") if v.strip()]


def _chunk_arg(text):
    import argparse
    try:
        n = int(text)
    except ValueError:
        n = 0
    if n < 1:
        raise argparse.ArgumentTypeError("--chunk takes a number of frames >= 1, got %r" % (text,))
    return n


def _activity_stats(out, acc):
    """``--activity-threshold``: one result's active-cell counts added to ``acc`` = per agent (sum, images, max)."""
    if acc is None:
        return
    c = out["activity_count"]
    live = c >= 0
    acc[0] += np.where(live, c, 0).sum(axis=1)
    acc[1] += live.sum(axis=1)
    if c.shape[1]:
        np.maximum(acc[2], c.max(axis=1), out=acc[2])


def _session(devices, **kw):
    """An ``EnsembleSession``, or a ``ShardedEnsembleSession`` over ``devices``."""
    return EnsembleSession(**kw) if devices is None else ShardedEnsembleSession(devices, **kw)


def _replay_chunked(bags, chunk, image_topic, odom_topic, recording, acc=None, devices=None, **kw):
    """The bags fed through one ``EnsembleSession`` ``chunk`` frames per bag at a time: per agent the templates, the
    frames created on, its bag's frame count and final arg-max (None for an empty bag), and the session's maps."""
    from . import rosbag_io as rb
    R = len(bags)
    its = [rb.iter_frames(bag, chunk, image_topic=image_topic, odom_topic=odom_topic) for bag in bags]
    s = _session(devices, n_recordings=R, recording=recording if R > 1 else 0, capacity=capacity_for(chunk), **kw)
    try:
        B = len(s.n_templates)
        created = np.zeros(B, np.int64)
        last = [None] * B
        while True:
            pieces = [next(it, None) for it in its]
            if all(p is None for p in pieces):
                break
            fr = [p[0] if p is not None else np.zeros((0,) + IM_SIZE, np.uint8) for p in pieces]
            od = [p[1] if p is not None else np.zeros((0, 2)) for p in pieces]
            out = s.feed(fr if R > 1 else fr[0], od if R > 1 else od[0])
            created += out["created"].sum(axis=1)
            _activity_stats(out, acc)
            for b in range(B):
                if out["length"][b]:
                    last[b] = tuple(int(c) for c in out["argmax"][b, out["length"][b] - 1])
        return s.n_templates, created, s.frames_fed, last, s.maps
    finally:
        s.close()


def _replay_all_messages(bags, chunk, image_topic, odom_topic, recording, acc=None, devices=None, **kw):
    """``--all-messages``: the bags' message streams fed through one ``EnsembleSession`` with ``feed_events``, ``chunk``
    images per bag at a time (each bag whole without it): per agent the templates, the images created on, its bag's
    image count and final arg-max, and the experience and loop-closure counts of its map."""
    from . import rosbag_io as rb
    R = len(bags)
    if chunk is None:
        its = [iter([rb.read_events(bag, image_topic=image_topic, odom_topic=odom_topic)]) for bag in bags]
    else:
        its = [rb.iter_events(bag, chunk, image_topic=image_topic, odom_topic=odom_topic) for bag in bags]
    s = _session(devices, n_recordings=R, recording=recording if R > 1 else 0,
                 capacity=capacity_for(chunk) if chunk is not None else None, **kw)
    try:
        B = len(s.n_templates)
        created = np.zeros(B, np.int64)
        last = [None] * B
        while True:
            pieces = [next(it, None) for it in its]
            if all(p is None for p in pieces):
                break
            ev = [p if p is not None else [] for p in pieces]
            out = s.feed_events(ev if R > 1 else ev[0])
            created += out["created"].sum(axis=1)
            _activity_stats(out, acc)
            for b in range(B):
                if out["length"][b]:
                    last[b] = tuple(int(c) for c in out["argmax"][b, out["length"][b] - 1])
        return s.n_templates, created, s.frames_fed, last, s.n_experiences, s.n_loop_closures
    finally:
        s.close()


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
    ap.add_argument("--chunk", type=_chunk_arg, metavar="FRAMES",
                    help="feed the bags through one session this many frames per bag at a time, decoding only those "
                         "frames (the output is the same as without it); with --all-messages, this many images")
    ap.add_argument("--all-messages", action="store_true",
                    help="replay every odometry message as its own pose-cell update, as the node's message loop does "
                         "(ros_simulate), instead of pairing each image with the last twist before it; also prints "
                         "every agent's experience count")
    ap.add_argument("--activity-threshold", type=float, metavar="T",
                    help="capture every agent's pose cells above T at each image on the device (0.002 is what the "
                         "viewers draw) and print each agent's mean and max active-cell count; only the counts come "
                         "back from the device")
    ap.add_argument("--devices", metavar="D1,D2,...",
                    help="split the agents over these CUDA devices (ShardedEnsembleSession); the output is the same")
    a = ap.parse_args(argv)
    from . import rosbag_io as rb
    thr = _list(a.match_threshold, float)
    gis = _list(a.global_inhibition, float)
    ens = _list(a.inject_energy, lambda s: None if s.lower() == "none" else float(s))
    combos = list(itertools.product(thr, gis, ens))
    several = len(a.bag) > 1
    agents = list(itertools.product(range(len(a.bag)), combos))     # bag-major
    kw = dict(n_agents=len(agents), match_threshold=[c[0] for _, c in agents],
              global_inhibition=[c[1] for _, c in agents], inject_energy=[c[2] for _, c in agents],
              experience_map="device" if a.experience_links or a.all_messages else False,
              experience_links=a.experience_links)
    acc, extra = None, {}
    if a.devices is not None:
        kw["devices"] = _list(a.devices, int)
    if a.activity_threshold is not None:
        kw.update(activity_threshold=a.activity_threshold, max_active_cells=0)
        acc = [np.zeros(len(agents), np.int64), np.zeros(len(agents), np.int64), np.full(len(agents), -1, np.int64)]
        extra = {"acc": acc}
    n_exp = None
    if a.all_messages:
        n_templates, created, fed, last, n_exp, loops = _replay_all_messages(a.bag, a.chunk, a.image_topic,
                                                                             a.odom_topic, [r for r, _ in agents], **kw,
                                                                             **extra)
        frames = [int(fed[r if several else 0]) for r, _ in agents]
    elif a.chunk is not None:
        n_templates, created, fed, last, maps = _replay_chunked(a.bag, a.chunk, a.image_topic, a.odom_topic,
                                                                [r for r, _ in agents], **kw, **extra)
        frames = [int(fed[r if several else 0]) for r, _ in agents]
        loops = maps.n_loop_closures if maps is not None else None
    else:
        recs = [rb.events_to_arrays(rb.read_events(bag, image_topic=a.image_topic, odom_topic=a.odom_topic))[:2]
                for bag in a.bag]
        if several:
            out = replay_ensemble([f for f, _ in recs], [o for _, o in recs], recording=[r for r, _ in agents], **kw)
        else:
            out = replay_ensemble(recs[0][0], recs[0][1], **kw)
        n_templates, maps, loops = out["n_templates"], out.get("maps"), out.get("n_loop_closures")
        _activity_stats(out, acc)
        frames = [len(recs[r][0]) for r, _ in agents]
        created = [int(out["created"][b].sum()) for b in range(len(agents))]
        last = [tuple(int(c) for c in out["argmax"][b, T - 1]) if T else None for b, T in enumerate(frames)]
    for b, (r, (t, g, e)) in enumerate(agents):
        line = ("agent %d  match_threshold %g  global_inhibition %g  inject_energy %s:  templates %d  created %d/%d  "
                "final arg-max %s" % (b, t, g, "none" if e is None else "%g" % e, n_templates[b],
                                      int(created[b]), frames[b], last[b]))
        if several:
            line = "bag %s  %s" % (a.bag[r], line)
        if n_exp is not None:
            line += "  experiences %d" % n_exp[b]
            if a.experience_links:
                line += "  loop closures %d" % loops[b]
        elif a.experience_links:
            line += "  experiences %d  loop closures %d" % (maps.n_experiences[b], loops[b])
        if acc is not None:
            line += "  active cells mean %.1f max %d" % (acc[0][b] / max(int(acc[1][b]), 1), max(int(acc[2][b]), 0))
        print(line)


if __name__ == "__main__":
    main()
