"""Offline replay of the ROS node's update loop (``ratslam/ros_simulate.py``) on the GPU path.

ROS itself (rospy, cv_bridge, rosbag) is transport and out of scope; what is kept is what the node
computes per message (``ros_simulate.py:52-57,67-70,98-105,125-137,152-166``):

* odometry twist ``(linear.x, angular.z)``: dropped unless one component exceeds 0.001 in magnitude,
  else ``vtrans = linear.x / 10``, ``vrot = angular.z / 10`` -> ``PoseCellNetwork.update`` ->
  ``ExperienceMap.update`` with the arg-max cell;
* camera frame (mono8, 256x256): ``ViewTemplates.match`` with the current arg-max cell -> template index.

The live node interleaves these on two threads; the replay fixes the order per time step as
odometry first, then the frame (the same order the oracle's ``replay_run`` uses).
"""
from __future__ import annotations

import math
import ctypes
from collections import deque

import numpy as np
import torch

from . import _native as nat

from .experience_map import ExperienceMap
from .posecell_network import PoseCellNetwork
from .view_templates import ViewTemplates

POSE_SIZE = (21, 21, 36)
IM_SIZE = (256, 256)
X_RANGE = (32, 96)
Y_RANGE = (32, 96)
X_STEP = 2
Y_STEP = 2
MATCH_THRESHOLD = 45000
ODOM_FREQ = 10


def key_scores(key):
    """int64 scores of packed ``(score << 32 | index)`` record keys, -1 where the key is ``UINT64_MAX`` (nothing was
    compared: an empty library, or no frame)."""
    k = np.asarray(key, dtype=np.uint64)
    return np.where(k == np.uint64(0xFFFFFFFFFFFFFFFF), -1, (k >> np.uint64(32)).astype(np.int64))


class RatslamRos(object):
    """The node's state and callbacks, fed from arrays instead of ROS topics."""

    def __init__(self, pose_size=POSE_SIZE, match_threshold=MATCH_THRESHOLD, inject_energy=None,
                 experience_links=False, **pcn_kwargs):
        # inject_energy: enable the view-template -> pose-cell coupling the reference left commented out
        # (ros_simulate.py:106-108): pcn.inject(energy, template_match.location()) after every match
        self.inject_energy = inject_energy
        self.im_count = 0
        self.pcn = PoseCellNetwork(shape=pose_size, **pcn_kwargs)
        self.pc_count = 0
        self.twist_data = deque()
        self.odom_freq = ODOM_FREQ
        midpoint = (math.floor(pose_size[0] / 2), math.floor(pose_size[1] / 2), math.floor(pose_size[2] / 2))
        self.pcn.inject(1, midpoint)
        self.vts = ViewTemplates(x_range=X_RANGE, y_range=Y_RANGE, x_step=X_STEP, y_step=Y_STEP,
                                 im_x=IM_SIZE[0], im_y=IM_SIZE[1], match_threshold=match_threshold)
        self.vt_count = 0
        # experience_links: link the experiences and close loops on (view template, pose cell) revisits -- the
        # reference's TODOs (experience_map.py:49,59); off by default = the reference's dead reckoning
        self.em = ExperienceMap(linked=experience_links, pc_dims=pose_size)
        self.em_count = 0
        self.published_index = []
        self.published_pose = []

    # ros_simulate.py:98-105 (image already decoded to a uint8 array)
    def vis_callback(self, im):
        pc_max = self.pcn.get_pc_max()
        n0 = len(self.vts.templates)
        tm = self.vts.match(input=im, pc_x=pc_max[0], pc_y=pc_max[1], pc_th=pc_max[2])
        index = tm.get_index()
        if self.inject_energy is not None:
            self.pcn.inject(self.inject_energy, tm.location())                              # :106-108
        self.published_index.append(index)
        return index, len(self.vts.templates) > n0

    # ros_simulate.py:125-129 (twist as a (linear.x, angular.z) pair)
    def odom_callback(self, twist):
        if abs(twist[0]) > 0.001 or abs(twist[1]) > 0.001:
            self.twist_data.append(twist)

    _NO_VT = object()

    def _em_update(self, vtrans, vrot, pc_max, vt=_NO_VT):
        """``ExperienceMap.update`` (ros_simulate.py:136-137); with experience_links the most recent template match
        rides along as the view the experience is tagged with."""
        if vt is self._NO_VT:
            vt = self.published_index[-1] if self.published_index else None
        self.em.update(vtrans, vrot, pc_max, vt if self.em.linked else None)

    # ros_simulate.py:134-146
    def update_posecells(self, vtrans, vrot):
        pc_max = self.pcn.update((vtrans, vrot))
        self._em_update(vtrans, vrot, pc_max)
        self.published_pose.append(self.em.get_current_point())

    # ------------------------------------------------------------------ fused fast path
    # One odometry update + one frame match per call with a single host synchronisation
    # (prs_frame_host): the create-or-match decision and the library append happen on the device.
    def _fused_setup(self):
        e, v = self.pcn._ens, self.vts
        dev = e.device
        self._f_scratch = torch.zeros(int(nat.lib().prs_frame_scratch_bytes()), dtype=torch.uint8, device=dev)
        self._f_pcwork = torch.zeros(3, dtype=torch.int64, device=dev)
        self._f_frame = torch.zeros((v.im_x, v.im_y), dtype=torch.uint8).pin_memory()
        self._f_odom = torch.zeros(2, dtype=torch.float64).pin_memory()
        self._f_res = torch.zeros(32, dtype=torch.uint8).pin_memory()
        self._f_result = nat.FrameResult.from_address(self._f_res.data_ptr())
        with torch.cuda.device(dev):
            nat.check(nat.lib().prs_pc_argmax(e._h, e._state.data_ptr(), self._f_pcwork.data_ptr(), nat.stream_ptr()),
                      "prs_pc_argmax")
        v._ensure_lib(torch.uint8)
        self._f_stream = torch.cuda.Stream(device=dev)
        self._f_plan = ctypes.c_void_p()
        self._f_plan_key = None
        self._f_inj = self._NO_INJECT    # the injection setting of _f_plan
        self._f_gen = e._state_gen       # the pose-cell state the cached arg-max (_f_pcwork) was computed from
        self._f_n_dev = None             # the template count the plans' device-side counter holds
        torch.cuda.current_stream(dev).synchronize()
        self._fused_ready = True

    def _fused_resync(self, plan):
        """Bring the device-side caches of the frame plans back in step with what happened OUTSIDE them: a pose-cell
        update / inject / assignment since the last fused frame invalidates the cached arg-max (it is recomputed on
        the frame stream, behind whatever the current stream still has queued), templates appended by
        ``vts.match`` / ``create`` invalidate the device-side library size and the rows of the device-side location
        table that the injection node reads."""
        e, v = self.pcn._ens, self.vts
        if e._state_gen != self._f_gen:
            self._f_stream.wait_stream(torch.cuda.current_stream(e.device))
            with torch.cuda.device(e.device):
                nat.check(nat.lib().prs_pc_argmax(e._h, e._state.data_ptr(), self._f_pcwork.data_ptr(),
                                                  ctypes.c_void_p(self._f_stream.cuda_stream)), "prs_pc_argmax")
            self._f_gen = e._state_gen
        if self._f_n_dev is not None and self._f_n_dev != v._n:
            self._f_stream.wait_stream(torch.cuda.current_stream(e.device))
            nat.check(nat.lib().prs_frame_set_count(plan, v._n, ctypes.c_void_p(self._f_stream.cuda_stream)),
                      "prs_frame_set_count")
        self._f_n_dev = v._n
        v._cell_sync(self._f_stream)

    # ------------------------------------------------------------------ injection inside the frame
    _NO_INJECT = (None, None)

    def _device_energy(self, strict=False):
        """The energy the frame plans inject on the device (``prs_frame_set_inject``), None for no injection there.
        The device node takes finite energies >= 0; another energy is injected by the host behind the frame
        (``fused_frame``) or, ``strict``, refused (the pipelined and native replays)."""
        en = self.inject_energy
        if en is None:
            return None
        en = float(en)
        if en >= 0 and math.isfinite(en):
            return en
        if strict:
            raise ValueError("the pipelined and native replays inject on the device, which takes finite energies "
                             ">= 0; got inject_energy=%r" % (self.inject_energy,))
        return None

    def _plan_inject(self, plan, current, energy):
        """Point ``plan``'s injection node at ``energy`` and the library's location table (None: no node).  Returns
        the setting, which the caller keeps beside the plan to skip the call while nothing changes."""
        want = self._NO_INJECT if energy is None else (energy, self.vts._cell_table(self.pcn.shape).data_ptr())
        if want != current:
            nat.check(nat.lib().prs_frame_set_inject(plan, 0.0 if energy is None else energy, want[1]),
                      "prs_frame_set_inject")
        return want

    def _inject_error(self, index):
        loc = self.vts.templates[index].location()
        return IndexError("index %r is out of bounds for shape %r" % (tuple(loc), self.pcn.shape))

    def _fused_plan(self):
        """(Re)create the CUDA-graph frame plan; needed again whenever the library buffer was reallocated."""
        e, v = self.pcn._ens, self.vts
        key = (v._lib.data_ptr(), v._capacity, v.match_threshold)
        if self._f_plan_key == key:
            return
        if self._f_plan:
            nat.lib().prs_frame_destroy(self._f_plan)
            self._f_plan = ctypes.c_void_p()
        torch.cuda.synchronize(e.device)
        nat.check(nat.lib().prs_frame_create(
            e._h, e._state.data_ptr(), e._gi.data_ptr(), self._f_pcwork.data_ptr(), v._lib.data_ptr(), v._n, v._capacity,
            float(v.match_threshold), v.mode, v.im_x, v.im_y, v.y_range[0], v.y_range[1], v.y_step, v.x_range[0],
            v.x_range[1], v.x_step, self._f_scratch.data_ptr(), self._f_odom.data_ptr(), self._f_frame.data_ptr(),
            self._f_res.data_ptr(), ctypes.byref(self._f_plan)), "prs_frame_create")
        self._f_plan_key = key
        self._f_inj = self._NO_INJECT
        self._f_n_dev = v._n

    def __del__(self):
        plans = [getattr(self, "_f_plan", None)] + [sl["plan"] for sl in getattr(self, "_p_slots", [])]
        for p in plans:
            if p:
                try:
                    nat.lib().prs_frame_destroy(p)
                except Exception:
                    pass

    def fused_frame(self, twist, im):
        """``odom_callback(twist)`` + ``spin_once()`` + ``vis_callback(im)`` in one device round trip.

        Returns ``(template_index, created)``.  Same decisions as the three separate calls; a pose-cell
        error (LUT hole, oversize shift) is raised after the frame instead of before it.  With ``inject_energy >= 0``
        the injection at the template's stored cell is the frame's last node on the device; a location outside the
        grid raises ``IndexError`` after the frame, the pose cells untouched."""
        if not getattr(self, "_fused_ready", False):
            self._fused_setup()
        e, v = self.pcn._ens, self.vts
        moved = twist is not None and (abs(twist[0]) > 0.001 or abs(twist[1]) > 0.001)   # ros_simulate.py:128
        vtrans = vrot = 0.0
        if moved:
            vtrans, vrot = twist[0] / self.odom_freq, twist[1] / self.odom_freq          # :157-158
            o = self._f_odom.numpy()
            o[0], o[1] = vtrans, vrot
        v._grow(v._n + 2)
        self._fused_plan()
        energy = self._device_energy()
        self._f_inj = self._plan_inject(self._f_plan, self._f_inj, energy)
        self._fused_resync(self._f_plan)
        self._f_frame.numpy()[...] = im
        nat.check(nat.lib().prs_frame_run(self._f_plan, 1 if moved else 0, ctypes.c_void_p(self._f_stream.cuda_stream)),
                  "prs_frame_run")
        r = self._f_result
        err = int(r.pc_err)
        if moved:
            e._raise_on_err(np.array([err & ~nat.ERR_INJECT_LOC], dtype=np.int32))
        X, Y, Th = self.pcn.shape
        flat = int(r.argmax)
        pc_max = (flat // (Y * Th), (flat // Th) % Y, flat % Th)
        # the record holds the arg-max the match was made with; after an injection the state has moved on
        self.pcn.max_pc, self.pcn._max_valid = pc_max, energy is None
        if moved:
            self._em_update(vtrans, vrot, pc_max)                                          # :136-137
            self.published_pose.append(self.em.get_current_point())
        if r.created:
            v._loc[v._n] = pc_max
        v._n = self._f_n_dev = int(r.n_templates)
        v.last_score = None if r.key == (1 << 64) - 1 else int(r.key >> 32)
        if energy is not None:
            v._cell_n = v._n                 # the created template's row was written on the device
            self._f_gen = e._state_gen       # the node kept the cached arg-max (_f_pcwork) current
            if err & nat.ERR_INJECT_LOC:
                raise self._inject_error(int(r.template_index))
        elif self.inject_energy is not None:  # an energy the device node does not take: the host injects
            loc = tuple(int(c) for c in v._loc[int(r.template_index)])
            with torch.cuda.stream(self._f_stream):
                self.pcn.inject(self.inject_energy, loc)
                with torch.cuda.device(e.device):    # keep the cached arg-max in step with the injected state
                    nat.check(nat.lib().prs_pc_argmax(e._h, e._state.data_ptr(), self._f_pcwork.data_ptr(),
                                                      nat.stream_ptr()), "prs_pc_argmax")
            self._f_stream.synchronize()
        self._f_gen = e._state_gen       # the plan's own update and the injection above are reflected in _f_pcwork
        self.published_index.append(int(r.template_index))
        return int(r.template_index), bool(r.created)

    # ------------------------------------------------------------------ pipelined frames
    # Two frame plans with their own pinned host buffers share the device-side state (pose cells, library,
    # template count) and are launched alternately on one stream: the device runs frame t while the host stages
    # frame t+1 and digests the result of frame t-1.  Same decisions as fused_frame; results arrive one call late.
    def _pipe_setup(self, n_slots=2):
        if not getattr(self, "_fused_ready", False):
            self._fused_setup()
        e, v = self.pcn._ens, self.vts
        self._p_slots = []
        for _ in range(n_slots):
            frame = torch.zeros((v.im_x, v.im_y), dtype=torch.uint8).pin_memory()
            odom = torch.zeros(2, dtype=torch.float64).pin_memory()
            res = torch.zeros(32, dtype=torch.uint8).pin_memory()
            self._p_slots.append({"frame": frame, "frame_np": frame.numpy(), "odom": odom, "odom_np": odom.numpy(),
                                  "res": res, "result": nat.FrameResult.from_address(res.data_ptr()),
                                  "plan": ctypes.c_void_p(), "inj": self._NO_INJECT, "event": torch.cuda.Event(),
                                  "meta": None})
        self._p_key = None
        self._p_inflight = 0

    def _pipe_plans(self):
        e, v = self.pcn._ens, self.vts
        key = (v._lib.data_ptr(), v._capacity, v.match_threshold)
        if self._p_key == key:
            return
        assert self._p_inflight == 0
        torch.cuda.synchronize(e.device)
        for sl in self._p_slots:
            if sl["plan"]:
                nat.lib().prs_frame_destroy(sl["plan"])
                sl["plan"] = ctypes.c_void_p()
            nat.check(nat.lib().prs_frame_create(
                e._h, e._state.data_ptr(), e._gi.data_ptr(), self._f_pcwork.data_ptr(), v._lib.data_ptr(), v._n,
                v._capacity, float(v.match_threshold), v.mode, v.im_x, v.im_y, v.y_range[0], v.y_range[1], v.y_step,
                v.x_range[0], v.x_range[1], v.x_step, self._f_scratch.data_ptr(), sl["odom"].data_ptr(),
                sl["frame"].data_ptr(), sl["res"].data_ptr(), ctypes.byref(sl["plan"])), "prs_frame_create")
            sl["inj"] = self._NO_INJECT
        self._p_key = key
        self._f_n_dev = v._n

    def pipe_submit(self, slot, twist, im):
        """Stage and launch one frame in ``slot`` (0 or 1) without waiting for it; ``pipe_finish(slot)`` returns its
        ``(template_index, created)``.  The previous frame of the same slot must have been finished.  ``inject_energy``
        must be None or a finite energy >= 0 (``ValueError``): the injection is the frame's last node on the device."""
        v = self.vts
        sl = self._p_slots[slot]
        assert sl["meta"] is None, "slot still in flight"
        energy = self._device_energy(strict=True)
        sl["inj"] = self._plan_inject(sl["plan"], sl["inj"], energy)
        if v._n + self._p_inflight + 2 > v._capacity:   # growing reallocates the library: drain, grow, re-plan
            raise RuntimeError("pipe_submit: library full; finish the frames in flight and call pipe_grow()")
        moved = twist is not None and (abs(twist[0]) > 0.001 or abs(twist[1]) > 0.001)   # ros_simulate.py:128
        vtrans = vrot = 0.0
        if moved:
            vtrans, vrot = twist[0] / self.odom_freq, twist[1] / self.odom_freq          # :157-158
            sl["odom_np"][0], sl["odom_np"][1] = vtrans, vrot
        sl["frame_np"][...] = im
        if self._p_inflight == 0:
            self._fused_resync(sl["plan"])
        nat.check(nat.lib().prs_frame_launch(sl["plan"], 1 if moved else 0, ctypes.c_void_p(self._f_stream.cuda_stream)),
                  "prs_frame_launch")
        sl["event"].record(self._f_stream)
        sl["meta"] = (moved, vtrans, vrot, energy is not None)
        self._p_inflight += 1

    def pipe_needs_grow(self):
        return self.vts._n + self._p_inflight + 2 > self.vts._capacity

    def pipe_grow(self):
        assert self._p_inflight == 0
        self.vts._grow(max(self.vts._n + 3, 2 * self.vts._capacity))
        self._pipe_plans()

    def pipe_finish(self, slot):
        e, v = self.pcn._ens, self.vts
        sl = self._p_slots[slot]
        moved, vtrans, vrot, injected = sl["meta"]
        sl["event"].synchronize()
        sl["meta"] = None
        self._p_inflight -= 1
        r = sl["result"]
        err = int(r.pc_err)
        if moved:
            e._raise_on_err(np.array([err & ~nat.ERR_INJECT_LOC], dtype=np.int32))
        X, Y, Th = self.pcn.shape
        flat = int(r.argmax)
        pc_max = (flat // (Y * Th), (flat // Th) % Y, flat % Th)
        self.pcn.max_pc, self.pcn._max_valid = pc_max, self._p_inflight == 0 and not injected
        if moved:
            self._em_update(vtrans, vrot, pc_max)                                          # :136-137
            self.published_pose.append(self.em.get_current_point())
        if r.created:
            v._loc[int(r.n_templates) - 1] = pc_max
        v._n = self._f_n_dev = int(r.n_templates)
        if injected:
            v._cell_n = v._n                 # the created template's row was written on the device
        self._f_gen = e._state_gen
        v.last_score = None if r.key == (1 << 64) - 1 else int(r.key >> 32)
        if injected and err & nat.ERR_INJECT_LOC:
            raise self._inject_error(int(r.template_index))
        self.published_index.append(int(r.template_index))
        return int(r.template_index), bool(r.created)

    # ------------------------------------------------------------------ the loop on the C side
    _RESULT_DTYPE = np.dtype([("argmax", "<i8"), ("key", "<u8"), ("created", "<i4"), ("template_index", "<i4"),
                              ("n_templates", "<i4"), ("pc_err", "<i4")])

    def replay_native(self, frames, odom, n_plans=2):
        """``run``'s loop (ros_simulate.py:152-166) over recorded arrays in ONE library call (``prs_replay_run``):
        staging, graph launches and result collection happen in C with ``n_plans`` frames in flight (two already hide the host); the host-side
        bookkeeping (experience map, template locations) is replayed from the returned records afterwards.
        Returns the structured result array (one ``prs_frame_result`` per frame).  Same decisions as the
        frame-by-frame calls; a pose-cell error is raised for the first offending frame after the batch, and so is the
        ``IndexError`` of a template location outside the grid.  ``inject_energy`` must be None or a finite energy >= 0
        (``ValueError``): the injection is every frame's last node on the device."""
        energy = self._device_energy(strict=True)
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        odom = np.asarray(odom, dtype=np.float64)
        T = len(frames)
        e, v = self.pcn._ens, self.vts
        if frames.ndim != 3 or tuple(frames.shape[1:]) != (v.im_x, v.im_y) or odom.shape != (T, 2):
            raise ValueError("replay_native: frames must be [T,%d,%d] and odom [T,2]" % (v.im_x, v.im_y))
        if getattr(self, "_p_slots", None) is None or len(self._p_slots) != n_plans:
            self._pipe_setup(n_plans)
        assert self._p_inflight == 0
        v._grow(v._n + T + 2)
        self._pipe_plans()
        for sl in self._p_slots:
            sl["inj"] = self._plan_inject(sl["plan"], sl["inj"], energy)
        self._fused_resync(self._p_slots[0]["plan"])
        moved = ((np.abs(odom[:, 0]) > 0.001) | (np.abs(odom[:, 1]) > 0.001)).astype(np.uint8)    # ros_simulate.py:128
        tw = np.ascontiguousarray(odom / float(self.odom_freq))                                    # :157-158
        res = np.zeros(T, dtype=self._RESULT_DTYPE)
        plans = (ctypes.c_void_p * n_plans)(*[sl["plan"].value for sl in self._p_slots])
        nat.check(nat.lib().prs_replay_run(plans, n_plans, frames.ctypes.data, tw.ctypes.data, moved.ctypes.data, T,
                                           res.ctypes.data, ctypes.c_void_p(self._f_stream.cuda_stream)),
                  "prs_replay_run")
        # host bookkeeping, in frame order
        X, Y, Th = self.pcn.shape
        flat = res["argmax"]
        amax = np.stack([flat // (Y * Th), (flat // Th) % Y, flat % Th], axis=1)
        pc_bad = ((res["pc_err"] & ~nat.ERR_INJECT_LOC) != 0) & (moved != 0)
        inj_bad = (res["pc_err"] & nat.ERR_INJECT_LOC) != 0 if energy is not None else np.zeros(T, np.bool_)
        bad = np.nonzero(pc_bad | inj_bad)[0]
        stop = int(bad[0]) if len(bad) else T
        # a pose-cell error stops before its frame, a bad template location after its frame's match (vis_callback order)
        booked = stop + 1 if len(bad) and not pc_bad[stop] else stop
        self._native_n_exp = np.zeros(T, np.int64)       # per-frame experience count / current point, for replay()
        self._native_em_xy = np.zeros((T, 2))
        for t in range(booked):
            pc_max = (int(amax[t, 0]), int(amax[t, 1]), int(amax[t, 2]))
            if moved[t]:
                self._em_update(float(tw[t, 0]), float(tw[t, 1]), pc_max,
                                int(res["template_index"][t - 1]) if t > 0 else None)                 # :136-137
                self.published_pose.append(self.em.get_current_point())
            if res["created"][t]:
                v._loc[int(res["n_templates"][t]) - 1] = pc_max
            self._native_n_exp[t] = len(self.em.experiences)
            if self.em.current_exp is not None:
                self._native_em_xy[t] = self.em.get_current_point()
        self.published_index.extend(int(i) for i in res["template_index"][:stop])
        if T:
            last = T - 1
            v._n = self._f_n_dev = int(res["n_templates"][last])
            if energy is not None:
                v._cell_n = v._n             # the created templates' rows were written on the device
            self._f_gen = e._state_gen
            self.pcn.max_pc = tuple(int(c) for c in amax[last])
            self.pcn._max_valid = energy is None     # the record's arg-max precedes the last frame's injection
            k = int(res["key"][last])
            v.last_score = None if k == (1 << 64) - 1 else k >> 32
        if len(bad):
            if pc_bad[stop]:
                e._raise_on_err(np.array([res["pc_err"][stop] & ~nat.ERR_INJECT_LOC], dtype=np.int32))
            raise self._inject_error(int(res["template_index"][stop]))
        return res

    # ros_simulate.py:152-166, one pass of the loop body
    def spin_once(self):
        if self.twist_data:
            twist = self.twist_data.popleft()
            self.update_posecells(twist[0] / self.odom_freq, twist[1] / self.odom_freq)
            return True
        return False


def replay(frames, odom, fused=False, pipelined=False, native=False, **kwargs):
    """Run the loop over ``frames[T,256,256]`` (uint8) and ``odom[T,2]``; returns per-frame records.

    ``fused=True`` uses ``RatslamRos.fused_frame`` (one device round trip per frame) instead of the three
    reference-shaped calls; ``pipelined=True`` additionally overlaps the host's staging and bookkeeping of
    neighbouring frames with the device work (two alternating frame plans); ``native=True`` runs the whole loop in
    one library call (``prs_replay_run``, two frames in flight) and replays the host bookkeeping from its records.
    The records are identical: ``template``, ``created``, ``argmax [T,3]`` (the cell each match was made with),
    ``score [T]`` (the best score the frame's match was made with, -1 where the library was empty), ``n_exp`` and
    ``em_xy``."""
    node = RatslamRos(**kwargs)
    T = len(frames)
    rec = {"template": np.zeros(T, np.int64), "created": np.zeros(T, np.bool_), "score": np.full(T, -1, np.int64),
           "argmax": np.zeros((T, 3), np.int64), "n_exp": np.zeros(T, np.int64), "em_xy": np.zeros((T, 2))}

    def note_score(t):
        if node.vts.last_score is not None:
            rec["score"][t] = node.vts.last_score

    if native:
        odom = np.asarray(odom, dtype=np.float64)
        res = node.replay_native(frames, odom)
        X, Y, Th = node.pcn.shape
        flat = res["argmax"]
        rec["argmax"] = np.stack([flat // (Y * Th), (flat // Th) % Y, flat % Th], axis=1).astype(np.int64)
        rec["template"] = res["template_index"].astype(np.int64)
        rec["created"] = res["created"] != 0
        rec["score"] = key_scores(res["key"])
        rec["n_exp"], rec["em_xy"] = node._native_n_exp, node._native_em_xy
        rec["n_templates"] = len(node.vts.templates)
        rec["node"] = node
        return rec
    if pipelined:
        node._device_energy(strict=True)
        node._pipe_setup()
        node.vts._grow(64)
        node._pipe_plans()

        def finish(t):
            idx, created = node.pipe_finish(t % 2)
            rec["argmax"][t] = node.pcn.max_pc
            rec["template"][t] = idx
            rec["created"][t] = created
            note_score(t)
            rec["n_exp"][t] = len(node.em.experiences)
            if node.em.current_exp is not None:
                rec["em_xy"][t] = node.em.get_current_point()

        for t in range(T):
            if node.pipe_needs_grow():
                if t >= 1:
                    finish(t - 1)
                node.pipe_grow()
                node.pipe_submit(t % 2, (float(odom[t, 0]), float(odom[t, 1])), frames[t])
                continue
            node.pipe_submit(t % 2, (float(odom[t, 0]), float(odom[t, 1])), frames[t])
            if t >= 1 and node._p_slots[(t - 1) % 2]["meta"] is not None:
                finish(t - 1)
        if T and node._p_slots[(T - 1) % 2]["meta"] is not None:
            finish(T - 1)
        rec["n_templates"] = len(node.vts.templates)
        rec["node"] = node
        return rec
    for t in range(T):
        if fused:
            idx, created = node.fused_frame((float(odom[t, 0]), float(odom[t, 1])), frames[t])
            rec["argmax"][t] = node.pcn.max_pc
        else:
            node.odom_callback((float(odom[t, 0]), float(odom[t, 1])))
            node.spin_once()
            rec["argmax"][t] = node.pcn.get_pc_max()
            idx, created = node.vis_callback(frames[t])
        rec["template"][t] = idx
        rec["created"][t] = created
        note_score(t)
        rec["n_exp"][t] = len(node.em.experiences)
        if node.em.current_exp is not None:
            rec["em_xy"][t] = node.em.get_current_point()
    rec["n_templates"] = len(node.vts.templates)
    rec["node"] = node
    return rec


def replay_events(events, fused=False, record=None, **kwargs):
    """Run the node over a message stream (``rosbag_io.read_events``): ``("odom", stamp, (lin_x, ang_z))`` ->
    ``odom_callback`` + one pass of ``run``'s loop body, ``("image", stamp, frame)`` -> ``vis_callback``, in the
    order given.  ``fused=True`` folds every odometry message that is directly followed by an image into one
    ``fused_frame`` call (same results).  ``record`` = path of a bag to write the node's outputs to, the way
    RECORD_ROSBAG does (``ros_simulate.py:92-95,116-117,147-148``): ``navbot/templatematches`` (std_msgs/Int32)
    and ``navbot/experiencemap`` (geometry_msgs/Pose2D)."""
    from . import rosbag_io as rb
    events = list(events)
    first = next((p for k, _, p in events if k == "image"), None)
    node = RatslamRos(**kwargs)
    if first is not None and tuple(first.shape) != (node.vts.im_x, node.vts.im_y):
        raise ValueError("frames are %r, the view-template mask was built for %r"
                         % (tuple(first.shape), (node.vts.im_x, node.vts.im_y)))
    writer = rb.BagWriter(record) if record else None
    rec = {"template": [], "created": [], "argmax": [], "n_exp": [], "em_xy": [], "image_stamp": []}

    def note_pose(stamp):
        if writer is not None and node.em.current_exp is not None:
            x, y = node.em.get_current_point()
            writer.write(rb.EM_TOPIC, "geometry_msgs/Pose2D", stamp, rb.encode_pose2d(x, y))

    def note_image(stamp, idx, created, pc_max):
        rec["template"].append(idx)
        rec["created"].append(created)
        rec["argmax"].append(tuple(int(c) for c in pc_max))       # the cell the match was made with
        rec["n_exp"].append(len(node.em.experiences))
        rec["em_xy"].append(node.em.get_current_point() if node.em.current_exp is not None else (0.0, 0.0))
        rec["image_stamp"].append(stamp[0] + stamp[1] * 1e-9)
        if writer is not None:
            writer.write(rb.MATCH_TOPIC, "std_msgs/Int32", stamp, rb.encode_int32(idx))

    try:
        i, n = 0, len(events)
        while i < n:
            kind, stamp, payload = events[i]
            if kind == "odom":
                twist = (float(payload[0]), float(payload[1]))
                if fused and i + 1 < n and events[i + 1][0] == "image":
                    _, istamp, frame = events[i + 1]
                    n_pose = len(node.published_pose)
                    idx, created = node.fused_frame(twist, frame)
                    if len(node.published_pose) > n_pose:
                        note_pose(stamp)
                    note_image(istamp, idx, created, node.pcn.max_pc)
                    i += 2
                    continue
                node.odom_callback(twist)
                if node.spin_once():
                    note_pose(stamp)
            elif kind == "image":
                if fused:
                    idx, created = node.fused_frame(None, payload)
                    pc_max = node.pcn.max_pc
                else:
                    pc_max = node.pcn.get_pc_max()
                    idx, created = node.vis_callback(payload)
                note_image(stamp, idx, created, pc_max)
            else:
                raise ValueError("unknown event kind %r" % (kind,))
            i += 1
    finally:
        if writer is not None:
            writer.close()
    out = {k: np.asarray(v) for k, v in rec.items()}
    out["argmax"] = out["argmax"].reshape(-1, 3)
    out["em_xy"] = out["em_xy"].reshape(-1, 2)
    out["n_templates"] = len(node.vts.templates)
    out["node"] = node
    return out


def replay_bag(path, fused=False, record=None, image_topic="navbot/camera/image", odom_topic="navbot/odom", **kwargs):
    """``replay_events`` over a recorded ROS1 bag (topics of ``ros_simulate.py:82-83``)."""
    from . import rosbag_io as rb
    return replay_events(rb.read_events(path, image_topic=image_topic, odom_topic=odom_topic), fused=fused,
                         record=record, **kwargs)


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description="Replay a ROS1 bag through the pose-cell / view-template loop")
    ap.add_argument("bag")
    ap.add_argument("--fused", action="store_true", help="one device round trip per frame")
    ap.add_argument("--inject-energy", type=float, default=None, metavar="E",
                    help="inject E at the matched template's pose cell after every frame (ros_simulate.py:106-108)")
    ap.add_argument("--record", default=None, help="write template matches and experience-map points to this bag")
    ap.add_argument("--npy", default=None, help="also save frames/odom arrays as <prefix>_frames.npy, <prefix>_odom.npy")
    ap.add_argument("--image-topic", default="navbot/camera/image")
    ap.add_argument("--odom-topic", default="navbot/odom")
    a = ap.parse_args(argv)
    from . import rosbag_io as rb
    events = rb.read_events(a.bag, image_topic=a.image_topic, odom_topic=a.odom_topic)
    if a.npy:
        frames, odom, _ = rb.events_to_arrays(events)
        np.save(a.npy + "_frames.npy", frames)
        np.save(a.npy + "_odom.npy", odom)
    out = replay_events(events, fused=a.fused, record=a.record, inject_energy=a.inject_energy)
    print("frames %d  templates %d  experiences %d" % (len(out["template"]), out["n_templates"],
                                                      len(out["node"].em.experiences)))


if __name__ == "__main__":
    main()
