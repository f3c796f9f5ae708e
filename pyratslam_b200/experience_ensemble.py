"""Every agent's experience map of an ensemble replay, built at once.

A parameter sweep (``ros_ensemble.replay_ensemble``) is judged by what each setting does to the map: how many
experiences it creates and how many loops it closes.  ``ensemble_experience_maps`` builds the map of each of B agents
from its records -- the template matched at every frame and the arg-max pose cell -- and the shared odometry:

* linked (``linked=True``): one CUDA thread per agent runs ``ExperienceMap(linked=True).update`` over the frames
  (``prs_em_linked_run``, csrc/experience_map.cu).  Creation, loop-closure and link decisions are bit-identical to the
  host class; positions and link geometry may differ by the ulps of the device's cos, sin, atan2 and hypot.  The maps
  stay on the device; ``EnsembleExperienceMaps`` reads one agent's arrays or rebuilds its host ``ExperienceMap``, which
  relaxes (``iterate``) on the host.
* unlinked (``linked=False``): the reference's map dead-reckons the shared odometry and ignores the records, so every
  agent has the same map.  It is computed once on the host, with the host class itself, and broadcast.

A frame's experience is tagged with the template of the frame before it (none at t = 0), as
``RatslamRos.replay_native`` does; a negative template means the frame matched none.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _native as nat
from .experience_map import ExperienceMap
from .ros_simulate import ODOM_FREQ

EXPERIENCE_DTYPE = np.dtype([("pc_x", np.int64), ("pc_y", np.int64), ("pc_th", np.int64), ("vt", np.int64),
                             ("m_x", np.float64), ("m_y", np.float64), ("th", np.float64)])
LINK_DTYPE = np.dtype([("from", np.int64), ("to", np.int64), ("d", np.float64), ("heading", np.float64),
                       ("facing", np.float64)])

# prs_em_linked_run's workspace (include/pyratslam_b200.h): (name, element type, rows: "T", "N" = templates, or a count)
_WORK = [("exp_x", torch.float64, "T"), ("exp_y", torch.float64, "T"), ("exp_th", torch.float64, "T"),
         ("link_d", torch.float64, "T"), ("link_heading", torch.float64, "T"), ("link_facing", torch.float64, "T"),
         ("rel", torch.float64, 3), ("exp_cell", torch.int64, "T"), ("exp_tag", torch.int32, "T"),
         ("exp_next", torch.int32, "T"), ("out_head", torch.int32, "T"), ("link_from", torch.int32, "T"),
         ("link_to", torch.int32, "T"), ("link_next", torch.int32, "T"), ("vt_head", torch.int32, "N"),
         ("counts", torch.int32, 4)]


def _work_layout(B, T, n_templates):
    """{name: (byte offset, element type, rows)} and the total bytes of the workspace."""
    off, lay = 0, {}
    for name, dt, rows in _WORK:
        rows = {"T": T, "N": n_templates}.get(rows, rows)
        lay[name] = (off, dt, rows)
        off += (rows * B * torch.empty((), dtype=dt).element_size() + 255) // 256 * 256
    return lay, off


def work_bytes(B, T, n_templates):
    """Device bytes of the linked maps' workspace (``prs_em_work_bytes``)."""
    return _work_layout(B, T, n_templates)[1]


def record_bytes(B, T):
    """Device bytes of the uploaded records and the per-frame outputs: int64 cell, int32 tag, int32 n_exp and exp_id,
    double em_xy[2] per agent-frame."""
    return B * T * (8 + 4 + 4 + 4 + 16)


def gate(odom):
    """``(moved uint8[T], tw float64[T,2])``: the 0.001 twist gate (ros_simulate.py:128) and the twist given to
    ``update`` (:157-158), from ``odom[T,2]`` = (linear.x, angular.z)."""
    odom = np.asarray(odom, dtype=np.float64)
    moved = ((np.abs(odom[:, 0]) > 0.001) | (np.abs(odom[:, 1]) > 0.001)).astype(np.uint8)
    return moved, np.ascontiguousarray(odom / float(ODOM_FREQ))


def dead_reckoning(moved, tw, start=None):
    """The reference's unlinked map over the shared odometry, which is every agent's: ``(n_exp int64[T],
    em_xy float64[T,2], accum)`` with accum = the final (accum_delta_x, accum_delta_y, accum_delta_th).  ``start`` =
    ``(n_exp, accum)`` after earlier frames of the same recording continues that map (an experience is created at the
    accumulated position, so the last one sits at accum's (x, y))."""
    T = len(moved)
    em = ExperienceMap()
    n0 = 0
    if start is not None:
        n0, (em.accum_delta_x, em.accum_delta_y, em.accum_delta_th) = int(start[0]), start[1]
    n_exp = np.zeros(T, np.int64)
    em_xy = np.zeros((T, 2))
    for t in range(T):
        if moved[t]:
            em.update(float(tw[t, 0]), float(tw[t, 1]), (0, 0, 0))    # the cell tags the experience, nothing else
        n_exp[t] = n0 + len(em.experiences)
        if em.current_exp is not None:
            em_xy[t] = em.get_current_point()
        elif n0:
            em_xy[t] = (em.accum_delta_x, em.accum_delta_y)
    return n_exp, em_xy, (em.accum_delta_x, em.accum_delta_y, em.accum_delta_th)


class EnsembleExperienceMaps:
    """The B linked maps ``prs_em_linked_run`` left in its device workspace.

    ``n_experiences``, ``n_links``, ``current`` (-1 = none) and ``n_loop_closures`` are int64 [B] on the host; an
    agent's experiences and links are copied from the device when asked for."""

    def __init__(self, work, B, T, n_templates, moved, tw, pose_size, delta_pc, correction, vt_ids=None, rec_of=None,
                 accum=None, cols=None):
        lay, _ = _work_layout(B, T, n_templates)
        self._vt_ids = vt_ids       # per agent: the caller's template id of each tag, when the ids were renumbered
        # cols: the workspace column of each agent, when the workspace holds them in another order (EnsembleSession)
        self._cols = np.arange(B) if cols is None else np.asarray(cols)
        self._v = {k: work[o:o + r * B * torch.empty((), dtype=dt).element_size()].view(dt).view(r, B)
                   for k, (o, dt, r) in lay.items()}
        counts = self._v["counts"].cpu().numpy().astype(np.int64)[:, self._cols]
        self.n_experiences, self.n_links, self.current, self.n_loop_closures = counts
        self._rel = self._v["rel"].cpu().numpy()[:, self._cols]
        # the dead reckoning of each recording (rec_of: agent b's column of moved [T,R], tw [T,R,2]), computed when a map
        # is rebuilt unless ``accum`` ({recording: accum}) gives it
        self._odom, self._rec_of, self._accum = (moved, tw), rec_of, {} if accum is None else dict(accum)
        self.pose_size, self.delta_pc, self.correction = tuple(pose_size), delta_pc, correction

    def __len__(self):
        return len(self.n_experiences)

    def _col(self, name, n, b):
        return self._v[name][:n, int(self._cols[b])].cpu().numpy()

    def experiences(self, b):
        """Agent b's experiences in index order, ``EXPERIENCE_DTYPE`` [n]: cell, view template (-1 = none), position
        and heading."""
        n = int(self.n_experiences[b])
        out = np.zeros(n, EXPERIENCE_DTYPE)
        X, Y, Th = self.pose_size
        cell = self._col("exp_cell", n, b)
        out["pc_x"], out["pc_y"], out["pc_th"] = cell // (Y * Th), cell // Th % Y, cell % Th
        vt = self._col("exp_tag", n, b).astype(np.int64)
        if self._vt_ids is not None:
            vt[vt >= 0] = self._vt_ids[b][vt[vt >= 0]]
        out["vt"] = vt
        for k, name in (("m_x", "exp_x"), ("m_y", "exp_y"), ("th", "exp_th")):
            out[k] = self._col(name, n, b)
        return out

    def links(self, b):
        """Agent b's links in creation order, ``LINK_DTYPE`` [n]: ends, length, heading and facing (radians)."""
        n = int(self.n_links[b])
        out = np.zeros(n, LINK_DTYPE)
        for k, name in (("from", "link_from"), ("to", "link_to"), ("d", "link_d"), ("heading", "link_heading"),
                        ("facing", "link_facing")):
            out[k] = self._col(name, n, b)
        return out

    def experience_map(self, b):
        """Agent b's map as a host ``ExperienceMap(linked=True)``: ``iterate`` relaxes it, ``update`` continues it."""
        r = 0 if self._rec_of is None else int(self._rec_of[b])
        if r not in self._accum:
            moved, tw = self._odom
            self._accum[r] = dead_reckoning(*((moved, tw) if self._rec_of is None else (moved[:, r], tw[:, r])))[2]
        return ExperienceMap.from_arrays(self.experiences(b), self.links(b), int(self.current[b]),
                                         rel=self._rel[:, b], accum=self._accum[r],
                                         n_loop_closures=int(self.n_loop_closures[b]), pc_dims=self.pose_size,
                                         delta_pc=self.delta_pc, correction=self.correction)


def _maps(tpl, flat, moved, tw, pose_size, linked, delta_pc, correction, device=None, vt_ids=None, rec_of=None):
    """The maps from records in frame-major layout: ``tpl`` int [T,B] (the template of each frame, < 0 = none; the
    kernel's workspace holds a candidate list per id up to the largest), ``flat`` int64 [T,B] (the C-order flat arg-max
    cell); ``vt_ids``: per agent, the caller's template id of each of its ``tpl`` values, when they were renumbered.
    ``rec_of`` int [B] (several recordings): ``moved`` is [T,R], ``tw`` [T,R,2], and agent b follows ``rec_of[b]``."""
    T, B = tpl.shape
    if not linked:
        if rec_of is None:
            n_exp, em_xy, _ = dead_reckoning(moved, tw)
            return {"n_exp": np.tile(n_exp, (B, 1)), "em_xy": np.tile(em_xy, (B, 1, 1)),
                    "exp_id": np.tile(n_exp - 1, (B, 1)), "n_loop_closures": np.zeros(B, np.int64), "maps": None}
        per = [dead_reckoning(moved[:, r], tw[:, r])[:2] for r in range(moved.shape[1])]   # once per recording
        n_exp = np.stack([per[r][0] for r in rec_of]) if B else np.zeros((0, T), np.int64)
        em_xy = np.stack([per[r][1] for r in rec_of]) if B else np.zeros((0, T, 2))
        return {"n_exp": n_exp, "em_xy": em_xy, "exp_id": n_exp - 1, "n_loop_closures": np.zeros(B, np.int64),
                "maps": None}
    tag = np.full((T, B), -1, np.int32)
    if T > 1:
        tag[1:] = np.maximum(tpl[:-1], -1)
    n_templates = int(tag.max()) + 1 if T else 0
    nat.require_cuda()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
    L = nat.lib()
    nbytes = work_bytes(B, T, n_templates)
    assert int(L.prs_em_work_bytes(B, T, n_templates)) == nbytes
    with torch.cuda.device(dev):
        work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        flat_d = torch.from_numpy(np.ascontiguousarray(flat, dtype=np.int64)).to(dev)
        tag_d = torch.from_numpy(tag).to(dev)
        tw_d = torch.from_numpy(np.ascontiguousarray(tw, dtype=np.float64)).to(dev)
        moved_d = torch.from_numpy(np.ascontiguousarray(moved, dtype=np.uint8)).to(dev)
        n_d = torch.empty((T, B), dtype=torch.int32, device=dev)
        id_d = torch.empty((T, B), dtype=torch.int32, device=dev)
        xy_d = torch.empty((T, B, 2), dtype=torch.float64, device=dev)
        X, Y, Th = pose_size
        if rec_of is None:
            nat.check(L.prs_em_linked_run(B, T, n_templates, flat_d.data_ptr(), tag_d.data_ptr(), tw_d.data_ptr(),
                                          moved_d.data_ptr(), X, Y, Th, float(delta_pc), work.data_ptr(),
                                          n_d.data_ptr(), id_d.data_ptr(), xy_d.data_ptr(), nat.stream_ptr()),
                      "prs_em_linked_run")
        else:
            rec_d = torch.from_numpy(np.asarray(rec_of, dtype=np.int32)).to(dev)
            nat.check(L.prs_em_linked_multi_run(B, T, n_templates, flat_d.data_ptr(), tag_d.data_ptr(), moved.shape[1],
                                                tw_d.data_ptr(), moved_d.data_ptr(), rec_d.data_ptr(), X, Y, Th,
                                                float(delta_pc), work.data_ptr(), n_d.data_ptr(), id_d.data_ptr(),
                                                xy_d.data_ptr(), nat.stream_ptr()), "prs_em_linked_multi_run")
        maps = EnsembleExperienceMaps(work, B, T, n_templates, moved, tw, pose_size, delta_pc, correction, vt_ids,
                                      rec_of)
        out = {"n_exp": n_d.cpu().numpy().T.astype(np.int64), "exp_id": id_d.cpu().numpy().T.astype(np.int64),
               "em_xy": xy_d.cpu().numpy().transpose(1, 0, 2), "n_loop_closures": maps.n_loop_closures.copy(),
               "maps": maps}
    return out


def ensemble_experience_maps(template, argmax, odom, pose_size, linked, delta_pc=1.0, correction=0.5):
    """Every agent's experience map from its records: ``template`` int [B,T] (the template each frame matched or
    created; < 0 = none), ``argmax`` int [B,T,3] (the arg-max pose cell), ``odom`` [T,2] = (linear.x, angular.z), shared.

    Returns a dict with ``n_exp`` int64 [B,T] (experiences after each frame), ``exp_id`` int64 [B,T] (the current
    experience, -1 = none), ``em_xy`` float64 [B,T,2] (its position, 0 while there is none), ``n_loop_closures`` int64
    [B] and ``maps``: ``EnsembleExperienceMaps`` when linked (built on the device), None otherwise (every agent's map
    is the shared dead reckoning, computed on the host).  ``delta_pc`` is the loop-closure radius in cells,
    ``correction`` the relaxation gain of the rebuilt host maps.  Template ids may be any integers: ids of T or more
    are renumbered per agent for the device and reported as given.  ``ValueError`` for bad shapes or cells outside the
    grid."""
    template = np.asarray(template)
    argmax = np.asarray(argmax)
    odom = np.asarray(odom, dtype=np.float64)
    pose_size = tuple(int(s) for s in pose_size)
    if template.ndim != 2 or argmax.shape != template.shape + (3,) or odom.shape != (template.shape[1], 2):
        raise ValueError("ensemble_experience_maps: template must be [B,T], argmax [B,T,3] and odom [T,2], got %r, %r "
                         "and %r" % (template.shape, argmax.shape, odom.shape))
    if len(pose_size) != 3 or min(pose_size) < 1:
        raise ValueError("ensemble_experience_maps: pose_size must be three positive sizes, got %r" % (pose_size,))
    if template.shape[0] < 1:
        raise ValueError("ensemble_experience_maps: no agents")
    for a in (template, argmax):
        if a.size and not np.issubdtype(a.dtype, np.integer):
            raise ValueError("ensemble_experience_maps: template and argmax must be integers, got %s" % a.dtype)
    template = template.astype(np.int64)
    argmax = argmax.astype(np.int64)
    if argmax.size and ((argmax < 0).any() or (argmax >= np.array(pose_size)).any()):
        raise ValueError("ensemble_experience_maps: arg-max cells outside the %r grid" % (pose_size,))
    X, Y, Th = pose_size
    flat = (argmax[..., 0] * Y + argmax[..., 1]) * Th + argmax[..., 2]
    moved, tw = gate(odom)
    B, T = template.shape
    vt_ids = None
    if linked and template.size and template.max() >= T:
        # ids beyond what T frames can create: number each agent's templates 0, 1, ... (at most T of them), so that the
        # kernel's per-template candidate lists stay O(T) per agent; experiences() maps the tags back
        vt_ids, dense = [], np.full_like(template, -1)
        for b in range(B):
            seen = template[b] >= 0
            ids, dense[b, seen] = np.unique(template[b, seen], return_inverse=True)
            vt_ids.append(ids)
        template = dense
    return _maps(np.ascontiguousarray(template.T), np.ascontiguousarray(flat.T), moved, tw, pose_size, linked,
                 delta_pc, correction, vt_ids=vt_ids)
