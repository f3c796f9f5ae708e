"""The node's message loop on the CPU oracle (test infrastructure only): ``replay_events_run`` is the specification
of a message-stream replay, built from the oracle's classes the way ``oracle.drivers.replay_run`` is, with the
agent's global inhibition given to the oracle's ``PoseCellNetwork``."""
from __future__ import annotations

import math

import numpy as np

from oracle import drivers as odrv
from oracle.experience_map import ExperienceMap, LinkedExperienceMap
from oracle.posecells import PC_GLOBAL_INHIB, PoseCellNetwork
from oracle.view_templates import ViewTemplates


def replay_events_run(events, shape=odrv.POSE_SIZE_ROS, match_threshold=odrv.MATCH_THRESHOLD, inject_energy=None,
                      experience_links=False, global_inhibition=PC_GLOBAL_INHIB):
    """``ros_simulate.replay_events(fused=False)`` on the oracle: an ``("odom", stamp, (lin, ang))`` message above the
    0.001 gate is one pose-cell update and one experience-map update (tagged, with links, by the most recent image's
    template), an ``("image", stamp, frame)`` is one match with the current arg-max (and the injection).  Returns the
    per-image records (``template``, ``created``, ``argmax``, ``n_exp``, ``em_xy``) and ``em``, ``final_state``,
    ``n_templates``, ``templates``, ``locations``.  On a stream in which odometry and images alternate this is
    ``replay_run(*events_to_arrays(events)[:2])``."""
    pcn = PoseCellNetwork(shape, global_inhibition=global_inhibition)
    pcn.inject(1, tuple(math.floor(s / 2) for s in shape))
    vts = ViewTemplates(odrv.X_RANGE, odrv.Y_RANGE, odrv.X_STEP, odrv.Y_STEP, odrv.IM_SIZE[0], odrv.IM_SIZE[1],
                        match_threshold)
    em = LinkedExperienceMap(shape) if experience_links else ExperienceMap()
    last_vt = None
    rec = {"template": [], "created": [], "argmax": [], "n_exp": [], "em_xy": []}
    for kind, _, payload in events:
        if kind == "odom":
            lin, ang = float(payload[0]), float(payload[1])
            if abs(lin) > 0.001 or abs(ang) > 0.001:
                vtrans, vrot = lin / odrv.ODOM_FREQ, ang / odrv.ODOM_FREQ
                pcn.update((vtrans, vrot))
                em.update(vtrans, vrot, pcn.get_pc_max(), last_vt if experience_links else None)
            continue
        pc_max = pcn.get_pc_max()
        n0 = len(vts.templates)
        tm = vts.match(payload, pc_max[0], pc_max[1], pc_max[2])
        if inject_energy is not None:
            pcn.inject(inject_energy, tm.location())
        last_vt = tm.get_index()
        rec["template"].append(tm.get_index())
        rec["created"].append(len(vts.templates) > n0)
        rec["argmax"].append(tuple(pc_max))
        rec["n_exp"].append(len(em.experiences))
        rec["em_xy"].append(em.get_current_point() if em.current_exp is not None else (0.0, 0.0))
    out = {"template": np.asarray(rec["template"], np.int64), "created": np.asarray(rec["created"], np.bool_),
           "argmax": np.asarray(rec["argmax"], np.int64).reshape(-1, 3),
           "n_exp": np.asarray(rec["n_exp"], np.int64), "em_xy": np.asarray(rec["em_xy"], np.float64).reshape(-1, 2)}
    out["em"] = em
    out["final_state"] = pcn.posecells
    out["n_templates"] = len(vts.templates)
    out["templates"] = np.stack([t.template for t in vts.templates]) if vts.templates else np.zeros((0, 32, 32))
    out["locations"] = np.array([t.location() for t in vts.templates], dtype=np.int64).reshape(-1, 3)
    return out
