"""Experience map -- host bookkeeping, as in the reference (``ratslam/experience_map.py``).

Graph relaxation and the viewers stay on the host (BASELINE north_star: "ExperienceMap graph relaxation ... stay on
the host as non-hot code"); so does this class's per-step update of a single agent.  For an ensemble replay, every
agent's per-frame linked update runs on the device instead (``experience_ensemble``, csrc/experience_map.cu), and
``ExperienceMap.from_arrays`` turns an agent's result back into this class.  By default it is the reference's class: it
dead-reckons a 2-D pose from the odometry and records one experience per update, tagged with the arg-max pose cell
(``experience_map.py:44-60``).

``ExperienceMap(linked=True)`` adds what the reference left as TODOs (``experience_map.py:49`` "linking will go here",
``:59`` "leaving vt stuff out"): experiences are linked by the odometry travelled between them, a revisit -- same view
template and a pose cell within ``delta_pc`` cells of a stored experience -- closes a loop instead of creating a new
experience, and ``iterate()`` relaxes the graph (the published RatSLAM experience-map algorithm).  The behaviour is
specified by ``oracle/experience_map.py:LinkedExperienceMap`` and tested against it; experiences, links and the
per-template candidate lists live in flat arrays / dicts here, so a lookup touches only the experiences that share
the view template.
"""
from __future__ import annotations

import math

_TWO_PI = 2 * math.pi


def clip_rad_180(angle):
    """Wrap an angle into (-pi, pi] the way ``experience_map.py:6-11`` does."""
    if angle > math.pi:
        return angle - math.ceil(angle / _TWO_PI) * _TWO_PI
    if angle <= -math.pi:
        return angle + math.ceil(abs(angle) / _TWO_PI) * _TWO_PI
    return angle


def signed_delta_rad(a, b):
    """Smallest signed rotation from heading ``a`` to heading ``b``."""
    d = clip_rad_180(b) - clip_rad_180(a)
    if d > math.pi:
        return d - _TWO_PI
    if d <= -math.pi:
        return d + _TWO_PI
    return d


class Experience:
    def __init__(self, pc_loc, em_loc, vt):
        self.pc_x, self.pc_y, self.pc_th = pc_loc[0], pc_loc[1], pc_loc[2]
        self.vt = vt
        self.m_x, self.m_y = em_loc[0], em_loc[1]

    def get_point(self):
        return (self.m_x, self.m_y)


class ExperienceMap:
    def __init__(self, linked=False, pc_dims=(21, 21, 36), delta_pc=1.0, correction=0.5):
        self.accum_delta_x = 0
        self.accum_delta_y = 0
        self.accum_delta_th = 0
        self.experiences = []
        self.current_exp = None
        # the extension (inactive unless linked=True)
        self.linked = bool(linked)
        self.pc_dims = tuple(pc_dims)
        self.delta_pc = delta_pc
        self.correction = correction
        self.rel_x = self.rel_y = self.rel_th = 0.0
        self.n_loop_closures = 0
        self._lfrom, self._lto, self._ld, self._lhead, self._lface = [], [], [], [], []   # links, creation order
        self._out = []            # per experience: indices of the links that start there
        self._by_vt = {}          # view template -> experience ids created with it

    @classmethod
    def from_arrays(cls, experiences, links, current, rel=(0.0, 0.0, 0.0), accum=(0.0, 0.0, 0.0), n_loop_closures=0,
                    pc_dims=(21, 21, 36), delta_pc=1.0, correction=0.5):
        """A linked map rebuilt from its arrays, e.g. one agent's map built on the device
        (``experience_ensemble.EnsembleExperienceMaps.experience_map``).

        ``experiences``: records with fields ``pc_x, pc_y, pc_th, vt`` (< 0: no view template), ``m_x, m_y, th``, in
        index order; ``links``: records with fields ``from, to, d, heading, facing``, in creation order; ``current``:
        the current experience's index (< 0: none); ``rel`` = (rel_x, rel_y, rel_th); ``accum`` = (accum_delta_x,
        accum_delta_y, accum_delta_th).  The result relaxes (``iterate``) and updates as the original map would."""
        em = cls(linked=True, pc_dims=pc_dims, delta_pc=delta_pc, correction=correction)
        for i, r in enumerate(experiences):
            vt = int(r["vt"])
            vt = None if vt < 0 else vt
            e = Experience((int(r["pc_x"]), int(r["pc_y"]), int(r["pc_th"])), (float(r["m_x"]), float(r["m_y"])), vt)
            e.th = float(r["th"])
            e.index = i
            em.experiences.append(e)
            em._out.append([])
            if vt is not None:
                em._by_vt.setdefault(vt, []).append(i)
        for li, r in enumerate(links):
            em._lfrom.append(int(r["from"]))
            em._lto.append(int(r["to"]))
            em._ld.append(float(r["d"]))
            em._lhead.append(float(r["heading"]))
            em._lface.append(float(r["facing"]))
            em._out[int(r["from"])].append(li)
        em.current_exp = em.experiences[int(current)] if int(current) >= 0 else None
        em.rel_x, em.rel_y, em.rel_th = (float(v) for v in rel)
        em.accum_delta_x, em.accum_delta_y, em.accum_delta_th = (float(v) for v in accum)
        em.n_loop_closures = int(n_loop_closures)
        return em

    # ------------------------------------------------------------------ the reference's class (experience_map.py:44-70)
    def create(self, pc_loc, vt=None):
        if self.linked:
            return self._create_linked(pc_loc, vt)
        self.current_exp = Experience(pc_loc, (self.accum_delta_x, self.accum_delta_y), vt)
        self.experiences.append(self.current_exp)

    def update(self, vtrans, vrot, pc_loc, vt=None):
        th = clip_rad_180(self.accum_delta_th + vrot)
        self.accum_delta_th = th
        self.accum_delta_x += vtrans * math.cos(th)
        self.accum_delta_y += vtrans * math.sin(th)
        if not self.linked:
            self.create(pc_loc)                 # experience_map.py:59-60: the reference ignores vt
            return
        self.rel_th = clip_rad_180(self.rel_th + vrot)
        self.rel_x += vtrans * math.cos(self.rel_th)
        self.rel_y += vtrans * math.sin(self.rel_th)
        match = self._find(pc_loc, vt)
        if match is None:
            self._create_linked(pc_loc, vt)
        elif match is not self.current_exp:
            self._add_link(self.current_exp, match)
            self.n_loop_closures += 1
            self._set_current(match)

    def get_points(self):
        return [e.get_point() for e in self.experiences]

    def get_current_point(self):
        return self.current_exp.get_point()

    # ------------------------------------------------------------------ links and loop closure (linked=True)
    @property
    def links(self):
        """``(from, to, d, heading_rad, facing_rad)`` per link, in creation order."""
        return list(zip(self._lfrom, self._lto, self._ld, self._lhead, self._lface))

    def get_poses(self):
        return [(e.m_x, e.m_y, e.th) for e in self.experiences]

    def _find(self, pc_loc, vt):
        if vt is None or self.current_exp is None:
            return None
        best, best_d2 = None, None
        px, py, pt = float(pc_loc[0]), float(pc_loc[1]), float(pc_loc[2])
        nx, ny, nt = self.pc_dims
        for i in self._by_vt.get(vt, ()):     # ascending ids: the first of equally near candidates wins
            e = self.experiences[i]
            dx = abs(e.pc_x - px) % nx
            dy = abs(e.pc_y - py) % ny
            dt = abs(e.pc_th - pt) % nt
            dx, dy, dt = min(dx, nx - dx), min(dy, ny - dy), min(dt, nt - dt)
            d2 = dx * dx + dy * dy + dt * dt
            # compare the distances themselves (sqrt is monotone but rounds): the specification tests sqrt(d2) <= delta_pc
            if math.sqrt(d2) <= self.delta_pc and (best is None or math.sqrt(d2) < best_d2):
                best, best_d2 = e, math.sqrt(d2)
        return best

    def _add_link(self, a, b):
        for li in self._out[a.index]:
            if self._lto[li] == b.index:
                return False
        self._lfrom.append(a.index)
        self._lto.append(b.index)
        self._ld.append(math.hypot(self.rel_x, self.rel_y))
        self._lhead.append(signed_delta_rad(a.th, math.atan2(self.rel_y, self.rel_x)))
        self._lface.append(signed_delta_rad(a.th, self.rel_th))
        self._out[a.index].append(len(self._lfrom) - 1)
        return True

    def _set_current(self, e):
        self.current_exp = e
        self.rel_x = self.rel_y = 0.0
        self.rel_th = e.th

    def _create_linked(self, pc_loc, vt):
        cur = self.current_exp
        base = (0.0, 0.0) if cur is None else (cur.m_x, cur.m_y)
        e = Experience(pc_loc, (base[0] + self.rel_x, base[1] + self.rel_y), vt)
        e.th = clip_rad_180(self.rel_th)
        e.index = len(self.experiences)
        self.experiences.append(e)
        self._out.append([])
        if vt is not None:
            self._by_vt.setdefault(vt, []).append(e.index)
        if cur is not None:
            self._add_link(cur, e)
        self._set_current(e)

    def iterate(self, loops=1):
        """Graph relaxation: ``loops`` Gauss-Seidel sweeps over the links, ordered by their start experience and
        then by creation, each moving both ends by ``correction`` times the link's position / heading error."""
        if not self.linked or not self._lfrom:
            return
        order = [li for outs in self._out for li in outs]
        x = [e.m_x for e in self.experiences]
        y = [e.m_y for e in self.experiences]
        th = [e.th for e in self.experiences]
        c = self.correction
        lf, lt, ld, lh, lc = self._lfrom, self._lto, self._ld, self._lhead, self._lface
        cos, sin = math.cos, math.sin
        for _ in range(loops):
            for li in order:
                a, b = lf[li], lt[li]
                ang = th[a] + lh[li]
                ex = (x[b] - (x[a] + ld[li] * cos(ang))) * c
                ey = (y[b] - (y[a] + ld[li] * sin(ang))) * c
                x[a] += ex
                y[a] += ey
                x[b] -= ex
                y[b] -= ey
                df = signed_delta_rad(th[a] + lc[li], th[b])
                th[a] = clip_rad_180(th[a] + df * c)
                th[b] = clip_rad_180(th[b] - df * c)
        for e, ex, ey, et in zip(self.experiences, x, y, th):
            e.m_x, e.m_y, e.th = ex, ey, et
