"""CPU-only checks of the product's host side: the C-ABI library loads and exports what the header
declares, the filter builders agree with the reference-generated fixtures, and the product never
falls back to a CPU path."""
import ctypes
import os
import re

import numpy as np
import pytest

import pyratslam_b200
from pyratslam_b200 import _native as nat
from pyratslam_b200 import kernels as K

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    names = set()
    inc = os.path.join(ROOT, "include")
    for f in os.listdir(inc):
        if f.endswith(".h"):
            src = open(os.path.join(inc, f)).read()
            names |= set(re.findall(r"PRS_API\s+[\w\s\*]+?\b(prs_\w+)\s*\(", src))
    return sorted(names)


def test_library_exports_every_declared_symbol():
    syms = _declared_symbols()
    assert len(syms) >= 20
    L = ctypes.CDLL(nat.LIB_PATH)
    for s in syms:
        assert hasattr(L, s), "missing export: " + s
    # and the ctypes table binds exactly the declared set
    assert sorted(nat.exported_symbols()) == syms


def test_library_reports_version_and_errors_without_gpu():
    L = nat.lib()
    assert L.prs_version() >= 100
    import torch
    if not torch.cuda.is_available():
        assert L.prs_device_count() <= 0
        cfg = nat.PcConfig()
        h = ctypes.c_void_p()
        assert L.prs_pc_create(ctypes.byref(cfg), ctypes.byref(h)) != 0
        assert len(L.prs_last_error()) > 0


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(nat.NativeError):
        pyratslam_b200.PoseCellNetwork((21, 21, 36))
    with pytest.raises(nat.NativeError):
        pyratslam_b200.ViewTemplates((32, 96), (32, 96), 2, 2, 256, 256, 45000)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "pyratslam_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f
                assert "scipy.ndimage" not in src, f


def test_builders_match_reference_fixtures(golden):
    g = golden("kernels.npz")
    k3 = K.diff_gaussian(order=3)
    assert np.abs(k3 - g["kernel_3d"]).max() <= 1e-15 * np.abs(g["kernel_3d"]).max()
    lut = K.build_diff_gaussian_set_2d()
    for k, f in zip([tuple(k) for k in g["lut_keys"].tolist()], g["lut_filters"]):
        assert np.abs(lut[k] - f).max() <= 1e-15
    for og in range(-5, 6):
        assert np.abs(K.diff_gaussian_offset_1d(origin=float(og)) - g["f1d_og%+d" % og]).max() <= 1e-15
    tab = K.theta_filter_table(nat.OG_RANGE)
    assert tab.shape == (2 * nat.OG_RANGE + 1, 7)
    # beyond |og| = 4 every tap is negative: the clamp at og = +-8 in the kernel cannot change a result
    for og in range(5, nat.OG_RANGE + 1):
        assert (tab[nat.OG_RANGE + og] < 0).all() and (tab[nat.OG_RANGE - og] < 0).all()
    # ... up to |og| = 64, the largest theta origin the kernels accept (PRS_ERR_THETA beyond): og 9..64 run with the
    # og = 8 filter, and an all-negative filter followed by the clamp at zero zeroes the state whichever it is
    wide = K.theta_filter_table(64)
    for og in range(5, 65):
        for f in (wide[64 + og], wide[64 - og], K.diff_gaussian_offset_1d(origin=float(og)),
                  K.diff_gaussian_offset_1d(origin=float(-og))):
            assert (f < 0).all(), og
    # |og| = 3, 4 are the asymmetric filters with two or one positive taps at the edge
    for og, npos in ((3, 2), (4, 1)):
        for s in (1, -1):
            f = tab[nat.OG_RANGE + s * og]
            assert int((f > 0).sum()) == npos and (f[-npos:] > 0 if s > 0 else f[:npos] > 0).all(), (s * og, f)


def test_separable_factorisation_reproduces_kernel_3d(golden):
    ge, gi, aE, aI = K.separable_dog_factors()
    rebuilt = (aE * np.einsum("i,j,k->ijk", ge, ge, ge) - aI * np.einsum("i,j,k->ijk", gi, gi, gi))
    ref = golden("kernels.npz")["kernel_3d"]
    assert np.abs(rebuilt - ref).max() <= 4e-16
    assert abs(rebuilt.sum() - 1.0) < 1e-14


def test_lower_order_kernels_normalised():
    for order in (1, 2, 3):
        f = K.diff_gaussian(order=order)
        assert f.shape == (7,) * order and abs(abs(f.sum()) - 1) < 1e-12
    assert K.diff_gaussian_separable().shape == (7,)
    assert abs(K.build_kernel(7, 1, order=2).sum() - 1) < 1e-12


def test_linked_experience_map_against_specification():
    """SURVEY 8f row 3: links, loop closure and relaxation (the reference's TODOs, experience_map.py:49,59) against
    the specification in oracle/experience_map.py, on a looped trajectory with revisits; the default mode stays the
    reference's class (one experience per update, no links)."""
    import math
    from oracle import experience_map as oem
    from pyratslam_b200.experience_map import ExperienceMap
    rng = np.random.default_rng(11)
    ours, spec = ExperienceMap(linked=True, pc_dims=(21, 21, 36), delta_pc=1.5), oem.LinkedExperienceMap((21, 21, 36), 1.5)
    plain_o, plain_s = ExperienceMap(), oem.ExperienceMap()
    raw = ExperienceMap(linked=True, pc_dims=(21, 21, 36), delta_pc=1.5)      # never relaxed
    T = 400
    for t in range(T):
        ph = 2 * math.pi * t / 100.0                      # four laps of a circle: lap k revisits lap 0
        vtrans, vrot = 0.3 + 0.02 * rng.standard_normal(), 2 * math.pi / 100.0 + 0.003 * rng.standard_normal()
        pc = (int(10 + 8 * math.cos(ph)) % 21, int(10 + 8 * math.sin(ph)) % 21, int(36 * (t % 100) / 100.0))
        vt = (t % 100) // 2 if t % 7 else None            # a view template per two steps; some frames without one
        for m in (ours, spec, raw):
            m.update(vtrans, vrot, pc, vt)
        for m in (plain_o, plain_s):
            m.update(vtrans, vrot, pc, vt)
        assert ours.get_current_point() == spec.get_current_point()
        if t % 50 == 49:
            ours.iterate(3)
            spec.iterate(3)
    assert len(ours.experiences) == len(spec.experiences) < T and ours.n_loop_closures == spec.n_loop_closures > 50
    assert ours.links == [(l.exp_from, l.exp_to, l.d, l.heading_rad, l.facing_rad) for l in spec.links]
    assert ours.get_poses() == spec.get_poses()
    assert (ours.accum_delta_x, ours.accum_delta_y, ours.accum_delta_th) == \
        (spec.accum_delta_x, spec.accum_delta_y, spec.accum_delta_th)
    # relaxation spreads the loop-closure errors over the graph: the sum of squared link residuals shrinks
    def residual(m):
        r = 0.0
        for a, b, d, h, _ in m.links:
            ea, eb = m.experiences[a], m.experiences[b]
            r += (eb.m_x - ea.m_x - d * math.cos(ea.th + h)) ** 2 + (eb.m_y - ea.m_y - d * math.sin(ea.th + h)) ** 2
        return r
    assert [l[:2] for l in raw.links] == [l[:2] for l in ours.links]   # relaxation moves poses (and with them the angles later links are measured from), never the graph
    assert residual(ours) < 0.8 * residual(raw)
    assert plain_o.get_points() == plain_s.get_points() and len(plain_o.experiences) == T
