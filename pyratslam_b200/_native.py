"""ctypes binding of libpyratslam_b200.so (the C ABI in include/pyratslam_b200.h).

There is no CPU fallback: if the shared library has not been built, or no CUDA
device is present when a compute entry is called, this module raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int, c_longlong, c_size_t, c_uint64, c_void_p

PKG = os.path.dirname(os.path.abspath(__file__))
# PYRATSLAM_B200_LIB: another build of the same library (profiling variants, bench_tools/variant_bench.py)
LIB_PATH = os.environ.get("PYRATSLAM_B200_LIB") or os.path.join(PKG, "_lib", "libpyratslam_b200.so")

PRS_F32, PRS_F64 = 0, 1
ERR_LUT_KEY, ERR_RADIUS, ERR_THETA = 1, 2, 4
ERR_INJECT_LOC = 8             # prs_frame_result.pc_err: the frame's template has no valid pose cell
E_LUT_KEY, E_RADIUS = -4, -5   # return codes of prs_pc_update_host
OG_RANGE = 8
VT_MODE_REF, VT_MODE_CIRCULAR = 0, 1


class NativeLibraryMissing(RuntimeError):
    pass


class PcConfig(Structure):
    _fields_ = [
        ("X", c_int), ("Y", c_int), ("Th", c_int), ("B", c_int), ("dtype", c_int),
        ("vtrans_scale", c_double), ("vrot_scale", c_double),
        ("ge", POINTER(c_double)), ("gi", POINTER(c_double)),
        ("aE", c_double), ("aI", c_double),
        ("f2d", POINTER(c_double)), ("f1d", POINTER(c_double)),
        ("cos_th", POINTER(c_double)), ("sin_th", POINTER(c_double)),
    ]


_SIGNATURES = {
    "prs_last_error": (c_char_p, []),
    "prs_version": (c_int, []),
    "prs_device_count": (c_int, []),
    "prs_pc_create": (c_int, [POINTER(PcConfig), POINTER(c_void_p)]),
    "prs_pc_destroy": (c_int, [c_void_p]),
    "prs_pc_state_bytes": (c_size_t, [c_void_p]),
    "prs_pc_path": (c_int, [c_void_p]),
    "prs_pc_set_path": (c_int, [c_void_p, c_int]),
    "prs_pc_set_option": (c_int, [c_void_p, c_int, c_int]),
    "prs_pc_invalidate_active": (c_int, [c_void_p, c_void_p]),
    "prs_pc_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_run": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_step_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_step_host_xyz": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_step_host_xyz_async": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                           ctypes.POINTER(c_int)]),
    "prs_pc_host_result_wait": (c_int, [c_void_p, c_int]),
    "prs_pc_update_host": (c_int, [c_void_p, c_void_p, c_double, c_double, c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_path_integration": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_inject": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double, c_void_p]),
    "prs_pc_active_work_bytes": (c_size_t, [c_void_p]),
    "prs_pc_active_cells": (c_int, [c_void_p, c_void_p, c_int, c_double, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "prs_pc_argmax": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_import_xyt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_pc_export_xyt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "prs_vt_extract_u8": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                  c_int, c_int, c_void_p]),
    "prs_vt_sweep_u8": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p]),
    "prs_vt_sweep_f32": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p]),
    "prs_vt_packed_bytes": (c_size_t, [c_longlong]),
    "prs_vt_pack_u8": (c_int, [c_void_p, c_longlong, c_void_p, c_longlong, c_void_p]),
    "prs_vt_unpack_u8": (c_int, [c_void_p, c_longlong, c_void_p, c_void_p]),
    "prs_vt_sweep_packed_u8": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p,
                                       c_void_p]),
    "prs_vt_sweep_any_u8": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_int, c_int, c_longlong, c_void_p, c_void_p,
                                    c_void_p]),
    "prs_vt_sweep_any_f32": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_int, c_int, c_longlong, c_void_p, c_void_p,
                                     c_void_p]),
    "prs_vt_match_host_u8": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p]),
}

_SIGNATURES["prs_frame_scratch_bytes"] = (c_size_t, [])
_SIGNATURES["prs_frame_host"] = (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double,
                                         c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                         c_void_p, c_void_p])
_SIGNATURES["prs_frame_create"] = (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_double,
                                           c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                           c_void_p, c_void_p, c_void_p, POINTER(c_void_p)])
_SIGNATURES["prs_frame_destroy"] = (c_int, [c_void_p])
_SIGNATURES["prs_frame_set_count"] = (c_int, [c_void_p, c_int, c_void_p])
_SIGNATURES["prs_frame_run"] = (c_int, [c_void_p, c_int, c_void_p])
_SIGNATURES["prs_frame_launch"] = (c_int, [c_void_p, c_int, c_void_p])
_SIGNATURES["prs_frame_set_inject"] = (c_int, [c_void_p, c_double, c_void_p])
_SIGNATURES["prs_replay_run"] = (c_int, [POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p])
_SIGNATURES["prs_ens_scratch_bytes"] = (c_size_t, [c_void_p, c_int, c_int, c_int])
_SIGNATURES["prs_ens_create"] = (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                         c_int, c_int, c_int, c_void_p, POINTER(c_void_p)])
_SIGNATURES["prs_ens_destroy"] = (c_int, [c_void_p])
_SIGNATURES["prs_ens_refresh_room"] = (c_int, [c_void_p, c_void_p])
_SIGNATURES["prs_ens_run"] = (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p])
_SIGNATURES["prs_ens_chunk"] = (c_int, [c_void_p])
_SIGNATURES["prs_ens_activity_bytes"] = (c_size_t, [c_void_p, c_int])
_SIGNATURES["prs_ens_set_activity"] = (c_int, [c_void_p, c_double, c_int, c_void_p])
_SIGNATURES["prs_ens_activity_pack"] = (c_int, [c_void_p, c_void_p, c_void_p, c_void_p])
_SIGNATURES["prs_ens_activity_copy"] = (c_int, [c_void_p, c_longlong, c_void_p, c_void_p, c_void_p])
_SIGNATURES["prs_ens_copy_stage_bytes"] = (c_size_t, [c_void_p, c_int, c_void_p, c_void_p, c_void_p])
_SIGNATURES["prs_ens_copy_agents"] = (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                              c_void_p])
_SIGNATURES["prs_ens_export_stage_bytes"] = (c_size_t, [c_void_p, c_int, c_void_p, c_void_p])
_SIGNATURES["prs_ens_export_agents"] = (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p])
_SIGNATURES["prs_ens_import_agents"] = (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_size_t, c_void_p])
_SIGNATURES["prs_stage_copy"] = (c_int, [c_void_p, c_int, c_void_p, c_int, c_size_t, c_void_p])
_SIGNATURES["prs_em_work_bytes"] = (c_size_t, [c_int, c_int, c_int])
_SIGNATURES["prs_em_linked_run"] = (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                            c_int, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p])
_SIGNATURES["prs_em_linked_multi_run"] = (c_int, [c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                                  c_void_p, c_int, c_int, c_int, c_double, c_void_p, c_void_p, c_void_p,
                                                  c_void_p, c_void_p])
_SIGNATURES["prs_em_session_bytes"] = (c_size_t, [c_int, c_int, c_int])
_SIGNATURES["prs_em_session_init"] = (c_int, [c_int, c_int, c_int, c_void_p, c_void_p])
_SIGNATURES["prs_em_session_grow"] = (c_int, [c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p])
_SIGNATURES["prs_em_session_copy_stage_bytes"] = (c_size_t, [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p])
_SIGNATURES["prs_em_session_copy_agents"] = (c_int, [c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                                     c_void_p, c_size_t, c_void_p])
_SIGNATURES["prs_em_session_export_stage_bytes"] = (c_size_t, [c_int, c_int, c_int, c_int, c_void_p, c_void_p])
_SIGNATURES["prs_em_session_export_agents"] = (c_int, [c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p,
                                                       c_void_p, c_size_t, c_void_p])
_SIGNATURES["prs_em_session_import_agents"] = (c_int, [c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p,
                                                       c_size_t, c_void_p])
_SIGNATURES["prs_em_linked_resume_run"] = (c_int, [c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                                   c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_void_p, c_void_p,
                                                   c_void_p, c_void_p, c_void_p])


_SIGNATURES["prs_xchg_create"] = (c_int, [c_int, c_int, POINTER(c_void_p)])
_SIGNATURES["prs_xchg_export"] = (c_int, [c_void_p, c_void_p])
_SIGNATURES["prs_xchg_connect"] = (c_int, [c_void_p, c_void_p])
_SIGNATURES["prs_xchg_set_timeout"] = (c_int, [c_void_p, c_double])
_SIGNATURES["prs_xchg_destroy"] = (c_int, [c_void_p])
_SIGNATURES["prs_vt_shard_exchange"] = (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p])
_SIGNATURES["prs_vt_shard_decide"] = (c_int, [c_void_p, c_void_p, c_double, c_int, c_void_p, c_void_p, c_longlong,
                                              c_longlong, c_int, c_void_p, c_void_p])
_SIGNATURES["prs_xchg_wait"] = (c_int, [c_void_p, c_void_p, c_double])
_SIGNATURES["prs_vt_shard_query"] = (c_int, [c_void_p, c_int, c_void_p, c_longlong, c_void_p, c_int, c_longlong, c_void_p,
                                             c_void_p, c_int, c_double, c_longlong, c_int, c_void_p, c_void_p])
XCHG_HANDLE_BYTES = 64
PRS_U8 = 2


class ShardResult(Structure):
    _fields_ = [("key", c_uint64), ("created", c_int), ("template_index", c_int), ("n_total", c_int),
                ("status", c_int), ("seq", c_uint64)]


class FrameResult(Structure):
    _fields_ = [("argmax", c_longlong), ("key", c_uint64), ("created", c_int), ("template_index", c_int),
                ("n_templates", c_int), ("pc_err", c_int)]


_lib = None


def lib():
    """The loaded shared library (loads on first use)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                "%s is missing: build it with `python -m pyratslam_b200.build` (needs nvcc). "
                "pyratslam_b200 has no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


class NativeError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        msg = lib().prs_last_error().decode(errors="replace")
        if rc == -1:
            raise ValueError("%s: %s" % (what, msg) if what else msg)
        raise NativeError("%s failed (%d): %s" % (what, rc, msg))


def stream_ptr():
    """The current torch CUDA stream as a void* for the C ABI."""
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise NativeError("pyratslam_b200 needs a CUDA device (sm_100a); there is no CPU path")
    lib()
