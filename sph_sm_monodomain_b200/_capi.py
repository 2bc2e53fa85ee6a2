"""ctypes binding of include/sphsm_b200.h — one Python function per exported symbol, nothing else.

The library is loaded from the in-tree build (sph_sm_monodomain_b200/libsphsm_b200.so).  There is no fallback:
if the extension is missing, loading raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPHSM_LIB_PATH", os.path.join(HERE, "libsphsm_b200.so"))  # (override: kernel-variant experiments)

NUM_KERNEL_GROUPS = 8
PARTICLE_STRIDE = 132


class Params(C.Structure):
    """sphsm_params (include/sphsm_b200.h) — field for field."""

    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("capacity", C.c_int32), ("world", C.c_float * 3),
        ("kernel_h", C.c_float), ("gravity", C.c_float * 3), ("K", C.c_float), ("stand_density", C.c_float),
        ("time_delta", C.c_float), ("wall_hit", C.c_float), ("mu", C.c_float), ("velocity_mixing", C.c_float),
        ("poly6_constant", C.c_float), ("spiky_constant", C.c_float), ("bspline_constant", C.c_float),
        ("alpha", C.c_float), ("beta", C.c_float), ("quadratic_match", C.c_int32), ("volume_conservation", C.c_int32),
        ("allow_flip", C.c_int32), ("Cm", C.c_float), ("Beta", C.c_float), ("sigma", C.c_float),
        ("stim_strength", C.c_float), ("FH_Vt", C.c_float), ("FH_Vp", C.c_float), ("FH_Vr", C.c_float),
        ("C1", C.c_float), ("C2", C.c_float), ("C3", C.c_float), ("C4", C.c_float), ("voltage_constant", C.c_float),
        ("max_pressure", C.c_float), ("max_voltage", C.c_float), ("particle_mass", C.c_float),
        ("diagnostics", C.c_int32), ("strict", C.c_int32), ("slab_axis", C.c_int32), ("reserved", C.c_int32 * 8),
    ]


# name -> (restype, argtypes); every symbol include/sphsm_b200.h declares
_H = C.c_void_p
_FP, _IP, _DP, _U8P = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_uint8)
SYMBOLS = {
    "sphsm_abi_version": (C.c_int, []),
    "sphsm_default_params": (C.c_int, [C.POINTER(Params)]),
    "sphsm_create": (C.c_int, [C.POINTER(Params), C.POINTER(_H)]),
    "sphsm_destroy": (C.c_int, [_H]),
    "sphsm_get_params": (C.c_int, [_H, C.POINTER(Params)]),
    "sphsm_set_params": (C.c_int, [_H, C.POINTER(Params)]),
    "sphsm_init_fluid": (C.c_int, [_H, _FP, C.c_int]),
    "sphsm_upload_aos": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_int]),
    "sphsm_download_aos": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_int]),
    "sphsm_download_positions": (C.c_int, [_H, _FP, C.c_int]),
    "sphsm_set_stim": (C.c_int, [_H, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]),
    "sphsm_stim_mesh": (C.c_int, [_H, _FP, C.c_int]),
    "sphsm_stim_cube": (C.c_int, [_H, _FP, C.c_int]),
    "sphsm_stim_off": (C.c_int, [_H]),
    "sphsm_set_stim_box": (C.c_int, [_H, _FP, _FP, C.c_float]),
    "sphsm_timer_mark": (C.c_int, [_H, C.c_int]),
    "sphsm_timer_ms": (C.c_int, [_H, _FP]),
    "sphsm_set_masks": (C.c_int, [_H, _U8P, _FP, C.c_int]),
    "sphsm_step": (C.c_int, [_H, C.c_int]),
    "sphsm_stage": (C.c_int, [_H, C.c_int]),
    "sphsm_sync": (C.c_int, [_H]),
    "sphsm_set_masks_async": (C.c_int, [_H, _U8P, _FP, C.c_int]),
    "sphsm_download_positions_async": (C.c_int, [_H, _FP, C.c_int]),
    "sphsm_download_owned_async": (C.c_int, [_H, _IP, _FP, C.c_int, _IP]),
    "sphsm_set_stim_owned_async": (C.c_int, [_H, _FP, C.c_int]),
    "sphsm_io_wait": (C.c_int, [_H]),
    "sphsm_save_state": (C.c_int, [_H, C.c_char_p]),
    "sphsm_load_state": (C.c_int, [_H, C.c_char_p]),
    "sphsm_num_particles": (C.c_int, [_H]),
    "sphsm_num_cells": (C.c_int, [_H]),
    "sphsm_grid_size": (C.c_int, [_H, _IP]),
    "sphsm_total_time_steps": (C.c_int, [_H]),
    "sphsm_enable_stage_timing": (C.c_int, [_H, C.c_int]),
    "sphsm_get_stage_times": (C.c_int, [_H, _DP]),
    "sphsm_get_cells_csr": (C.c_int, [_H, _IP, _IP]),
    "sphsm_get_neighbor_sets": (C.c_int, [_H, C.c_int, _IP, C.c_int, C.c_int, _IP, _IP]),
    "sphsm_get_sm_transform": (C.c_int, [_H, _FP, _FP, _FP]),
    "sphsm_get_launch_count": (C.c_int, [_H, C.POINTER(C.c_longlong)]),
    "sphsm_reset_launch_count": (C.c_int, [_H]),
    "sphsm_last_step_ms": (C.c_int, [_H, _FP]),
    "sphsm_profile_step": (C.c_int, [_H, C.c_int, _FP]),
    "sphsm_kernel_group_name": (C.c_char_p, [C.c_int]),
    "sphsm_comm_unique_id": (C.c_int, [C.c_void_p]),
    "sphsm_comm_init": (C.c_int, [_H, C.c_int, C.c_int, C.c_void_p]),
    "sphsm_comm_set_slab": (C.c_int, [_H, C.c_int, C.c_int]),
    "sphsm_comm_info": (C.c_int, [_H, _IP]),
    "sphsm_comm_x1_sizes": (C.c_int, [_H, _IP]),
    "sphsm_comm_p2p": (C.c_int, [_H]),
    "sphsm_download_owned": (C.c_int, [_H, _IP, _FP, C.c_int, _IP]),
    "sphsm_comm_init_local": (C.c_int, [C.POINTER(_H), C.c_int]),
    "sphsm_step_group": (C.c_int, [C.POINTER(_H), C.c_int, C.c_int]),
    "sphsm_record_start": (C.c_int, [_H, C.c_float, C.c_float, _IP, C.c_int, C.c_int]),
    "sphsm_record_stop": (C.c_int, [_H]),
    "sphsm_record_reset": (C.c_int, [_H]),
    "sphsm_get_activation": (C.c_int, [_H, _IP, _IP, _IP, _IP, C.c_int]),
    "sphsm_get_probe_trace": (C.c_int, [_H, C.c_int, _IP, _IP, _FP, _U8P]),
    "sphsm_egm_start": (C.c_int, [_H, _FP, C.c_int, C.c_float, C.c_float, C.c_int]),
    "sphsm_egm_stop": (C.c_int, [_H]),
    "sphsm_egm_reset": (C.c_int, [_H]),
    "sphsm_get_egm": (C.c_int, [_H, C.c_int, _IP, _IP, _DP]),
    "sphsm_tune": (C.c_int, [C.c_char_p, C.c_int]),
    "sphsm_last_error": (C.c_char_p, [_H]),
}

_lib = None


def load():
    """dlopen the in-tree CUDA library and type every entry point.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m sph_sm_monodomain_b200.build` "
            "(there is no CPU fallback for the SPH/SM/monodomain step)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    assert lib.sphsm_abi_version() == 1
    _lib = lib
    return lib


class SphsmError(RuntimeError):
    pass


def check(lib, handle, rc):
    if rc != 0:
        msg = lib.sphsm_last_error(handle)
        raise SphsmError(f"sphsm error {rc}: {msg.decode() if msg else ''}")
