"""CPU: the C-ABI library loads and exports every symbol include/sphsm_b200.h declares (no compute calls)."""
import os
import re

from sph_sm_monodomain_b200 import _capi, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "sphsm_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return set(re.findall(r"\b(sphsm_[a-z0-9_]+)\s*\(", src))


def test_library_builds_and_exports_header_symbols():
    build.build()
    lib = _capi.load()
    declared = header_symbols()
    assert declared, "no declarations parsed from the header"
    assert declared == set(_capi.SYMBOLS), declared ^ set(_capi.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.sphsm_abi_version() == 1


def test_default_params_match_reference_ctor():
    """sphsm_default_params restates the reference ctor (cpp:13-69); compare with the golden constants."""
    import numpy as np

    p = _capi.Params()
    lib = _capi.load()
    assert lib.sphsm_default_params(p) == 0
    k = dict(np.load(os.path.join(ROOT, "tests", "golden", "kats.npz")))
    ref = dict(zip([str(s) for s in k["const_names"]], k["const_values"]))
    mine = {"K": p.K, "Stand_Density": p.stand_density, "Time_Delta": p.time_delta, "mu": p.mu, "Poly6_constant": p.poly6_constant,
            "Spiky_constant": p.spiky_constant, "B_spline_constant": p.bspline_constant, "sigma": p.sigma, "alpha": p.alpha,
            "beta": p.beta, "kernel": p.kernel_h, "stim_strength": p.stim_strength, "velocity_mixing": p.velocity_mixing,
            "Wall_Hit": p.wall_hit, "Cm": p.Cm, "Beta": p.Beta}
    for name, v in mine.items():
        assert np.float32(v).tobytes() == np.float32(ref[name]).tobytes(), name
    assert p.capacity == 50000 and list(p.world) == [1.5, 1.5, 1.5]
    assert p.struct_size == __import__("ctypes").sizeof(_capi.Params)


def test_tune_accepts_only_the_existing_switches():
    """sphsm_tune (no device needed) takes "warp_path" and "x1_dynamic" at 0 / 1 and rejects every other name or value."""
    lib = _capi.load()
    err_invalid = -1  # SPHSM_ERR_INVALID
    try:
        for name in (b"warp_path", b"x1_dynamic"):
            for value in (0, 1):
                assert lib.sphsm_tune(name, value) == 0, (name, value)
            for value in (-1, 2, 4, 64):
                assert lib.sphsm_tune(name, value) == err_invalid, (name, value)
        for name, value in ((b"pass", 4), (b"pass", 6), (b"stage6", 1), (b"t6", 128), (b"b_step6", 2), (b"no_such_switch", 0)):
            assert lib.sphsm_tune(name, value) == err_invalid, (name, value)
        assert lib.sphsm_tune(None, 0) == err_invalid
    finally:
        assert lib.sphsm_tune(b"warp_path", 1) == 0 and lib.sphsm_tune(b"x1_dynamic", 0) == 0  # the defaults


def test_create_without_gpu_fails_loudly():
    """No CUDA device -> sphsm_create returns an error (no CPU fallback). Skipped where a GPU exists."""
    import ctypes as C

    import pytest
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _capi.load()
    p = _capi.Params()
    lib.sphsm_default_params(p)
    h = C.c_void_p()
    rc = lib.sphsm_create(p, C.byref(h))
    assert rc != 0 and not h.value
    assert lib.sphsm_last_error(None)
