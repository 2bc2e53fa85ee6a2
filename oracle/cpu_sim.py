"""TEST INFRASTRUCTURE ONLY — ctypes front end over the two CPU oracles (see oracle/__init__.py)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))

# Same layout as the reference's `Particle` (Particle.h:7-35), 132 bytes.
PARTICLE_DTYPE = np.dtype(
    [
        ("pos", "<f4", 3), ("vel", "<f4", 3), ("predicted_vel", "<f4", 3), ("inter_vel", "<f4", 3),
        ("corrected_vel", "<f4", 3), ("acc", "<f4", 3), ("mass", "<f4"), ("orig", "<f4", 3), ("goal", "<f4", 3),
        ("fixed", "u1"), ("_pad", "u1", 3), ("dens", "<f4"), ("pres", "<f4"), ("Vm", "<f4"), ("Inter_Vm", "<f4"),
        ("Iion", "<f4"), ("stim", "<f4"), ("w", "<f4"),
    ]
)
assert PARTICLE_DTYPE.itemsize == 132

_LIBS = {
    "port": os.path.join(_HERE, "_build", "libsphsm_oracle.so"),
    "ref": os.path.join(_HERE, "_ref", "libsphsm_ref.so"),
    "ref_ofast": os.path.join(_HERE, "_ref", "libsphsm_ref_ofast.so"),
}
_PREFIX = {"port": "ora_", "ref": "ref_", "ref_ofast": "ref_"}


def lib_path(backend: str) -> str:
    return _LIBS[backend]


def build_oracle(ref: bool = True) -> None:
    """Compile the C restatement, and the genuine reference when $SPHSM_REFERENCE_DIR names a checkout of its sources."""
    subprocess.run(["make", "-C", _HERE, "oracle"], check=True, capture_output=True)
    if not ref:
        return
    ref_dir = os.environ.get("SPHSM_REFERENCE_DIR")
    if ref_dir and os.path.isdir(os.path.join(ref_dir, "SPH_SM_monodomain")):
        subprocess.run(["make", "-C", _HERE, "ref", "ref_ofast", "REF=" + os.path.abspath(ref_dir)], check=True, capture_output=True)
        return
    why = f"$SPHSM_REFERENCE_DIR={ref_dir!r} has no SPH_SM_monodomain/" if ref_dir else "$SPHSM_REFERENCE_DIR is not set"
    sys.stderr.write(f"oracle: genuine reference not built ({why}): the 'ref' back ends are unavailable, the tests compare "
                     "with its stored results only, and bench.py --impl reference times the C restatement\n")


def available_backends():
    if not os.path.exists(_LIBS["port"]):
        build_oracle(ref=False)
    return [b for b, p in _LIBS.items() if os.path.exists(p)]


_loaded = {}


def _load(backend):
    if backend in _loaded:
        return _loaded[backend]
    path = _LIBS[backend]
    if backend == "port" and not os.path.exists(path):
        build_oracle(ref=False)
    if not os.path.exists(path):
        raise FileNotFoundError(f"oracle backend {backend!r} not built: {path}")
    lib = C.CDLL(path)
    pre = _PREFIX[backend]
    f = lambda name: getattr(lib, pre + name)  # noqa: E731
    vp, fp, ip = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)
    sig = {
        "destroy": (None, [vp]),
        "init_fluid": (None, [vp, fp, C.c_int]),
        "stim_mesh": (None, [vp, fp, C.c_int]),
        "stim_cube": (None, [vp, fp, C.c_int]),
        "set_stim": (None, [vp] + [C.c_float] * 5),
        "stim_off": (None, [vp]),
        "flip_quadratic": (C.c_int, [vp]),
        "flip_volume": (C.c_int, [vp]),
        "add_viscosity": (None, [vp, C.c_float]),
        "n": (C.c_int, [vp]),
        "particles": (vp, [vp]),
        "num_cells": (C.c_int, [vp]),
        "stage": (None, [vp, C.c_int]),
        "steps": (None, [vp, C.c_int]),
        "constants": (None, [vp, fp]),
        "cells_csr": (C.c_int, [vp, ip, ip]),
        "cell_hash": (C.c_int, [vp, C.c_float, C.c_float, C.c_float]),
        "poly6": (C.c_float, [vp, C.c_float]),
        "spiky": (C.c_float, [vp, C.c_float]),
        "visco": (C.c_float, [vp, C.c_float]),
        "bspline2": (C.c_float, [vp, C.c_float]),
        "polar3": (None, [fp, fp]),
        "invert3": (C.c_int, [fp]),
        "invert9": (None, [fp]),
    }
    for name, (res, args) in sig.items():
        fn = f(name)
        fn.restype, fn.argtypes = res, args
    if backend == "port":
        lib.ora_create.restype, lib.ora_create.argtypes = vp, [C.c_int, C.c_float, C.c_float, C.c_float]
        lib.ora_set_moments_in_double.restype, lib.ora_set_moments_in_double.argtypes = None, [vp, C.c_int]
        lib.ora_neighbors.restype, lib.ora_neighbors.argtypes = C.c_int, [vp, C.c_int, C.c_int, ip, C.c_int]
        lib.ora_sm_debug.restype, lib.ora_sm_debug.argtypes = None, [vp, fp, fp, fp]
    else:
        lib.ref_create.restype, lib.ref_create.argtypes = vp, []
        lib.ref_resize.restype, lib.ref_resize.argtypes = None, [vp, C.c_int, C.c_float, C.c_float, C.c_float]
        lib.ref_sizeof_particle.restype = C.c_int
        assert lib.ref_sizeof_particle() == PARTICLE_DTYPE.itemsize
    _loaded[backend] = (lib, f)
    return _loaded[backend]


def _fptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


class CpuSim:
    """One CPU simulation object; method names follow the reference class (SPH_SM_monodomain.h:89-155)."""

    STAGES = {
        "step": 0, "Find_neighbors": 1, "calculate_corrected_velocity": 2, "calculate_intermediate_velocity": 3,
        "Compute_Density_SingPressure": 4, "calculate_cell_model": 5, "Compute_Force": 6, "Update_Properties": 7,
    }

    def __init__(self, backend="port", capacity=50000, world=(1.5, 1.5, 1.5), moments_in_double=False):
        self.backend = backend
        self.lib, self._f = _load(backend)
        self.capacity = capacity
        self.world = tuple(float(w) for w in world)
        default = capacity == 50000 and self.world == (1.5, 1.5, 1.5)
        if backend == "port":
            self.h = self.lib.ora_create(capacity, *self.world)
            if moments_in_double:
                self.lib.ora_set_moments_in_double(self.h, 1)
        else:
            if moments_in_double:
                raise ValueError("the genuine reference accumulates in float only")
            self.h = self.lib.ref_create()
            if not default:
                self.lib.ref_resize(self.h, capacity, *self.world)

    def close(self):
        if getattr(self, "h", None):
            self._f("destroy")(self.h)
            self.h = None

    __del__ = close

    # ---- init / control -------------------------------------------------
    def Init_Fluid(self, positions):
        p = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        self._f("init_fluid")(self.h, _fptr(p), len(p))

    def turnOnStim_Mesh(self, positions):
        p = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        self._f("stim_mesh")(self.h, _fptr(p), len(p))

    def turnOnStim_Cube(self, positions):
        p = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        self._f("stim_cube")(self.h, _fptr(p), len(p))

    def set_stim(self, center, radius, strength):
        self._f("set_stim")(self.h, float(center[0]), float(center[1]), float(center[2]), float(radius), float(strength))

    def turnOffStim(self):
        self._f("stim_off")(self.h)

    def flip_quadratic(self):
        return bool(self._f("flip_quadratic")(self.h))

    def flip_volume(self):
        return bool(self._f("flip_volume")(self.h))

    def add_viscosity(self, v):
        self._f("add_viscosity")(self.h, float(v))

    # ---- stepping -------------------------------------------------------
    def stage(self, name_or_id):
        sid = self.STAGES[name_or_id] if isinstance(name_or_id, str) else int(name_or_id)
        self._f("stage")(self.h, sid)

    def Animation(self, nsteps=1):
        self._f("steps")(self.h, int(nsteps))

    # ---- accessors ------------------------------------------------------
    @property
    def n(self):
        return self._f("n")(self.h)

    Get_Particle_Number = lambda self: self.n  # noqa: E731

    @property
    def num_cells(self):
        return self._f("num_cells")(self.h)

    def particles(self):
        """Borrowed, mutable numpy view of the live AoS array (Get_Paticles, h:150)."""
        n = self.n
        ptr = self._f("particles")(self.h)
        buf = (C.c_char * (n * PARTICLE_DTYPE.itemsize)).from_address(ptr)
        return np.frombuffer(buf, dtype=PARTICLE_DTYPE, count=n)

    def set_fields(self, **fields):
        """Overwrite per-particle fields in place (the reference's callers do this through Get_Paticles())."""
        p = self.particles()
        for k, v in fields.items():
            p[k] = v

    def constants(self):
        out = np.zeros(16, np.float32)
        self._f("constants")(self.h, _fptr(out))
        names = ["K", "Stand_Density", "Time_Delta", "mu", "Poly6_constant", "Spiky_constant", "B_spline_constant", "sigma",
                 "alpha", "beta", "kernel", "stim_strength", "velocity_mixing", "Wall_Hit", "Cm", "Beta"]
        return dict(zip(names, out))

    def cells_csr(self):
        nc = self.num_cells
        start = np.zeros(nc + 1, np.int32)
        idx = np.zeros(max(self.n, 1), np.int32)
        tot = self._f("cells_csr")(self.h, start.ctypes.data_as(C.POINTER(C.c_int)), idx.ctypes.data_as(C.POINTER(C.c_int)))
        return start, idx[:tot]

    def cell_hash(self, x, y, z):
        return self._f("cell_hash")(self.h, float(x), float(y), float(z))

    def neighbors(self, i, kind):
        assert self.backend == "port"
        cap = 4096
        out = np.zeros(cap, np.int32)
        cnt = self.lib.ora_neighbors(self.h, int(i), int(kind), out.ctypes.data_as(C.POINTER(C.c_int)), cap)
        assert cnt <= cap
        return out[:cnt].copy()

    def sm_debug(self):
        assert self.backend == "port"
        cm, ocm, x = np.zeros(3, np.float32), np.zeros(3, np.float32), np.zeros(27, np.float32)
        self.lib.ora_sm_debug(self.h, _fptr(cm), _fptr(ocm), _fptr(x))
        return cm, ocm, x

    # ---- scalar kernels / small matrices ---------------------------------
    def Poly6(self, r2):
        return self._f("poly6")(self.h, float(r2))

    def Spiky(self, r):
        return self._f("spiky")(self.h, float(r))

    def Visco(self, r):
        return self._f("visco")(self.h, float(r))

    def B_spline_2(self, r):
        return self._f("bspline2")(self.h, float(r))

    def polar3(self, a):
        a = np.ascontiguousarray(a, np.float32).reshape(9)
        r = np.zeros(9, np.float32)
        self._f("polar3")(_fptr(a), _fptr(r))
        return r.reshape(3, 3)

    def invert3(self, a):
        a = np.array(a, np.float32).reshape(9).copy()
        ok = self._f("invert3")(_fptr(a))
        return bool(ok), a.reshape(3, 3)

    def invert9(self, a):
        a = np.array(a, np.float32).reshape(81).copy()
        self._f("invert9")(_fptr(a))
        return a.reshape(9, 9)
