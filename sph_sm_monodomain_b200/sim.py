"""Host-side mirror of the reference's ``SPH_SM_monodomain`` class (SPH_SM_monodomain.h:29-168) over the C-ABI.

Same method names, argument meaning and (silent) error behaviour as the reference class so that the parity tests
read like calls on the reference object; all numerical work happens in libsphsm_b200.so on the GPU.  The C++
drop-in with the identical surface is include/SPH_SM_monodomain.h.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi, slabs
from ._capi import Params, SphsmError  # noqa: F401

# the reference's Particle layout (Particle.h:7-35), 132 bytes
PARTICLE_DTYPE = np.dtype(
    [
        ("pos", "<f4", 3), ("vel", "<f4", 3), ("predicted_vel", "<f4", 3), ("inter_vel", "<f4", 3),
        ("corrected_vel", "<f4", 3), ("acc", "<f4", 3), ("mass", "<f4"), ("orig", "<f4", 3), ("goal", "<f4", 3),
        ("fixed", "u1"), ("_pad", "u1", 3), ("dens", "<f4"), ("pres", "<f4"), ("Vm", "<f4"), ("Inter_Vm", "<f4"),
        ("Iion", "<f4"), ("stim", "<f4"), ("w", "<f4"),
    ]
)
assert PARTICLE_DTYPE.itemsize == _capi.PARTICLE_STRIDE

STAGES = {
    "step": 0, "Find_neighbors": 1, "calculate_corrected_velocity": 2, "calculate_intermediate_velocity": 3,
    "Compute_Density_SingPressure": 4, "calculate_cell_model": 5, "Compute_Force": 6, "Update_Properties": 7,
}


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def tune(name: str, value: int):
    """sphsm_tune: process-wide switch "warp_path" (1 | 0) or "x1_dynamic" (0 | 1); the first value is the default.
    warp_path=0 changes the order of the floating-point sums on small dense sets."""
    lib = _capi.load()
    _capi.check(lib, None, lib.sphsm_tune(name.encode(), int(value)))


def default_params() -> Params:
    lib = _capi.load()
    p = Params()
    _capi.check(lib, None, lib.sphsm_default_params(C.byref(p)))
    return p


class Sim:
    """``SPH_SM_monodomain`` on one B200.

    capacity / world default to the reference ctor's 50000 / (1.5,1.5,1.5) (cpp:19,29).  ``diagnostics=True``
    (default, = the drop-in behaviour) keeps every Particle field current after each step; ``False`` runs the fused
    fast path that only maintains persistent state.  ``strict=True`` selects the reference-order arithmetic.
    """

    def __init__(self, capacity=50000, world=(1.5, 1.5, 1.5), device=0, diagnostics=True, strict=False, slab_axis=-1, **overrides):
        self.lib = _capi.load()
        p = default_params()
        p.capacity = int(capacity)
        p.world[:] = [float(w) for w in world]
        p.device = int(device)
        p.diagnostics = int(bool(diagnostics))
        p.strict = int(bool(strict))
        p.slab_axis = int(slab_axis)
        for k, v in overrides.items():
            if k == "halo_capacity":  # params.reserved[0]: particles per halo / migrant message (0 = default)
                p.reserved[0] = int(v)
            else:
                setattr(p, k, v)
        self.h = C.c_void_p()
        _capi.check(self.lib, None, self.lib.sphsm_create(C.byref(p), C.byref(self.h)))
        self._stage_time = np.zeros(7)

    # ---- lifetime ---------------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.sphsm_destroy(self.h)
            self.h = C.c_void_p()

    __del__ = close

    def _ck(self, rc):
        _capi.check(self.lib, self.h, rc)

    # ---- parameters -------------------------------------------------------------------------------------
    def get_params(self) -> Params:
        p = Params()
        self._ck(self.lib.sphsm_get_params(self.h, C.byref(p)))
        return p

    def set_params(self, **kw):
        p = self.get_params()
        for k, v in kw.items():
            setattr(p, k, v)
        self._ck(self.lib.sphsm_set_params(self.h, C.byref(p)))

    def flip_quadratic(self):  # h:154
        q = not self.get_params().quadratic_match
        self.set_params(quadratic_match=int(q))
        return q

    def flip_volume(self):  # h:155
        v = not self.get_params().volume_conservation
        self.set_params(volume_conservation=int(v))
        return v

    def add_viscosity(self, value):  # cpp:87-91
        mu = np.float32(self.get_params().mu)
        value = np.float32(value)
        self.set_params(mu=float(mu + (value if (mu + value) >= 0 else np.float32(0))))

    # ---- init / control ---------------------------------------------------------------------------------
    def Init_Fluid(self, positions):  # cpp:93-99
        p = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        self._ck(self.lib.sphsm_init_fluid(self.h, _fp(p), len(p)))

    def set_stim(self, center, radius, strength):  # cpp:704-717
        self._ck(self.lib.sphsm_set_stim(self.h, float(center[0]), float(center[1]), float(center[2]), float(radius), float(strength)))

    def turnOnStim_Mesh(self, positions):  # cpp:745-762
        p = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        self._ck(self.lib.sphsm_stim_mesh(self.h, _fp(p), len(p)))

    def turnOnStim_Cube(self, positions):  # cpp:719-743
        p = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        self._ck(self.lib.sphsm_stim_cube(self.h, _fp(p), len(p)))

    def set_stim_box(self, lo, hi, strength):
        """set_stim for every particle inside the box [lo, hi] (sphsm_set_stim_box)."""
        a, b = np.asarray(lo, np.float32), np.asarray(hi, np.float32)
        self._ck(self.lib.sphsm_set_stim_box(self.h, _fp(a), _fp(b), float(strength)))

    def timer_mark(self, which):
        self._ck(self.lib.sphsm_timer_mark(self.h, int(which)))

    def timer_ms(self):
        v = C.c_float()
        self._ck(self.lib.sphsm_timer_ms(self.h, C.byref(v)))
        return v.value

    def turnOffStim(self):  # cpp:764-783
        self._ck(self.lib.sphsm_stim_off(self.h))

    def set_masks(self, fixed=None, stim=None):
        f = None if fixed is None else np.ascontiguousarray(np.asarray(fixed).astype(np.uint8))
        s = None if stim is None else np.ascontiguousarray(stim, dtype=np.float32)
        n = len(f) if f is not None else (len(s) if s is not None else self.n)  # slab mode: the GLOBAL count (ids are global)
        self._ck(self.lib.sphsm_set_masks(self.h, None if f is None else f.ctypes.data_as(C.POINTER(C.c_uint8)),
                                          None if s is None else _fp(s), n))

    def set_masks_async(self, fixed=None, stim=None):
        """sphsm_set_masks_async: the arrays (ideally page-locked) must stay alive and untouched until io_wait() / sync()."""
        n = len(fixed) if fixed is not None else (len(stim) if stim is not None else self.n)
        assert fixed is None or (fixed.dtype == np.uint8 and fixed.flags.c_contiguous)
        assert stim is None or (stim.dtype == np.float32 and stim.flags.c_contiguous)
        self._ck(self.lib.sphsm_set_masks_async(self.h, None if fixed is None else fixed.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                None if stim is None else _fp(stim), n))

    def download_positions_async(self, out):
        """sphsm_download_positions_async into `out` ((n, 3) float32, ideally page-locked); valid after io_wait() / sync()."""
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size >= 3 * self.n
        self._ck(self.lib.sphsm_download_positions_async(self.h, _fp(out), self.n))

    def io_wait(self):
        self._ck(self.lib.sphsm_io_wait(self.h))

    def save_state(self, path):
        self._ck(self.lib.sphsm_save_state(self.h, str(path).encode()))

    def load_state(self, path):
        self._ck(self.lib.sphsm_load_state(self.h, str(path).encode()))

    def set_fields(self, **fields):
        """Overwrite per-particle fields (what reference callers do by writing through Get_Paticles())."""
        if set(fields) <= {"fixed", "stim"}:
            return self.set_masks(fields.get("fixed"), fields.get("stim"))
        p = self.particles()
        for k, v in fields.items():
            p[k] = v
        self.upload(p)

    # ---- stepping ---------------------------------------------------------------------------------------
    def Animation(self, nsteps=1):  # cpp:826-829
        self._ck(self.lib.sphsm_step(self.h, int(nsteps)))

    compute_SPH_SM_monodomain = Animation

    def stage(self, name_or_id):
        sid = STAGES[name_or_id] if isinstance(name_or_id, str) else int(name_or_id)
        self._ck(self.lib.sphsm_stage(self.h, sid))

    def Find_neighbors(self): self.stage(1)  # noqa: E704
    def calculate_corrected_velocity(self): self.stage(2)  # noqa: E704
    def calculate_intermediate_velocity(self): self.stage(3)  # noqa: E704
    def Compute_Density_SingPressure(self): self.stage(4)  # noqa: E704
    def calculate_cell_model(self): self.stage(5)  # noqa: E704
    def Compute_Force(self): self.stage(6)  # noqa: E704
    def Update_Properties(self): self.stage(7)  # noqa: E704

    def sync(self):
        self._ck(self.lib.sphsm_sync(self.h))

    # ---- accessors --------------------------------------------------------------------------------------
    @property
    def n(self):
        return self.lib.sphsm_num_particles(self.h)

    def Get_Particle_Number(self):  # h:148
        return self.n

    @property
    def num_cells(self):
        return self.lib.sphsm_num_cells(self.h)

    def Get_World_Size(self):  # h:149
        return tuple(self.get_params().world)

    def Get_stand_dens(self):  # h:152
        return self.get_params().stand_density

    @property
    def total_time_steps(self):  # h:101
        return self.lib.sphsm_total_time_steps(self.h)

    def particles(self):
        """Get_Paticles() (h:150): a host copy of the AoS array in the caller's particle order."""
        n = self.n
        out = np.zeros(n, dtype=PARTICLE_DTYPE)
        if n:
            self._ck(self.lib.sphsm_download_aos(self.h, out.ctypes.data_as(C.c_void_p), n, PARTICLE_DTYPE.itemsize))
        return out

    Get_Paticles = particles

    def positions(self):
        n = self.n
        out = np.zeros((n, 3), np.float32)
        if n:
            self._ck(self.lib.sphsm_download_positions(self.h, _fp(out), n))
        return out

    def upload(self, particles):
        p = np.ascontiguousarray(particles)
        assert p.dtype.itemsize >= PARTICLE_DTYPE.itemsize
        self._ck(self.lib.sphsm_upload_aos(self.h, p.ctypes.data_as(C.c_void_p), len(p), p.dtype.itemsize))

    def cells_csr(self):
        nc, n = self.num_cells, self.n
        start = np.zeros(nc + 1, np.int32)
        idx = np.zeros(max(n, 1), np.int32)
        self._ck(self.lib.sphsm_get_cells_csr(self.h, _ip(start), _ip(idx)))
        return start, idx[: start[-1]]

    def neighbor_sets(self, query, kind, cap=512):
        q = np.ascontiguousarray(query, dtype=np.int32)
        counts = np.zeros(len(q), np.int32)
        idx = np.zeros((len(q), cap), np.int32)
        self._ck(self.lib.sphsm_get_neighbor_sets(self.h, int(kind), _ip(q), len(q), cap, _ip(counts), _ip(idx)))
        assert counts.max(initial=0) <= cap, "neighbour list capacity exceeded"
        return [idx[i, : counts[i]].copy() for i in range(len(q))]

    def sm_transform(self):
        cm, ocm, x = np.zeros(3, np.float32), np.zeros(3, np.float32), np.zeros(27, np.float32)
        self._ck(self.lib.sphsm_get_sm_transform(self.h, _fp(cm), _fp(ocm), _fp(x)))
        return cm, ocm, x

    # ---- multi-GPU slab layer (no reference counterpart; include/sphsm_b200.h) ---------------------------------------
    @staticmethod
    def comm_unique_id() -> bytes:
        lib = _capi.load()
        buf = C.create_string_buffer(128)
        _capi.check(lib, None, lib.sphsm_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, nranks, rank, unique_id: bytes):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._ck(self.lib.sphsm_comm_init(self.h, int(nranks), int(rank), buf))

    def set_slab(self, lo, hi):
        if not self.comm_info()["slab_on"]:
            self._n_global = self.n  # (every rank holds the whole set until its first slab is applied; ids stay global)
        self._ck(self.lib.sphsm_comm_set_slab(self.h, int(lo), int(hi)))

    def comm_info(self):
        out = np.zeros(8, np.int32)
        self._ck(self.lib.sphsm_comm_info(self.h, _ip(out)))
        keys = ("mode", "nranks", "rank", "n_local", "own_begin", "own_end", "halo_capacity", "slab_on")
        return dict(zip(keys, (int(v) for v in out)))

    def push_exchange(self):
        """True when exchange 1 runs as direct stores into the neighbours' memory (CUDA IPC over NVLink) instead of ncclSend / ncclRecv."""
        return bool(self.lib.sphsm_comm_p2p(self.h) & 1)

    def push_allreduce(self):
        """True when the small allreduces of the slab step (shape-matching moment sums + error flag) run as the one-kernel push allreduce
        over the same IPC mappings instead of ncclAllReduce."""
        return bool(self.lib.sphsm_comm_p2p(self.h) & 2)

    def x1_sizes(self):
        """Capacities (particles) of the exchange-1 messages packed last: to left, to right, from left, from right."""
        out = np.zeros(4, np.int32)
        self._ck(self.lib.sphsm_comm_x1_sizes(self.h, _ip(out)))
        return tuple(int(v) for v in out)

    def download_owned(self):
        """(ids, positions) of the particles this rank owns (all particles on a single GPU)."""
        cap = max(self.n, 1)
        ids = np.zeros(cap, np.int32)
        xyz = np.zeros((cap, 3), np.float32)
        cnt = C.c_int()
        self._ck(self.lib.sphsm_download_owned(self.h, _ip(ids), _fp(xyz), cap, C.byref(cnt)))
        return ids[: cnt.value].copy(), xyz[: cnt.value].copy()

    # ---- recorder of the Vm wave (include/sphsm_b200.h: sphsm_record_*) ------------------------------------------------
    def record_start(self, vm_up, vm_down=None, probes=None, trace_rows=0):
        """Record activation / recovery times (Vm rising through vm_up, falling through vm_down; vm_down defaults to vm_up) of
        every particle and, for the original ids in `probes`, (pos, Vm) after every step in a ring of `trace_rows` rows."""
        ids = np.ascontiguousarray(np.asarray([] if probes is None else probes, dtype=np.int32).ravel())
        down = vm_up if vm_down is None else vm_down
        self._ck(self.lib.sphsm_record_start(self.h, float(vm_up), float(down), _ip(ids) if len(ids) else None, len(ids), int(trace_rows)))
        self._probes, self._trace_rows = ids.copy(), int(trace_rows)

    def record_stop(self):
        self._ck(self.lib.sphsm_record_stop(self.h))

    def record_reset(self):
        self._ck(self.lib.sphsm_record_reset(self.h))

    def activation(self, n=None):
        """{"first_up", "last_up", "last_down", "n_up"}: int32 arrays by original id (n = the particle count, global in slab mode);
        steps never seen are -1."""
        if n is None:
            n = self._n_global if self.comm_info()["slab_on"] else self.n
        out = {k: np.zeros(n, np.int32) for k in ("first_up", "last_up", "last_down", "n_up")}
        self._ck(self.lib.sphsm_get_activation(self.h, _ip(out["first_up"]), _ip(out["last_up"]), _ip(out["last_down"]),
                                               _ip(out["n_up"]), int(n)))
        return out

    def probe_trace(self):
        """(first_step, xyzv (rows, K, 4) float32 = (pos.xyz, Vm) after each step, owned (rows, K) bool), oldest row first."""
        k = len(getattr(self, "_probes", ()))
        cap = self._trace_rows if k else 0
        rows, first = C.c_int(), C.c_int()
        xyzv = np.zeros((max(cap, 1), max(k, 1), 4), np.float32)
        owned = np.zeros((max(cap, 1), max(k, 1)), np.uint8)
        self._ck(self.lib.sphsm_get_probe_trace(self.h, cap, C.byref(rows), C.byref(first), _fp(xyzv),
                                                owned.ctypes.data_as(C.POINTER(C.c_uint8))))
        r = rows.value
        return first.value, xyzv[:r, :k].copy(), owned[:r, :k].astype(bool)

    # ---- electrograms at virtual electrodes (include/sphsm_b200.h: sphsm_egm_*) -------------------------------------
    def egm_start(self, electrodes, gain=1.0, softening=None, rows=1024):
        """Every step, phi_e = gain * sum_i vol_i L_i / sqrt(|x_i - e|^2 + softening^2) at each electrode e (an (E, 3) array of
        fixed world positions, E <= 256), kept on the device in a ring of `rows` steps.  softening defaults to kernel_h."""
        el = np.ascontiguousarray(np.asarray(electrodes, dtype=np.float32).reshape(-1, 3))
        eps = self.get_params().kernel_h if softening is None else softening
        self._ck(self.lib.sphsm_egm_start(self.h, _fp(el), len(el), float(gain), float(eps), int(rows)))
        self._egm_shape = (int(rows), len(el))

    def egm_stop(self):
        self._ck(self.lib.sphsm_egm_stop(self.h))

    def egm_reset(self):
        self._ck(self.lib.sphsm_egm_reset(self.h))

    def electrogram(self):
        """(first_step, phi (rows, E) float64), oldest row first: the rows held, up to the ring's length."""
        cap, e = getattr(self, "_egm_shape", (0, 1))
        rows, first = C.c_int(), C.c_int()
        phi = np.zeros((max(cap, 1), e), np.float64)
        self._ck(self.lib.sphsm_get_egm(self.h, cap, C.byref(rows), C.byref(first), phi.ctypes.data_as(C.POINTER(C.c_double))))
        return first.value, phi[: rows.value].copy()

    # ---- timers / counters --------------------------------------------------------------------------------
    def enable_stage_timing(self, on=True):
        self._ck(self.lib.sphsm_enable_stage_timing(self.h, int(on)))

    def stage_times(self):
        out = np.zeros(7, np.float64)
        self._ck(self.lib.sphsm_get_stage_times(self.h, out.ctypes.data_as(C.POINTER(C.c_double))))
        return out

    def launch_count(self):
        v = C.c_longlong()
        self._ck(self.lib.sphsm_get_launch_count(self.h, C.byref(v)))
        return v.value

    def reset_launch_count(self):
        self._ck(self.lib.sphsm_reset_launch_count(self.h))

    def last_step_ms(self):
        v = C.c_float()
        self._ck(self.lib.sphsm_last_step_ms(self.h, C.byref(v)))
        return v.value

    def profile_step(self, nsteps=1):
        out = np.zeros(_capi.NUM_KERNEL_GROUPS, np.float32)
        self._ck(self.lib.sphsm_profile_step(self.h, int(nsteps), _fp(out)))
        return {self.lib.sphsm_kernel_group_name(g).decode(): float(out[g]) for g in range(_capi.NUM_KERNEL_GROUPS)}

    def print_report(self, avg_fps=0.0, avg_step_d=0.0):
        """The reference's 23-field ';'-separated report line (cpp:785-792); stage columns are device seconds/step."""
        p = self.get_params()
        steps = max(self.total_time_steps, 1)
        t = self.stage_times() / steps
        head = [avg_fps, avg_step_d, self.total_time_steps] + list(t)
        tail = [p.K, p.alpha, p.beta, p.mu, p.sigma, p.stim_strength, p.FH_Vt, p.FH_Vp, p.FH_Vr, p.C1, p.C2, p.C3, p.C4]
        line = ";".join(f"{x:g}" for x in head) + ";" + ";".join(f"{x:g}" for x in tail)
        print(line)
        return line


class LocalGroup:
    """Virtual ranks on ONE device (sphsm_comm_init_local / sphsm_step_group): the slab logic of the multi-GPU path with
    device copies in place of NCCL.  Used by the GPU tests; production runs one process per GPU (bench.py)."""

    def __init__(self, sims):
        self.sims = list(sims)
        self.lib = self.sims[0].lib
        self._arr = (C.c_void_p * len(self.sims))(*[s.h for s in self.sims])
        _capi.check(self.lib, self.sims[0].h, self.lib.sphsm_comm_init_local(self._arr, len(self.sims)))

    def step(self, nsteps=1):
        rc = self.lib.sphsm_step_group(self._arr, len(self.sims), int(nsteps))
        if rc:
            msgs = [self.lib.sphsm_last_error(s.h).decode() for s in self.sims]
            raise SphsmError(f"sphsm_step_group failed ({rc}): {msgs}")

    def activation(self, n_global):
        """The recorder's activation maps of every virtual rank, merged (slabs.merge_activation)."""
        return slabs.merge_activation(s.activation(n_global) for s in self.sims)

    def probe_trace(self):
        """The recorder's probe traces of every virtual rank, merged (slabs.merge_traces): (first_step, xyzv, owned)."""
        return slabs.merge_traces(s.probe_trace() for s in self.sims)

    def electrogram(self):
        """The electrograms of every virtual rank, summed in rank order (slabs.merge_electrograms): (first_step, phi)."""
        return slabs.merge_electrograms(s.electrogram() for s in self.sims)

    def gather_positions(self, n_global):
        """Owned particles of every virtual rank assembled by original id; also returns the owner rank per particle."""
        pos = np.full((n_global, 3), np.nan, np.float32)
        owner = np.full(n_global, -1, np.int32)
        for r, s in enumerate(self.sims):
            ids, xyz = s.download_owned()
            assert (owner[ids] == -1).all(), "a particle is owned by two ranks"
            pos[ids] = xyz
            owner[ids] = r
        return pos, owner
