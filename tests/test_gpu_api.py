"""GPU: behaviour of the class-level API (init, stimulation / fixation control, accessors, error paths) against the
oracle, plus size-independent properties of the neighbour search at sizes the oracle cannot reach."""
import ctypes as C

import numpy as np
import pytest

from oracle import CpuSim
from sph_sm_monodomain_b200 import inputs
from tests.common import bits_equal, load_golden

pytestmark = pytest.mark.gpu

FIELDS = ["pos", "vel", "predicted_vel", "inter_vel", "corrected_vel", "acc", "mass", "orig", "goal", "fixed", "dens", "pres",
          "Vm", "Inter_Vm", "Iion", "stim", "w"]


@pytest.fixture(scope="module")
def Sim():
    from sph_sm_monodomain_b200 import Sim as S

    return S


def both(Sim, pos, **kw):
    a, b = CpuSim("port", **kw), Sim(**kw)
    a.Init_Fluid(pos)
    b.Init_Fluid(pos)
    return a, b


def same(a, b, fields=FIELDS):
    pa, pb = a.particles(), b.particles()
    return [f for f in fields if not bits_equal(pa[f], pb[f])]


def test_init_fluid_matches_reference_and_drops_overflow(Sim):
    pos = inputs.init_cube_positions()
    a, b = both(Sim, pos, capacity=3000)
    assert a.n == b.n == 3000  # cpp:103: particles beyond Max_Number_Paticles are silently dropped
    assert same(a, b) == []
    b.Init_Fluid(pos[:10])
    assert b.n == 3000


def test_init_fluid_appends(Sim):
    pos = inputs.init_cube_positions()
    a, b = both(Sim, pos[:1000])
    a.Init_Fluid(pos[1000:1500])
    b.Init_Fluid(pos[1000:1500])
    assert a.n == b.n == 1500 and same(a, b) == []


def test_stim_mesh_cube_setstim_off(Sim):
    g, _ = load_golden("cfg1_4944")
    pos = g["positions"]
    a, b = both(Sim, pos)
    a.turnOnStim_Mesh(pos)
    b.turnOnStim_Mesh(pos)
    assert same(a, b) == [] and a.particles()["fixed"].sum() == 1675
    a.turnOffStim()
    b.turnOffStim()
    assert same(a, b) == []
    cube = inputs.init_cube_positions()
    a, b = both(Sim, cube)
    a.turnOnStim_Cube(cube)
    b.turnOnStim_Cube(cube)
    assert same(a, b) == []
    p = b.particles()
    assert p["fixed"].sum() == 34 and (p["stim"] > 0).sum() == 578  # SURVEY.md §8c
    # set_stim compares the SQUARED distance with `radius` (Q11)
    a, b = both(Sim, cube)
    for s in (a, b):
        s.set_stim((0.6, 0.1, 0.6), 0.004, 123.0)
    assert same(a, b) == [] and 0 < (b.particles()["stim"] == 123.0).sum() < len(cube)


def test_aos_round_trip_and_positions(Sim):
    rng = np.random.Generator(np.random.PCG64(5))
    g, _ = load_golden("cube_4913")
    a, b = both(Sim, g["positions"])
    p = a.particles().copy()
    for f in FIELDS:
        if f == "fixed":
            p[f] = rng.integers(0, 2, len(p))
        else:
            p[f] = rng.random(p[f].shape, dtype=np.float32) + np.float32(0.25)
    b.upload(p)
    q = b.particles()
    for f in FIELDS:
        assert bits_equal(p[f], q[f]), f
    assert bits_equal(b.positions(), p["pos"])
    # order survives a re-sort: Find_neighbors permutes the device arrays, the caller's order must not change
    b.stage("Find_neighbors")
    q = b.particles()
    for f in FIELDS:
        assert bits_equal(p[f], q[f]), f


def test_fixed_particles_keep_goal_and_predicted_velocity(Sim):
    """mFixed particles never get predicted_vel / mGoalPos rewritten (cpp:228,326): values uploaded for them persist."""
    g, _ = load_golden("cube_4913")
    a, b = both(Sim, g["positions"])
    a.turnOnStim_Cube(g["positions"])
    p = a.particles()
    fixed = p["fixed"] != 0
    p["predicted_vel"][fixed] = np.float32([0.25, -0.5, 0.125])
    p["goal"][fixed] += np.float32(0.01)
    b.upload(p)
    a.Animation(3)
    b.Animation(3)
    pa, pb = a.particles(), b.particles()
    assert bits_equal(pa["predicted_vel"][fixed], pb["predicted_vel"][fixed])
    assert bits_equal(pa["goal"][fixed], pb["goal"][fixed])
    assert np.abs(pa["pos"] - pb["pos"]).max() < 1e-5


def test_parameter_toggles(Sim):
    b = Sim()
    assert b.flip_quadratic() is True and b.flip_quadratic() is False
    assert b.flip_volume() is False and b.flip_volume() is True
    a = CpuSim("port")
    for v in (-30.0, -500.0, 12.5):
        a.add_viscosity(v)
        b.add_viscosity(v)
        assert np.float32(b.get_params().mu) == a.constants()["mu"]
    assert b.Get_stand_dens() == 1112.0 and b.Get_World_Size() == (1.5, 1.5, 1.5)
    assert b.num_cells == 54872


def test_error_paths(Sim):
    from sph_sm_monodomain_b200 import SphsmError, _capi

    lib = _capi.load()
    p = _capi.Params()
    lib.sphsm_default_params(p)
    h = C.c_void_p()
    p.struct_size = 4
    assert lib.sphsm_create(p, C.byref(h)) == -1 and b"struct_size" in lib.sphsm_last_error(None)
    lib.sphsm_default_params(p)
    p.device = 99
    assert lib.sphsm_create(p, C.byref(h)) == -2
    b = Sim(capacity=100)
    with pytest.raises(SphsmError):
        b.upload(np.zeros(101, dtype=b.particles().dtype))
    with pytest.raises(SphsmError):
        b.stage(42)
    with pytest.raises(SphsmError):
        b.set_params(kernel_h=0.05)
    b.Animation(3)  # zero particles: a no-op, like the reference's empty loops
    assert b.n == 0 and b.total_time_steps == 3


def test_single_particle_and_out_of_grid(Sim):
    """N == 1: projectPositions returns early (cpp:236) and the goal stays; isolated-particle density is 9791.76."""
    a, b = both(Sim, np.asarray([[0.5, 0.5, 0.5]], np.float32))
    for s in (a, b):
        s.set_stim((0.5, 0.5, 0.5), 0.01, 300.0)
        s.Animation(4)
    pa, pb = a.particles(), b.particles()
    assert pb["dens"][0] == pytest.approx(9791.76, rel=1e-6)
    for f in ("pos", "vel", "goal", "dens", "pres", "Vm"):
        assert np.allclose(pa[f], pb[f], rtol=1e-6, atol=1e-9), f


def test_walls_reflect_and_clamp(Sim):
    rng = np.random.Generator(np.random.PCG64(11))
    n = 600
    pos = (rng.random((n, 3), dtype=np.float32) * np.float32(1.5)).astype(np.float32)
    vel = (rng.standard_normal((n, 3)) * 40).astype(np.float32)
    a, b = both(Sim, pos)
    for s in (a, b):
        s.set_fields(vel=vel, stim=np.full(n, 300, np.float32))
    c = Sim(strict=True)
    c.upload(b.particles())
    a.Animation(25)
    c.Animation(25)
    pa, pc = a.particles(), c.particles()
    for f in ("pos", "vel", "Vm", "dens"):
        assert bits_equal(pa[f], pc[f]), f
    assert pc["pos"].min() >= 0.0 and pc["pos"].max() <= 1.5


# ---- properties at sizes the oracle cannot reach ----------------------------------------------------------------
@pytest.mark.parametrize("n,world", [(1_000_000, (3.68, 3.68, 3.68)), (300_000, (18.52, 4.6, 4.6))])
def test_large_random_cloud_grid_properties(Sim, n, world):
    """Cell table of large random clouds: 1M particles in 0.8M padded cells take the counting sort, 300k particles in 6.3M
    padded cells the three-pass LSD radix sort.  The CSR is a permutation, every particle sits in the bucket numpy computes for
    it, buckets are ascending, and sampled candidate sets equal brute force."""
    rng = np.random.Generator(np.random.PCG64(17))
    w = np.asarray(world, np.float32)
    pos = (rng.random((n, 3), dtype=np.float32) * (w - np.float32(0.001))).astype(np.float32)
    sim = Sim(capacity=n, world=world, diagnostics=False)
    sim.Init_Fluid(pos)
    sim.stage("Find_neighbors")
    start, idx = sim.cells_csr()
    assert start[-1] == n and np.array_equal(np.sort(idx), np.arange(n))
    h = np.float32(0.04)
    cell = (pos / h).astype(np.int32)
    G = np.ceil(w / h).astype(np.int64)
    hsh = cell[:, 0] + G[0] * (cell[:, 1] + G[1] * cell[:, 2])
    owner = np.repeat(np.arange(len(start) - 1), np.diff(start))
    assert np.array_equal(hsh[idx], owner)
    same_cell = owner[1:] == owner[:-1]
    assert np.all(idx[1:][same_cell] > idx[:-1][same_cell])
    query = rng.integers(0, n, 64).astype(np.int32)
    got = sim.neighbor_sets(query, 0, cap=2048)
    for q, gq in zip(query, got):
        near = np.all(np.abs(cell - cell[q]) <= 1, axis=1)
        assert np.array_equal(gq, np.flatnonzero(near)), int(q)
    assert bits_equal(sim.positions(), pos)


def test_async_io_matches_sync(Sim):
    """set_masks_async / download_positions_async (copy streams beside the compute stream) give exactly what the
    synchronous calls give, step after step, also when calls are queued back to back without waiting."""
    from sph_sm_monodomain_b200 import inputs

    pos, world = inputs.lattice(24, 10, 12, jitter=0.05)
    n = len(pos)
    rng = np.random.default_rng(5)
    a = Sim(capacity=n, world=world, diagnostics=False)
    b = Sim(capacity=n, world=world, diagnostics=False)
    for s in (a, b):
        s.Init_Fluid(pos)
    outs = [np.zeros((n, 3), np.float32) for _ in range(6)]
    stims = [np.where(rng.random(n) < 0.2, np.float32(300), np.float32(0)).astype(np.float32) for _ in range(6)]
    fixed = (rng.random(n) < 0.05).astype(np.uint8)
    a.set_masks(fixed, None)
    b.set_masks_async(fixed, None)
    ref = []
    for k in range(6):
        a.set_masks(None, stims[k])
        a.Animation(3)
        ref.append(a.positions())
    for k in range(6):  # queued without waiting: every buffer is distinct and stays alive
        b.set_masks_async(None, stims[k])
        b.Animation(3)
        b.download_positions_async(outs[k])
    b.io_wait()
    for k in range(6):
        assert np.array_equal(outs[k], ref[k]), k


@pytest.mark.parametrize("strict", [True, False], ids=["strict", "fast"])
def test_snapshot_restart(Sim, tmp_path, strict):
    """save_state / load_state: a run restarted from a snapshot continues like the uninterrupted one — bit for bit in strict
    mode (sequential sums in original particle order); within 1e-6 of the field scale on the fast path, whose moment sums
    are grouped by slot order (the restarted run begins in original order, the uninterrupted one in cell order)."""
    g, kw = load_golden("lattice_24x10x12")
    pos = g["positions"]
    a = Sim(strict=strict, **kw)
    a.Init_Fluid(pos)
    a.set_fields(fixed=g["init.fixed"], stim=g["init.stim"])
    a.add_viscosity(0.25)
    a.Animation(7)
    path = tmp_path / "state.sphsm"
    a.save_state(path)
    a.Animation(9)
    b = Sim(strict=strict, **kw)
    b.load_state(path)
    assert b.n == a.n and b.lib.sphsm_total_time_steps(b.h) == 7
    assert b.get_params().mu == a.get_params().mu
    b.Animation(9)
    pa, pb = a.particles(), b.particles()
    for f in ("pos", "vel", "dens", "Vm", "Iion", "w", "stim", "fixed", "orig", "mass"):
        if strict:
            assert bits_equal(pa[f], pb[f]), f
        else:
            scale = max(1e-30, float(np.abs(pa[f].astype(np.float64)).max()))
            assert float(np.abs(pa[f].astype(np.float64) - pb[f].astype(np.float64)).max()) <= 1e-6 * scale, f
    small = Sim(capacity=100, world=kw["world"])
    with pytest.raises(Exception):
        small.load_state(path)  # more particles than capacity
    with pytest.raises(Exception):
        b.load_state(tmp_path / "missing.sphsm")


def test_prefiled_sort_counts_are_dropped_when_particles_move_elsewhere(Sim):
    """On the single-GPU fast path pass B files the next step's counting-sort input (key / rank / per-cell count).  Anything
    else that moves or replaces particles between two steps (the staged Update_Properties, Init_Fluid appending particles,
    upload of a new state) must void it.  Reference: the same call sequence on the radix-sort path (params.reserved[2] = 1),
    which never pre-files; the two differ only by summation order inside cells."""
    g, kw = load_golden("lattice_24x10x12")
    pos = g["positions"]
    n = len(pos)
    extra = (pos[:200] + np.float32(0.011)).astype(np.float32)

    def run(mode):
        s = Sim(capacity=n + 400, world=kw["world"], diagnostics=False)
        p = s.get_params()
        p.reserved[2] = mode
        s._ck(s.lib.sphsm_set_params(s.h, p))
        s.Init_Fluid(pos)
        s.set_fields(fixed=g["init.fixed"], stim=g["init.stim"])
        s.Animation(3)
        for st in range(1, 8):  # one staged step: stage 7 moves the particles behind pass B's back
            s.stage(st)
        s.Animation(2)
        s.cells_csr()           # consumes the pre-filed counts; the next step must count again
        s.Animation(2)
        s.Init_Fluid(extra)     # appends particles
        s.Animation(2)
        st8 = s.particles()
        s.upload(st8)           # replaces the state (same values)
        s.Animation(2)
        return s.particles()

    a, b = run(0), run(1)
    assert len(a) == n + 200
    for f in ("pos", "vel", "dens", "Vm"):
        scale = max(1e-30, float(np.abs(b[f].astype(np.float64)).max()))
        assert float(np.abs(a[f].astype(np.float64) - b[f].astype(np.float64)).max()) <= 2e-5 * scale, f


@pytest.mark.parametrize("name", ["lattice_24x10x12", "cfg2_5211_wave"])
def test_graph_replay_is_bit_identical(Sim, name):
    """Small single-GPU steps are captured into CUDA graphs and replayed (params.reserved[4] = 1 turns that off).  A replayed
    step launches exactly the kernels of the eager step, so the state must agree BIT FOR BIT — also across everything that
    changes what a step launches or reads: mask updates (rest-state sums become dirty), parameter changes (new device parameter
    block), appended particles, staged calls and downloads in between."""
    g, kw = load_golden(name)
    pos = g["positions"]
    extra = (pos[:50] + np.float32(0.013)).astype(np.float32)
    if "capacity" in kw:
        kw = dict(kw, capacity=kw["capacity"] + 100)
    rng = np.random.default_rng(11)
    stim2 = np.where(rng.random(len(pos)) < 0.3, np.float32(300), np.float32(0)).astype(np.float32)
    fixed2 = (rng.random(len(pos)) < 0.03).astype(np.uint8)

    def run(graphs_off):
        s = Sim(diagnostics=False, **kw)
        p = s.get_params()
        p.reserved[4] = 1 if graphs_off else 0
        s._ck(s.lib.sphsm_set_params(s.h, p))
        s.Init_Fluid(pos)
        s.set_fields(fixed=g["init.fixed"], stim=g["init.stim"])
        snaps = []
        s.Animation(12)
        snaps.append(s.positions())
        s.set_masks(None, stim2)       # stimulation only: graphs stay valid
        s.Animation(7)
        s.set_masks(fixed2, None)      # fixed flags: rest-state sums are recomputed by one eager step
        s.Animation(7)
        snaps.append(s.positions())
        s.add_viscosity(0.5)           # new parameter block
        s.Animation(6)
        s.stage("Find_neighbors")      # a staged call between steps
        s.cells_csr()
        s.Animation(5)
        s.Init_Fluid(extra)            # more particles
        s.Animation(9)
        snaps.append(s.positions())
        return snaps, s.particles()

    (sa, a), (sb, b) = run(True), run(False)
    for x, y in zip(sa, sb):
        assert bits_equal(x, y)
    for f in ("pos", "vel", "dens", "pres", "Vm", "Iion", "w", "stim", "fixed", "orig", "mass"):
        assert bits_equal(a[f], b[f]), f


@pytest.mark.parametrize("mode", ["fast", "diagnostics", "strict"])
def test_midrun_fixation_matches_oracle(Sim, mode, parity_record):
    """A particle fixed BETWEEN steps freezes at the mGoalPos / predicted_vel the last step computed for it (the reference just
    stops updating them, cpp:228, 326) — also on the fast path without diagnostics, which does not keep those two arrays: the
    library recomputes them from the last step's transform and the velocity the particle had before that step."""
    from tests.test_gpu_parity import TOL, assert_close, make_params

    g, _ = load_golden("cube_4913")
    pos = g["positions"]
    ora = CpuSim("port")
    sim = Sim(diagnostics=(mode != "fast"), strict=(mode == "strict"))
    for s in (ora, sim):
        s.Init_Fluid(pos)
        s.turnOnStim_Cube(pos)
        s.Animation(4)
    rng = np.random.default_rng(5)
    newly = (rng.random(len(pos)) < 0.08) & (g["init.fixed"] == 0)
    fixed = ((g["init.fixed"] != 0) | newly).astype(np.uint8)
    ora.set_fields(fixed=fixed)
    sim.set_masks(fixed, None)
    params = make_params(g)
    for step in range(3):
        ora.Animation(1)
        sim.Animation(1)
        got, want = sim.particles(), ora.particles()
        assert np.array_equal(got["fixed"], want["fixed"])
        if mode == "strict":
            for f in ("goal", "predicted_vel", "pos", "vel", "dens", "Vm"):
                assert bits_equal(got[f], want[f]), (step, f)
            continue
        for f in ("goal", "predicted_vel"):  # frozen values of the newly fixed particles
            err = assert_close(f, got[f][newly], want[f][newly], params, tol=100 * TOL)
            parity_record("midrun_fixation", f"{mode}/step{step + 1}", f + "(newly fixed)", err, 100 * TOL)
        for f in ("pos", "dens", "Vm", "corrected_vel", "inter_vel"):
            tol = (1e-3 if f in ("corrected_vel", "inter_vel") else TOL) * 100
            err = assert_close(f, got[f], want[f], params, tol=tol)
            parity_record("midrun_fixation", f"{mode}/step{step + 1}", f, err, tol)
    assert np.abs(want["predicted_vel"][newly]).max() > 1e-3  # the case is not vacuous: they were moving when they froze
