"""GPU: the CUDA step in the regimes the golden sets never reach (tests/regimes.py builds the inputs; tests/test_regimes_cpu.py
shows each one reaches the branch it is named for).

A. The reference's own random clouds (linear / quadratic shape matching, volume conservation on / off), particles thrown at the
   walls and the lifted world, driven through the protocols of tests/test_oracle_vs_ref.py and compared with the reference's
   stored digests: strict mode bit for bit, stage by stage and fused; the fast path from identical state against the restatement.
B. Shape matching far from rest (rotations, a mirror, compressions that reach the volume clamp, stretch, shear, fixed particles,
   singular and nearly singular rest shapes): the transform, goal and velocities against the restatement.
C. The LSD radix-sort grid at 1-4 passes (k_cell_order_fix in strict mode), with particle counts on a SORT_TILE edge, and
   counting-sort cell tables on the SCAN_TILE edges.
D. Particle counts on and next to the launch-geometry boundaries.

Tolerance classes are those of tests/test_gpu_parity.py.  Violent clouds may contain DISCRETE events decided by rounding: a
particle that reaches a wall within an ulp is reflected in one run and not in the other (cpp:620-646).  Such a particle is the
only outlier a comparison admits: only in pos / vel, only in a comparison that ran stage 7, and only when it sits on a wall in
exactly one of the two runs.
"""
import numpy as np
import pytest

from oracle import CpuSim
from tests import regimes as R
from tests.common import STAGE_OUT, bits_equal
from tests.test_gpu_parity import TOL
from tests.test_gpu_scale_parity import acc_bound, per_particle_err
from tests.test_oracle_vs_ref import (CLOUD_STEPS, CLOUDS, FIELDS, GOLDEN, assert_final, digests, lifted_world, pres_is_defined,
                                      random_cloud, walls)

pytestmark = pytest.mark.gpu

DIAG_OFF_FIELDS = ("pos", "vel", "dens", "Vm")
CHECK_STEPS = (0, 6, 11)


@pytest.fixture(scope="module")
def Sim():
    from sph_sm_monodomain_b200 import Sim as S

    return S


@pytest.fixture(scope="module")
def ref():
    return dict(np.load(GOLDEN))


def factory(Sim, **kw0):
    return lambda **kw: Sim(**kw0, **kw)


def params_of(state):
    c = CpuSim("port").constants()
    return {"alpha": float(c["alpha"]), "Time_Delta": float(c["Time_Delta"]), "pos_scale": float(np.abs(state["pos"]).max())}


def on_wall(p, world):
    w = np.float32(world) - np.float32(0.0001)
    return ((p["pos"] == 0.0) | (p["pos"] == w)).any(axis=1)


WALL_EVENT_FIELDS = ("pos", "vel")  # what stage 7's reflection writes (cpp:620-646)


def compare(record, case, f, got, want, params, tol, world=(1.5, 1.5, 1.5), ran_stage7=False):
    """max per-particle §8c error of field f within tol.  Where the comparison ran stage 7, a particle beyond the tolerance in pos / vel
    is admitted only when it was reflected in one run and not in the other (on a wall in exactly one of them; module docstring)."""
    e = per_particle_err(f, got[f], want[f], params)
    bad = np.flatnonzero(e > tol)
    if len(bad):
        event = on_wall(got, world) != on_wall(want, world)
        assert ran_stage7 and f in WALL_EVENT_FIELDS and event[bad].all(), (
            case, f, "particles beyond the tolerance without a wall event", bad[~event[bad]][:5], float(e[bad].max()), tol)
        e = np.delete(e, bad)
        record(case, f + " (wall events excluded)", len(bad), None)
    err = float(e.max(initial=0.0))
    record(case, f, err, tol)
    return err


def assert_bits(got, want, fields, where):
    bad = [f for f in fields if not bits_equal(got[f], want[f])]
    assert bad == [], (where, "fields differing", bad)


def assert_digests(sim, want, mask, where):
    bad = [f for f, g, w, m in zip(FIELDS, digests(sim), want, mask) if m and g != w]
    assert bad == [], (where, "fields differing from the reference", bad)


def gpu_with(Sim, state, quadratic=False, volume=True, **kw):
    s = Sim(**kw)
    if quadratic:
        assert s.flip_quadratic()
    if not volume:
        assert not s.flip_volume()
    s.upload(state)
    return s


def fused_tol(f, quadratic):
    """test_fused_step_vs_double_moment_oracle's classes."""
    return 5e-4 if f == "acc" else (2 * TOL if quadratic else TOL)


def stage_tol(f, quadratic):
    """test_stage_parity_from_identical_state's classes."""
    return 2 * TOL if (quadratic and f in ("goal", "corrected_vel")) else TOL


# ==== A. the reference's random clouds, walls and lifted world ========================================================
@pytest.mark.parametrize("seed,quadratic,volume", CLOUDS)
def test_cloud_strict_staged_equals_reference(Sim, ref, seed, quadratic, volume):
    """Strict mode, the seven stages called one by one: every field digest equals the genuine reference's after every stage."""
    key = f"cloud{seed}"
    want = ref[key + ".digests"]
    mask = np.ones(len(FIELDS), bool)
    for sims, step, st in random_cloud([factory(Sim, strict=True)], seed, quadratic, volume):
        mask[FIELDS.index("pres")] = pres_is_defined(step, st)
        assert_digests(sims[0], want[step, st - 1], mask, (key, step, st))
    assert_final(sims, ref, key)


@pytest.mark.parametrize("seed,quadratic,volume", CLOUDS)
def test_cloud_strict_fused_equals_reference(Sim, ref, seed, quadratic, volume):
    """Strict mode, fused steps with diagnostics: every field digest equals the reference's after stage 7 of each step."""
    key = f"cloud{seed}"
    want = ref[key + ".digests"]
    n = 0
    for sims, step, st in random_cloud([factory(Sim, strict=True)], seed, quadratic, volume, fused=True):
        assert_digests(sims[0], want[step, 6], np.ones(len(FIELDS), bool), (key, step))
        n += 1
    assert n == CLOUD_STEPS
    assert_final(sims, ref, key)


def test_walls_and_lifted_world_strict_equal_reference(Sim, ref):
    sims = walls([factory(Sim, strict=True)])
    assert_digests(sims[0], ref["walls.digests"], np.ones(len(FIELDS), bool), "walls")
    assert_final(sims, ref, "walls")
    sims = lifted_world([factory(Sim, strict=True)])
    assert sims[0].num_cells == int(ref["lifted.num_cells"])
    assert_digests(sims[0], ref["lifted.digests"], np.ones(len(FIELDS), bool), "lifted")
    assert_final(sims, ref, "lifted")


@pytest.mark.parametrize("seed,quadratic,volume", CLOUDS)
def test_cloud_fast_from_identical_state(Sim, seed, quadratic, volume, parity_record):
    """Fast path at steps 0, 6 and 11 of each cloud, from the restatement's state: every stage 2..7 alone against the
    restatement, and one fused step (diagnostics on and off) against the restatement with double moment sums."""
    case = f"cloud{seed}"
    rec = lambda c, f, e, t: parity_record("gpu_regimes.cloud_fast_from_identical_state", c, f, e, t)  # noqa: E731
    stage_sim = None
    for sims, step, st in random_cloud(["port"], seed, quadratic, volume):
        ora = sims[0]
        if step not in CHECK_STEPS:
            continue
        want = ora.particles()
        params = params_of(want)
        if st >= 2:  # the GPU ran stage st from the state the restatement had before it
            got = stage_sim.particles()
            for f in STAGE_OUT[st]:
                compare(rec, f"{case}/step{step}/stage{st}", f, got, want, params, stage_tol(f, quadratic), ran_stage7=st == 7)
        if st == 1:  # stage 1 moves nothing: this is the state at the start of the step
            state = want.copy()
            dbl = R.clone(state, quadratic, volume, moments_in_double=True)
            dbl.Animation(1)
            for diag in (True, False):
                gpu = gpu_with(Sim, state, quadratic, volume, diagnostics=diag)
                gpu.Animation(1)
                got, w = gpu.particles(), dbl.particles()
                fields = [f for s2 in range(2, 8) for f in STAGE_OUT[s2]] if diag else DIAG_OFF_FIELDS
                for f in fields:
                    compare(rec, f"{case}/step{step}/fused" + ("" if diag else "/diagnostics_off"), f, got, w, params, fused_tol(f, quadratic),
                            ran_stage7=True)
        if st < 7:
            stage_sim = gpu_with(Sim, ora.particles().copy(), quadratic, volume)
            stage_sim.stage(st + 1)


# ==== B. shape matching far from rest =================================================================================
SM_FIELDS = ("goal", "predicted_vel", "corrected_vel")
MODES = [(False, True), (False, False), (True, True), (True, False)]
MODE_IDS = ["linear", "linear_volume_off", "quadratic", "quadratic_volume_off"]


BODIES_DEGENERATE = {k: v[3] for k, v in R.BODIES.items()}


def fast_comparable(state, quadratic, volume):
    """(comparable, condition number): the fast path's sums differ from the restatement's in the last bits, and an ill-conditioned
    rest-shape matrix (Aqq, or A9qq in quadratic mode) amplifies that without bound.  Rows that are exactly zero in float are carried
    through exactly by every implementation: an Aqq exactly singular in float takes invert3's failure path (A = Apq Aqq, well
    conditioned) in both, and the truncated Jacobi inverse keeps A9qq's zero rows zero.  So the condition number is taken without
    them (tests/regimes.py reduced_cond)."""
    s, cm, ocm, x = R.solve_state(state, quadratic, volume, dbl=True)
    aqq = R.restatement_aqq(state, ocm)
    cond = R.reduced_cond(R.restatement_a9qq(state, ocm) if quadratic else aqq)
    if cond <= 1e6 and not aqq.any(axis=1).all():
        assert not s.invert3(aqq)[0]  # a zero row: the case takes invert3's failure path
    return cond <= 1e6, cond


def assert_transform(rec, case, got, want, tol):
    for name, g, w in zip(("cm", "ocm", "xform"), got, want):
        e = float(np.abs(g.astype(np.float64) - w).max() / max(float(np.abs(w).max()), 1e-30))
        rec(case, name, e, tol)
        assert e <= tol, (case, name, e, tol, g, w)


@pytest.mark.parametrize("quadratic,volume", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("name", list(R.BODIES))
def test_shape_matching_far_from_rest(Sim, name, quadratic, volume, parity_record):
    """After stage 2 and after one fused step: sm_transform (cm, ocm, the 27 entries) and goal / predicted / corrected velocity
    per particle.  Strict: bit-identical to the restatement.  Fast: TOL of the §8c metric against the double-moment restatement
    (2 TOL on the quadratic goal), on every body whose Aqq is not nearly singular."""
    state = R.body_state(name)
    rec = lambda c, f, e, t: parity_record("gpu_regimes.shape_matching_far_from_rest", c, f, e, t)  # noqa: E731
    case = f"{name}/{MODE_IDS[MODES.index((quadratic, volume))]}"
    # strict
    for fused in (False, True):
        ora = R.clone(state, quadratic, volume)
        gpu = gpu_with(Sim, state, quadratic, volume, strict=True)
        ora.Animation(1) if fused else ora.stage(2)
        gpu.Animation(1) if fused else gpu.stage(2)
        for g, w, what in zip(gpu.sm_transform(), ora.sm_debug(), ("cm", "ocm", "xform")):
            assert bits_equal(g, w), (case, "strict", "fused" if fused else "stage 2", what, g, w)
        assert_bits(gpu.particles(), ora.particles(), SM_FIELDS + (("pos", "vel") if fused else ()), (case, "strict", fused))
    # fast
    ok, cond = fast_comparable(state, quadratic, volume)
    if not ok:
        assert BODIES_DEGENERATE[name] and cond > 1e6  # the only reason a case is strict-only
        return
    params = params_of(state)
    tol_sm = 2 * TOL if quadratic else TOL
    for fused, diag in ((False, True), (True, True), (True, False)):
        ora = R.clone(state, quadratic, volume, moments_in_double=True)
        gpu = gpu_with(Sim, state, quadratic, volume, diagnostics=diag)
        ora.Animation(1) if fused else ora.stage(2)
        gpu.Animation(1) if fused else gpu.stage(2)
        sub = case + ("/fused" if fused else "/stage2") + ("" if diag else "/diagnostics_off")
        assert_transform(rec, sub, gpu.sm_transform(), ora.sm_debug(), tol_sm)
        if diag:
            got, want = gpu.particles(), ora.particles()
            for f in SM_FIELDS:
                compare(rec, sub, f, got, want, params, stage_tol(f, quadratic))


@pytest.mark.parametrize("strict", [False, True], ids=["fast", "strict"])
@pytest.mark.parametrize("change", ["orig", "mass"])
def test_rest_shape_change_invalidates_cached_sums(Sim, change, strict, parity_record):
    """After steps on one rest shape, a new rest shape (or new masses) uploaded between steps: the next step's transform follows
    it.  The fast path caches the rest-state sums (centre, Aqq and their inverses) between steps."""
    rest, pos, fixed = R.body("cube_stretch")
    gpu = Sim(strict=strict, diagnostics=False)
    gpu.Init_Fluid(rest)
    gpu.set_fields(pos=pos)
    gpu.Animation(3)
    state = gpu.particles()
    c = state["orig"].astype(np.float64).mean(axis=0)
    if change == "orig":
        state["orig"] = (c + (state["orig"] - c) @ R.rotation((0, 0, 1), np.pi / 2).T * 0.8).astype(np.float32)
    else:
        state["mass"] = (state["mass"] * np.linspace(0.5, 2.0, len(state))).astype(np.float32)
    gpu.upload(state)
    ora = R.clone(state, moments_in_double=not strict)
    gpu.Animation(1)
    ora.Animation(1)
    got, want = gpu.sm_transform(), ora.sm_debug()
    if strict:
        for g, w in zip(got, want):
            assert bits_equal(g, w)
    else:
        assert_transform(lambda c_, f, e, t: parity_record("gpu_regimes.rest_shape_change", c_, f, e, t), change, got, want, TOL)


# ==== C. the radix-sort grid and strict in-cell order =================================================================
def set_reserved(sim, **slots):
    p = sim.get_params()
    for k, v in slots.items():
        p.reserved[int(k[1:])] = v
    sim._ck(sim.lib.sphsm_set_params(sim.h, p))


# Launches tallied from grid_sort / grid_finish / corrected_velocity / fused_step (sphsm_host_step.cuh).  The grid (passes = 0: the
# counting sort):
#   radix sort: k_hash + P x k_radix_pass (+ k_cell_order_fix in strict mode); cell table and gather: k_cell_bounds + gather
#   counting sort: (k_cell_count unless pass B filed the counts) + k_scan_onepass + k_cell_scatter + k_cell_sort_big + gather
def grid_launches(strict, passes, counts_filed):
    if passes:
        return 1 + passes + (1 if strict else 0) + 2
    return (0 if counts_filed else 1) + 4


# The rest of a step is five launches on either path:
#   strict: k_slot_of + k_sm_strict + k_goal_cvel + pass A + pass B
#   fast (steady state, rest sums cached): k_moments + k_sum_partials_par + k_sm_solve + pass A + pass B
def launches_per_step(strict, passes):
    return grid_launches(strict, passes, counts_filed=not strict) + 5


def sort_signature(passes):
    """Launches of a fast-mode Find_neighbors on a fresh set (nothing filed) and of a steady fast step.  Neither count alone tells every
    radix pass count from the counting sort (1 pass: 4 + 5 per step either way; 2 passes: 5 per Find_neighbors either way); the pair does."""
    return grid_launches(False, passes, False), launches_per_step(False, passes)


def measured_signature(sim):
    sim.reset_launch_count()
    sim.stage(1)
    find = sim.launch_count()
    sim.Animation(2)
    sim.reset_launch_count()
    sim.Animation(3)
    return find, sim.launch_count() / 3


def grid_path_sim(Sim, world, pos, mode, **kw):
    s = Sim(capacity=len(pos), world=world, **kw)
    set_reserved(s, r2=mode)
    s.Init_Fluid(pos)
    return s


def assert_csr_properties(sim, world, ordered, where):
    """The CSR is a permutation, every particle sits in the bucket numpy computes from the GPU's own positions, and (where the
    path promises it) the in-cell order is ascending original index."""
    start, idx = sim.cells_csr()
    n = sim.n
    assert start[-1] == n and np.array_equal(np.sort(idx), np.arange(n)), where
    pos = sim.positions()
    g = np.asarray(R.grid_dims(world), np.int64)
    cell = np.floor(pos / R.H).astype(np.int64)
    hsh = cell[:, 0] + g[0] * (cell[:, 1] + g[1] * cell[:, 2])
    owner = np.repeat(np.arange(len(start) - 1), np.diff(start))
    assert np.array_equal(hsh[idx], owner), where
    if ordered:
        same = owner[1:] == owner[:-1]
        assert np.all(idx[1:][same] > idx[:-1][same]), where


def strict_run_vs_restatement(Sim, world, pos, mode, passes, steps, where):
    ora = CpuSim("port", capacity=len(pos), world=world)
    ora.Init_Fluid(pos)
    gpu = grid_path_sim(Sim, world, pos, mode, strict=True)
    ora.stage(1)
    gpu.stage(1)
    for a, b in zip(gpu.cells_csr(), ora.cells_csr()):
        assert np.array_equal(a, b), (where, "CSR after Find_neighbors")
    for step in range(steps):
        gpu.reset_launch_count()
        gpu.Animation(1)
        assert gpu.launch_count() == launches_per_step(True, passes), (where, step, gpu.launch_count())
        ora.Animation(1)
        assert_bits(gpu.particles(), ora.particles(), FIELDS, (where, "strict step", step + 1))
    ora.stage(1)  # the restatement's buckets of the current positions (stage 1 moves nothing)
    for a, b in zip(gpu.cells_csr(), ora.cells_csr()):
        assert np.array_equal(a, b), (where, "CSR after steps")
    assert_csr_properties(gpu, world, True, where)


# fields of one step that do not depend on the shape-matching transform
SM_FREE_FIELDS = ("predicted_vel", "dens", "pres", "Iion", "w", "Inter_Vm", "Vm")


def fast_step_vs_double(Sim, world, pos, mode, record, case, jitter):
    """One fused fast step from the initial state against the double-moment restatement, classes of
    test_fused_step_vs_double_moment_oracle.  These sets start at rest and fall freely, so acc is a cancelling sum whose infinity norm
    is a rounding residue: it is bounded as in test_gpu_scale_parity (what the velocity differences imply, plus TOL of its norm).  A
    rest shape too ill-conditioned for the fast path's summation order (fast_comparable) compares the fields the transform does not
    reach."""
    ora = CpuSim("port", capacity=len(pos), world=world, moments_in_double=True)
    ora.Init_Fluid(pos)
    gpu = grid_path_sim(Sim, world, pos, mode)
    ok, cond = fast_comparable(ora.particles().copy(), False, True)
    assert ok or (len(pos) <= 3 and cond > 1e6), (case, cond)
    ora.Animation(1)
    gpu.Animation(1)
    got, want = gpu.particles(), ora.particles()
    params = params_of(want)
    for st in range(2, 8):
        for f in STAGE_OUT[st]:
            if not ok and f not in SM_FREE_FIELDS:
                continue
            if f == "acc":
                bound = acc_bound(got, want, ora.constants(), jitter)
                dacc = float(np.abs(got["acc"].astype(np.float64) - want["acc"]).max())
                record(case, "acc (absolute; bound = what the velocity differences imply)", dacc, bound)
                assert dacc <= bound, (case, dacc, bound)
                continue
            compare(record, case, f, got, want, params, fused_tol(f, False), world, ran_stage7=True)


def counting_vs_radix(Sim, world, pos, radix_mode, where, steps=10):
    """Forced counting against the radix path on the same set: the two differ only by the summation order inside cells."""
    out = []
    for mode in (2, radix_mode):
        s = grid_path_sim(Sim, world, pos, mode, diagnostics=False)
        s.Animation(steps)
        assert_csr_properties(s, world, mode == 2, (where, mode))
        out.append(s.particles())
    a, b = out
    for f in DIAG_OFF_FIELDS:
        scale = max(1e-30, float(np.abs(b[f].astype(np.float64)).max()))
        assert float(np.abs(a[f].astype(np.float64) - b[f].astype(np.float64)).max()) <= 2e-5 * scale, (where, f)


@pytest.mark.parametrize("name", list(R.RADIX_CASES))
def test_radix_grid(Sim, name, parity_record):
    world, pos, mode, passes = R.radix_case(name)
    assert R.sort_passes(world) == passes and R.counting_sort_auto(world, len(pos)) == (mode == 1)
    g = R.grid_dims(world)
    probe = Sim(capacity=len(pos), world=world)
    assert probe.num_cells == g[0] * g[1] * g[2]
    del probe
    # the path: strict and fast mode share grid_sort's choice (use_counting_sort: params.reserved[2], cell count, particle count), so
    # the fast-mode launch signature of this world and set proves the path of both
    assert sort_signature(passes) != sort_signature(0)
    assert measured_signature(grid_path_sim(Sim, world, pos, mode, diagnostics=False)) == sort_signature(passes), name
    assert measured_signature(grid_path_sim(Sim, world, pos, 2, diagnostics=False)) == sort_signature(0), (name, "counting")
    strict_run_vs_restatement(Sim, world, pos, mode, passes, 20, name)
    fast_step_vs_double(Sim, world, pos, mode, lambda c_, f, e, t: parity_record("gpu_regimes.radix_grid", c_, f, e, t), name,
                        R.RADIX_JITTER[name])
    counting_vs_radix(Sim, world, pos, mode, name)


@pytest.mark.parametrize("name", list(R.TILE_CASES))
def test_cell_table_at_scan_tile_edges(Sim, name, parity_record):
    world, pos, m = R.tile_case(name)
    assert R.padded_cells(world) + 1 == m and R.counting_sort_auto(world, len(pos))
    strict_run_vs_restatement(Sim, world, pos, 0, 0, 20, name)
    fast_step_vs_double(Sim, world, pos, 0, lambda c_, f, e, t: parity_record("gpu_regimes.cell_table_at_scan_tile_edges", c_, f, e, t), name,
                        R.FILL_JITTER)
    s = grid_path_sim(Sim, world, pos, 0, diagnostics=False)
    s.Animation(5)
    assert_csr_properties(s, world, True, name)


# ==== D. particle counts at launch boundaries =========================================================================
@pytest.mark.parametrize("n", R.BOUNDARY_COUNTS)
def test_launch_boundary_counts(Sim, n, parity_record):
    pos = R.boundary_set(n)
    ora = CpuSim("port")
    ora.Init_Fluid(pos)
    gpu = Sim(strict=True)
    gpu.Init_Fluid(pos)
    for step in range(5):
        ora.Animation(1)
        gpu.Animation(1)
        assert_bits(gpu.particles(), ora.particles(), FIELDS, (n, "strict step", step + 1))
    fast_step_vs_double(Sim, (1.5, 1.5, 1.5), pos, 0, lambda c_, f, e, t: parity_record("gpu_regimes.launch_boundary_counts", c_, f, e, t), f"n{n}",
                        R.BOUNDARY_JITTER)
    runs = []
    for graphs_off in (True, False):
        s = Sim(diagnostics=False)
        set_reserved(s, r4=1 if graphs_off else 0)
        s.Init_Fluid(pos)
        s.Animation(8)  # step 1 eager (rest sums), 2-3 first sightings of the two ping-pong signatures, 4-5 captured, 6-8 replayed
        runs.append(s.particles())
    assert_bits(runs[0], runs[1], ("pos", "vel", "dens", "pres", "Vm", "Iion", "w"), (n, "graph replay"))
