"""CPU: the C restatement against the GENUINE reference on seeded random inputs beyond the committed fixtures — random
clouds stage by stage, particles thrown at the walls, a lifted world.

The reference's results are stored in tests/golden/oracle_vs_ref.npz (tools/make_oracle_vs_ref_golden.py): a 64-bit
digest of every Particle field after every compared stage, and the final positions and voltages.  Every run compares
the restatement with them bit for bit.  Where oracle/_ref was built (build() with $SPHSM_REFERENCE_DIR naming a checkout
of the reference's sources) the genuine class also runs alongside, live."""
import hashlib
import os

import numpy as np
import pytest

from oracle import CpuSim, available_backends
from sph_sm_monodomain_b200 import inputs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref.npz")
FIELDS = [f for f in CpuSim("port").particles().dtype.names if f != "_pad"]
CLOUDS = [(1, False, True), (2, True, True), (3, False, False), (4, True, False)]
CLOUD_STEPS = 12


def digests(sim):
    """One 64-bit digest of the bytes of each Particle field (FIELDS order)."""
    p = sim.particles()
    return np.array([np.frombuffer(hashlib.blake2b(np.ascontiguousarray(p[f]).tobytes(), digest_size=8).digest(), "<u8")[0]
                     for f in FIELDS], np.uint64)


def pres_is_defined(step, stage):
    # `pres` is uninitialised heap memory in the reference until stage 4 first writes it
    # (Init_Particle, cpp:101-125, never sets it); the restatement zero-fills.
    return not (step == 0 and stage < 4)


# ---- the three protocols; each drives every simulation given in lockstep ------------------------------------------------
def random_cloud(backends, seed, quadratic, volume):
    """Yields (sims, step, stage) after every stage of CLOUD_STEPS steps; stimulation off after step 6."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = 1500
    pos = (rng.random((n, 3), dtype=np.float32) * np.float32(0.5) + np.float32(0.4)).astype(np.float32)
    sims = [CpuSim(b) for b in backends]
    for s in sims:
        s.Init_Fluid(pos)
        s.set_stim((0.6, 0.6, 0.6), 0.02, 300.0)
        s.set_fields(fixed=(pos[:, 0] < 0.45).astype(np.uint8))
        if quadratic:
            s.flip_quadratic()
        if not volume:
            s.flip_volume()
    for step in range(CLOUD_STEPS):
        for st in range(1, 8):
            for s in sims:
                s.stage(st)
            yield sims, step, st
        if step == 6:
            for s in sims:
                s.turnOffStim()


def walls(backends):
    """Particles thrown at all six walls: stage 7's reflection/clamp path (cpp:618-649), 25 steps."""
    rng = np.random.Generator(np.random.PCG64(11))
    n = 600
    pos = (rng.random((n, 3), dtype=np.float32) * np.float32(1.5)).astype(np.float32)
    vel = (rng.standard_normal((n, 3)) * 40).astype(np.float32)
    sims = [CpuSim(b) for b in backends]
    for s in sims:
        s.Init_Fluid(pos)
        s.set_fields(vel=vel, stim=np.full(n, 300, np.float32))
        s.Animation(25)
    return sims


def lifted_world(backends):
    pos, world = inputs.lattice(14, 9, 11, jitter=0.1, seed=5)
    fixed, stim = inputs.lattice_masks(pos, 14, 3)
    sims = [CpuSim(b, capacity=len(pos), world=world) for b in backends]
    for s in sims:
        s.Init_Fluid(pos)
        s.set_fields(fixed=fixed, stim=np.where(stim, 300, 0).astype(np.float32))
        s.Animation(20)
    return sims


# ---- tests ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ref():
    return dict(np.load(GOLDEN))


def backends():
    """The restatement, plus the genuine reference where it was built here."""
    return ["port"] + (["ref"] if "ref" in available_backends() else [])


def assert_matches(sims, want, mask=None, where=""):
    """Digests of the restatement equal the stored reference digests, and every other back end equals the restatement."""
    mask = np.ones(len(FIELDS), bool) if mask is None else mask
    got = digests(sims[0])
    bad = [f for f, g, w, m in zip(FIELDS, got, want, mask) if m and g != w]
    assert bad == [], (where, "fields differing from the reference", bad)
    for other in sims[1:]:
        live = [f for f, g, o, m in zip(FIELDS, got, digests(other), mask) if m and g != o]
        assert live == [], (where, other.backend, "fields differing live", live)


def assert_final(sims, ref, key):
    p = sims[0].particles()
    for f in ("pos", "Vm"):
        want = ref[f"{key}.{f}"]
        assert p[f].tobytes() == want.tobytes(), (key, f, float(np.abs(p[f].astype(np.float64) - want).max()))


@pytest.mark.parametrize("seed,quadratic,volume", CLOUDS)
def test_random_cloud_bit_identical(seed, quadratic, volume, ref):
    key = f"cloud{seed}"
    want = ref[key + ".digests"]
    assert want.shape == (CLOUD_STEPS, 7, len(FIELDS))
    mask = np.ones(len(FIELDS), bool)
    for sims, step, st in random_cloud(backends(), seed, quadratic, volume):
        mask[FIELDS.index("pres")] = pres_is_defined(step, st)
        assert_matches(sims, want[step, st - 1], mask, where=(step, st))
    assert_final(sims, ref, key)


def test_walls_and_clamps_bit_identical(ref):
    sims = walls(backends())
    assert_matches(sims, ref["walls.digests"])
    assert_final(sims, ref, "walls")
    p = sims[0].particles()["pos"]
    assert p.min() >= 0.0 and p.max() <= 1.5


def test_lifted_world_bit_identical(ref):
    sims = lifted_world(backends())
    assert all(s.num_cells == int(ref["lifted.num_cells"]) for s in sims)
    assert_matches(sims, ref["lifted.digests"])
    assert_final(sims, ref, "lifted")
