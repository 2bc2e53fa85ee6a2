"""Inputs shared by tests/test_regimes_cpu.py (which proves on the restatement and in numpy that each case reaches the branch
it is named for) and tests/test_gpu_regimes.py (which runs the same cases on the GPU): shape-matching bodies far from their
rest shape, worlds sized for a given padded cell count, and particle sets whose counts sit on launch boundaries."""
import numpy as np

from oracle import CpuSim
from sph_sm_monodomain_b200 import inputs

H = np.float32(0.04)
CENTRE = np.float32([0.75, 0.75, 0.75])  # deformed bodies are placed about the middle of the default 1.5^3 world
RADIX_BITS = 8


# ---- shape matching far from rest ------------------------------------------------------------------------------------
def rotation(axis, angle):
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    k = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + np.sin(angle) * k + (1 - np.cos(angle)) * (k @ k)


def _small_lattice():
    pos, _ = inputs.lattice(7, 6, 5, origin=(0.6, 0.6, 0.6), jitter=0.2, seed=31)
    return pos


def _sheet(z):
    cube = inputs.init_cube_positions()
    layer = cube[cube[:, 2] == cube[0, 2]].copy()
    layer[:, 2] = np.float32(z)
    return layer


_GENERIC = rotation((1.0, 2.0, 3.0), 0.7)
# name: (rest-shape builder, deformation matrix applied about the rest centroid, fixed rule, degenerate rest shape)
BODIES = {
    "cube_rot_x90": (inputs.init_cube_positions, rotation((1, 0, 0), np.pi / 2), None, False),
    "cube_rot_y90": (inputs.init_cube_positions, rotation((0, 1, 0), np.pi / 2), None, False),
    "cube_rot_z90": (inputs.init_cube_positions, rotation((0, 0, 1), np.pi / 2), None, False),
    "cube_rot_z180": (inputs.init_cube_positions, rotation((0, 0, 1), np.pi), None, False),
    "cube_rot_generic": (inputs.init_cube_positions, _GENERIC, None, False),
    "cube_mirror_x": (inputs.init_cube_positions, np.diag([-1.0, 1.0, 1.0]), None, False),
    "cube_compress_0.5": (inputs.init_cube_positions, 0.5 * np.eye(3), None, False),
    "cube_compress_0.3": (inputs.init_cube_positions, 0.3 * np.eye(3), None, False),
    "cube_stretch": (inputs.init_cube_positions, np.diag([1.4, 0.8, 1.15]), None, False),
    "cube_shear": (inputs.init_cube_positions, np.array([[1.0, 0.6, 0.0], [0.0, 1.0, 0.25], [0.0, 0.0, 1.0]]), None, False),
    "cube_third_fixed": (inputs.init_cube_positions, _GENERIC @ np.diag([1.2, 0.9, 1.0]), "third", False),
    "lattice_rot_generic": (_small_lattice, _GENERIC, None, False),
    "lattice_mirror_x": (_small_lattice, np.diag([-1.0, 1.0, 1.0]), None, False),
    "lattice_compress_0.3": (_small_lattice, 0.3 * np.eye(3), None, False),
    "sheet_z0.5": (lambda: _sheet(0.5), _GENERIC @ np.diag([1.2, 0.9, 1.0]), None, True),
    "sheet_z0.45": (lambda: _sheet(0.45), _GENERIC @ np.diag([1.2, 0.9, 1.0]), None, True),
    "line": (lambda: np.stack([np.float32(0.5) + np.float32(0.01) * np.arange(40, dtype=np.float32),
                               np.full(40, 0.3, np.float32), np.full(40, 0.7, np.float32)], 1), _GENERIC, None, True),
    "n2": (lambda: np.float32([[0.70, 0.71, 0.72], [0.73, 0.70, 0.74]]), _GENERIC, None, True),
    "n3": (lambda: np.float32([[0.70, 0.71, 0.72], [0.73, 0.70, 0.74], [0.71, 0.75, 0.70]]), _GENERIC, None, True),
}


def body(name):
    """(rest positions, deformed positions, fixed mask) of a body: pos = CENTRE + M (rest - centroid), float32."""
    build, m, fixed_rule, _ = BODIES[name]
    rest = np.ascontiguousarray(build(), np.float32)
    c = rest.astype(np.float64).mean(axis=0)
    pos = (CENTRE + (rest.astype(np.float64) - c) @ np.asarray(m).T).astype(np.float32)
    fixed = (np.arange(len(rest)) % 3 == 0) if fixed_rule == "third" else np.zeros(len(rest), bool)
    return rest, pos, fixed.astype(np.uint8)


def body_state(name):
    """The restatement's AoS for a body: Init_Fluid at rest (orig, mass, density), then the deformed positions."""
    rest, pos, fixed = body(name)
    s = CpuSim("port")
    s.Init_Fluid(rest)
    s.set_fields(pos=pos, fixed=fixed)
    return s.particles().copy()


def clone(state, quadratic=False, volume=True, **kw):
    """A restatement holding `state` (a full AoS) with the given shape-matching switches."""
    s = CpuSim("port", **kw)
    s.Init_Fluid(state["pos"])
    s.particles()[:] = state
    if quadratic:
        assert s.flip_quadratic()
    if not volume:
        assert not s.flip_volume()
    return s


def centred(p, ocm, cm=None):
    q = (p["orig"] - ocm).astype(np.float32)
    x = None if cm is None else (p["pos"] - cm).astype(np.float32)
    return x, q


def restatement_aqq(p, ocm):
    """Aqq as the double-moment restatement forms it: float products m q_a q_b, double sums, one rounding to float."""
    _, q = centred(p, ocm)
    mq = (p["mass"][:, None] * q).astype(np.float32)
    prod = (mq[:, :, None] * q[:, None, :]).astype(np.float32)
    return prod.astype(np.float64).sum(axis=0).astype(np.float32)


def restatement_a9qq(p, ocm):
    """A9qq of the quadratic mode, formed like restatement_aqq over q9 = (q, q_a^2, q_x q_y, q_y q_z, q_z q_x)."""
    _, q = centred(p, ocm)
    q9 = np.concatenate([q, q * q, q * np.roll(q, -1, axis=1)], axis=1).astype(np.float32)
    mq = (p["mass"][:, None] * q9).astype(np.float32)
    return (mq[:, :, None] * q9[:, None, :]).astype(np.float32).astype(np.float64).sum(axis=0).astype(np.float32)


def reduced_cond(m):
    """Condition number of m without its exactly zero rows / columns (which every implementation carries through exactly)."""
    live = np.flatnonzero(np.asarray(m).any(axis=1))
    return float(np.linalg.cond(np.asarray(m, np.float64)[np.ix_(live, live)])) if len(live) else np.inf


def restatement_apq(p, cm, ocm):
    x, q = centred(p, ocm, cm)
    mx = (p["mass"][:, None] * x).astype(np.float32)
    prod = (mx[:, :, None] * q[:, None, :]).astype(np.float32)
    return prod.astype(np.float64).sum(axis=0).astype(np.float32)


def solve_state(state, quadratic=False, volume=True, dbl=True):
    """Stage 2 of the restatement on `state`: (sim, cm, ocm, xform)."""
    s = clone(state, quadratic, volume, moments_in_double=dbl)
    s.stage(2)
    cm, ocm, x = s.sm_debug()
    return s, cm, ocm, x


# ---- grids by padded cell count ---------------------------------------------------------------------------------------
def grid_dims(world):
    """Cells per axis, ceilf(world / h) in float as the library and the reference compute them."""
    return tuple(int(np.ceil(np.float32(w) / H)) for w in world)


def padded_cells(world):
    """Keys of the device grid: one empty border cell on each side of the two inner axes, (G0+2)(G1+2)G2."""
    g = grid_dims(world)
    return (g[0] + 2) * (g[1] + 2) * g[2]


def sort_passes(world):
    """8-bit LSD passes for keys 0..padded (the last one is the limbo bucket of particles outside the grid)."""
    bits = max(1, int(padded_cells(world)).bit_length())
    return (bits + RADIX_BITS - 1) // RADIX_BITS


def counting_sort_auto(world, n):
    """The automatic choice of the library: counting sort unless the grid has more than 8n + 2^20 cells."""
    return padded_cells(world) <= 8 * max(n, 1) + (1 << 20)


def world_for(g):
    """A world of exactly g cells per axis (half a cell short of the next boundary, so no rounding can decide it)."""
    return tuple(float(np.float32((k - 0.5) * 0.04)) for k in g)


FILL_JITTER = 0.1  # fraction of the spacing, as inputs.lattice


def fill(world, seed, jitter=FILL_JITTER, limit=None):
    """A seeded jittered lattice of spacing 0.9 h inside `world`, clear of the walls by half a spacing."""
    s = float(H) * 0.9
    axes = [np.arange(0.5 * s, w - 0.5 * s, s) for w in world]
    axes = [a if len(a) else np.array([0.5 * w]) for a, w in zip(axes, world)]
    Z, Y, X = np.meshgrid(axes[2], axes[1], axes[0], indexing="ij")
    pos = np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1)
    rng = np.random.Generator(np.random.PCG64(seed))
    pos = pos + (rng.random(pos.shape) * 2 - 1) * jitter * s
    hi = np.asarray(world) - 1e-3
    pos = np.clip(pos, 1e-3, hi).astype(np.float32)
    if limit is not None and len(pos) > limit:
        pos = pos[np.sort(rng.choice(len(pos), limit, replace=False))]
    return np.ascontiguousarray(pos)


BOUNDARY_JITTER = 0.1


def _tiny():
    return inputs.lattice(3, 3, 3, origin=(0.02, 0.02, 0.02), jitter=RADIX_JITTER["forced_1pass"], seed=41)[0]


RADIX_JITTER = {"forced_1pass": 0.2, "forced_2pass": 0.0, "auto_3pass": 0.0, "auto_4pass": 0.0,
                "forced_2pass_n4095": BOUNDARY_JITTER, "forced_2pass_n4096": BOUNDARY_JITTER, "forced_2pass_n4097": BOUNDARY_JITTER}
# name: (world, particle builder, params.reserved[2] (0 auto, 1 radix), radix passes)
# The _nK cases put the particle count, which the radix passes tile by SORT_TILE (4096 keys), on either side of a tile edge.
RADIX_CASES = {
    "forced_1pass": ((0.12, 0.12, 0.12), _tiny, 1, 1),
    "forced_2pass": ((1.5, 1.5, 1.5), inputs.init_cube_positions, 1, 2),
    "auto_3pass": ((4.2, 4.2, 4.2), inputs.init_cube_positions, 0, 3),
    "auto_4pass": ((10.4, 10.4, 10.4), inputs.init_cube_positions, 0, 4),
    "forced_2pass_n4095": ((1.5, 1.5, 1.5), lambda: boundary_set(4095), 1, 2),
    "forced_2pass_n4096": ((1.5, 1.5, 1.5), lambda: boundary_set(4096), 1, 2),
    "forced_2pass_n4097": ((1.5, 1.5, 1.5), lambda: boundary_set(4097), 1, 2),
}
# padded cell count + 1 (the counting sort's cell-table length: cells + the limbo bucket, scanned in tiles of SCAN_TILE = 2048
# entries) on either side of one and two tiles, and one count far from both; each a product (G0+2)(G1+2)G2, plus 1
TILE_CASES = {
    "m2047": ((4, 9, 31), 2047),
    "m2048": ((21, 87, 1), 2048),
    "m2049": ((6, 14, 16), 2049),
    "m4095": ((21, 87, 2), 4095),
    "m4096": ((7, 11, 35), 4096),
    "m4097": ((14, 14, 16), 4097),
    "m1002": ((5, 9, 13), 1002),
}


def radix_case(name):
    world, build, mode, passes = RADIX_CASES[name]
    return world, build(), mode, passes


def tile_case(name):
    g, m = TILE_CASES[name]
    world = world_for(g)
    return world, fill(world, seed=m, limit=3000), m


# ---- particle counts at launch boundaries -----------------------------------------------------------------------------
# k_moments: 2048 particles per block, 4-deep unrolled body + tail; neighbour passes: 128-thread blocks, the rest 256; warps of 32
BOUNDARY_COUNTS = (2, 3, 31, 32, 33, 127, 128, 129, 255, 256, 257, 2047, 2048, 2049, 4095, 4096, 4097, 8193)


def boundary_set(n):
    pos, _ = inputs.lattice(24, 20, 20, origin=(0.04, 0.02, 0.04), jitter=BOUNDARY_JITTER, seed=53)
    rng = np.random.Generator(np.random.PCG64(n))
    return np.ascontiguousarray(pos[np.sort(rng.choice(len(pos), n, replace=False))])
