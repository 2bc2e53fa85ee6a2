#!/usr/bin/env python
"""Generate tests/golden/*.npz from the GENUINE reference (oracle/_ref/libsphsm_ref.so, built by
`make -C oracle ref` from $SPHSM_REFERENCE_DIR, g++ -O2 -ffp-contract=off).

The reference has no tests or golden vectors of its own (SURVEY.md §4), so these files — outputs of the
unmodified reference class on its own inputs — are the committed pin for the C restatement (oracle/) and
the CUDA path.  Runs only where $SPHSM_REFERENCE_DIR names a checkout of the reference; the fixtures travel via git.

    python tools/make_golden.py            # ~2.5 min
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import CpuSim  # noqa: E402
from sph_sm_monodomain_b200 import inputs  # noqa: E402

REF_DIR = os.environ.get("SPHSM_REFERENCE_DIR")
if not REF_DIR or not os.path.isdir(os.path.join(REF_DIR, "Resources")):
    sys.exit("set SPHSM_REFERENCE_DIR to a checkout of the reference (this tool reads its Resources/*.csv)")
RES = os.path.join(REF_DIR, "Resources", "")
OUT = os.path.join(ROOT, "tests", "golden")

STATE = ("pos", "vel", "dens", "pres", "Vm", "Inter_Vm", "Iion", "w", "stim")
STAGE_OUT = {  # what each stage of compute_SPH_SM_monodomain writes (SURVEY.md §3.4)
    2: ("predicted_vel", "goal", "corrected_vel"),
    3: ("inter_vel",),
    4: ("dens", "pres"),
    5: ("Iion", "w"),
    6: ("acc", "Inter_Vm"),
    7: ("vel", "pos", "Vm"),
}


def snap(sim, fields, prefix, out):
    p = sim.particles()
    for f in fields:
        out[f"{prefix}.{f}"] = p[f].copy()


def first_step_by_stage(sim, out):
    sim.stage(1)
    start, idx = sim.cells_csr()
    occ = np.flatnonzero(np.diff(start) > 0).astype(np.int32)
    out["s1.occupied_cells"] = occ
    out["s1.occupied_start"] = start[occ].astype(np.int32)
    out["s1.occupied_count"] = np.diff(start)[occ].astype(np.int32)
    out["s1.bucket_items"] = idx.astype(np.int32)
    for st in range(2, 8):
        sim.stage(st)
        snap(sim, STAGE_OUT[st], f"s1.stage{st}", out)


def run_config(name, pos, setup, checkpoints, stim_off_before=None, quadratic=False, by_stage=True, **simkw):
    sim = CpuSim("ref", **simkw)
    sim.Init_Fluid(pos)
    setup(sim)
    if quadratic:
        assert sim.flip_quadratic()
    out = {"positions": pos}
    p = sim.particles()
    out["init.fixed"] = p["fixed"].copy()
    out["init.stim"] = p["stim"].copy()
    done = 0
    if by_stage:
        first_step_by_stage(sim, out)
        done = 1
        if 1 in checkpoints:
            snap(sim, STATE, "step1", out)
    for cp in sorted(checkpoints):
        if cp <= done:
            continue
        while done < cp:
            if stim_off_before is not None and done == stim_off_before:
                sim.turnOffStim()  # main.cpp:329-334 issues it just before the (k+1)-th Animation()
            sim.Animation()
            done += 1
        snap(sim, STATE, f"step{cp}", out)
    out["checkpoints"] = np.asarray(sorted(checkpoints), np.int32)
    out["stim_off_before"] = np.int32(-1 if stim_off_before is None else stim_off_before)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: N={sim.n} -> {path} ({os.path.getsize(path) / 1e6:.2f} MB)")
    sim.close()


def kats():
    sim = CpuSim("ref")
    rng = np.random.Generator(np.random.PCG64(7))
    out = {}
    c = sim.constants()
    out["const_names"] = np.asarray(list(c.keys()))
    out["const_values"] = np.asarray(list(c.values()), np.float32)
    h = np.float32(0.04)
    r = np.concatenate([np.linspace(0, 0.1, 257, dtype=np.float32), np.asarray([h, np.nextafter(h, np.float32(1)), np.nextafter(h, np.float32(0)), 2 * h, np.nextafter(2 * h, np.float32(0))], np.float32)])
    r2 = np.concatenate([(r * r).astype(np.float32), np.asarray([h * h, np.nextafter(h * h, np.float32(1)), 1e-12, 0.0], np.float32)])
    out["r"], out["r2"] = r, r2
    out["poly6"] = np.asarray([sim.Poly6(x) for x in r2], np.float32)
    out["spiky"] = np.asarray([sim.Spiky(x) for x in r], np.float32)
    out["visco"] = np.asarray([sim.Visco(x) for x in r], np.float32)
    out["bspline2"] = np.asarray([sim.B_spline_2(x) for x in r], np.float32)
    pts = (rng.random((512, 3), dtype=np.float32) * np.float32(1.7) - np.float32(0.1)).astype(np.float32)
    pts[:8] = np.asarray([[0, 0, 0], [1.5, 1.5, 1.5], [1.4999, 1.4999, 1.4999], [0.04, 0.08, 0.12], [0.12, 0.04, 0.08],
                          [0.28, 0.28, 0.28], [0.039999, 0.04, 0.040001], [1.48, 0.0, 1.48]], np.float32)
    out["hash_points"] = pts
    out["hash_values"] = np.asarray([sim.cell_hash(*p) for p in pts], np.int32)
    mats3 = rng.standard_normal((64, 3, 3)).astype(np.float32)
    mats3[0] = np.eye(3)
    mats3[1] = np.diag([2, 3, 4])
    mats3[2] = 0  # singular: invert() must leave it unchanged, polar() yields zeros
    mats3[3] = np.asarray([[1, 2, 3], [2, 4, 6], [1, 1, 1]], np.float32)  # rank deficient
    out["m3"] = mats3
    out["m3_polar"] = np.stack([sim.polar3(m) for m in mats3])
    inv = [sim.invert3(m) for m in mats3]
    out["m3_inv_ok"] = np.asarray([o for o, _ in inv], np.bool_)
    out["m3_inv"] = np.stack([m for _, m in inv])
    mats9 = []
    for k in range(16):
        q = rng.standard_normal((40, 9)).astype(np.float32) * np.float32(0.3 if k % 2 else 1.0)
        mats9.append((q.T @ q).astype(np.float32))
    mats9[0] = np.eye(9, dtype=np.float32)
    mats9 = np.stack(mats9)
    out["m9"] = mats9
    out["m9_inv"] = np.stack([sim.invert9(m) for m in mats9])
    path = os.path.join(OUT, "kats.npz")
    np.savez_compressed(path, **out)
    print("kats ->", path)


def main():
    os.makedirs(OUT, exist_ok=True)
    kats()
    mesh = lambda pos: (lambda s: s.turnOnStim_Mesh(pos))  # noqa: E731
    # BASELINE.json config 1: 4944 mesh, main.cpp defaults, 1000 steps, stim off at the half-way point
    p1 = inputs.read_cloud(RES + "biceps_simple_out_4944.csv")
    run_config("cfg1_4944", p1, mesh(p1), [1, 2, 10, 100, 500, 501, 1000], stim_off_before=500)
    # config 2: 18475 file through main.cpp's subsample rule -> 5211, variant (i) all stimulated
    p2 = inputs.read_cloud(RES + "biceps_simple_out_18475.csv", 7)
    run_config("cfg2_5211", p2, mesh(p2), [1, 100, 1000], stim_off_before=500)

    # variant (ii): stimulate only the x <= 0.07 end -> a travelling wave (SURVEY.md §8c)
    def wave(s):
        s.turnOnStim_Mesh(p2)
        p = s.particles()
        p["stim"] = np.where(p["pos"][:, 0] <= np.float32(0.07), np.float32(300.0), np.float32(0.0))

    run_config("cfg2_5211_wave", p2, wave, [1, 50, 200])
    # init_cube lattice (main.cpp:464-477) + turnOnStim_Cube
    pc = inputs.init_cube_positions()
    run_config("cube_4913", pc, lambda s: s.turnOnStim_Cube(pc), [1, 100, 500])
    # quadratic shape matching: per-step parity only (truncated 9x9 Jacobi, Q7)
    run_config("cube_4913_quadratic", pc, lambda s: s.turnOnStim_Cube(pc), [1, 2, 20], quadratic=True)
    run_config("cfg1_4944_quadratic", p1, mesh(p1), [1, 2, 5], quadratic=True)

    # small jittered lattice in a lifted world (exercises ref_resize / non-default grid)
    pl, world = inputs.lattice(24, 10, 12, jitter=0.05)
    fixed, stim = inputs.lattice_masks(pl, 24, 4)

    def lat(s):
        p = s.particles()
        p["fixed"] = fixed
        p["stim"] = np.where(stim, np.float32(300), np.float32(0))

    run_config("lattice_24x10x12", pl, lat, [1, 10, 100], capacity=len(pl), world=world)
    np.save(os.path.join(OUT, "lattice_24x10x12.world.npy"), np.asarray(world, np.float32))


if __name__ == "__main__":
    main()
