#!/usr/bin/env python
"""One small scenario for compute-sanitizer (tools/gpu_sanitize.sh): a few steps through the C-ABI on a chosen kernel path.
    python tools/sanitize_case.py thread|warp|radix|slab3|strict|io"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sph_sm_monodomain_b200 import LocalGroup, Sim, inputs, slabs  # noqa: E402

case = sys.argv[1]
G = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
if case in ("thread", "radix", "strict", "io"):
    pos = inputs.init_cube_positions()  # 4913 particles: thread-per-particle kernels
    sim = Sim(diagnostics=(case == "io"), strict=(case == "strict"))
    if case == "radix":
        p = sim.get_params()
        p.reserved[2] = 1  # LSD radix sort (decoupled look-back) instead of the counting sort
        sim._ck(sim.lib.sphsm_set_params(sim.h, p))
    sim.Init_Fluid(pos)
    sim.turnOnStim_Cube(pos)
    sim.Animation(3)
    if case == "io":
        sim.flip_quadratic()
        sim.Animation(2)
        sim.particles()
        sim.cells_csr()
        sim.neighbor_sets(np.arange(64, dtype=np.int32), 2)
        sim.turnOffStim()
        sim.Animation(1)
    print(case, "ok", float(np.abs(sim.positions()).max()))
elif case == "warp":
    g = np.load(os.path.join(G, "cfg2_5211_wave.npz"))  # the reference's dense mesh: warp-per-particle kernels, big-cell sort
    sim = Sim(diagnostics=False)
    sim.Init_Fluid(g["positions"])
    sim.set_fields(fixed=g["init.fixed"], stim=g["init.stim"])
    sim.Animation(3)
    print(case, "ok", float(np.abs(sim.positions()).max()))
elif case == "slab3":
    pos, world = inputs.lattice(30, 8, 8, jitter=0.05)
    fixed, stim = inputs.lattice_masks(pos, 30, 4)
    parts = slabs.partition_planes(slabs.plane_histogram(pos, 0, slabs.num_planes(world, 0)), 3)
    sims = []
    for _ in range(3):
        s = Sim(capacity=len(pos), world=world, diagnostics=False, slab_axis=0)
        s.Init_Fluid(pos)
        s.set_masks(fixed.astype(np.uint8), np.where(stim, np.float32(300), np.float32(0)).astype(np.float32))
        sims.append(s)
    grp = LocalGroup(sims)
    for s, (lo, hi) in zip(sims, parts):
        s.set_slab(lo, hi)
    grp.step(3)
    got, owner = grp.gather_positions(len(pos))
    print(case, "ok", bool((owner >= 0).all()))
else:
    raise SystemExit("unknown case")
