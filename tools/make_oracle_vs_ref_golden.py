#!/usr/bin/env python
"""Write tests/golden/oracle_vs_ref.npz: the reference's results on the seeded inputs of tests/test_oracle_vs_ref.py
(the same protocols, imported from there) — per-field digests after every compared stage, final positions and voltages.

    python tools/make_oracle_vs_ref_golden.py [--backend ref|port]

--backend ref (the default) runs the genuine reference class: build() with $SPHSM_REFERENCE_DIR naming a checkout of the
reference's sources first.  --backend port writes the C restatement's results instead; the committed file was written
that way, by the restatement as it stood when tests/test_oracle_vs_ref.py first compared it live with the genuine class on
these inputs, bit for bit (oracle/sphsm_oracle.c has not changed since).
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import available_backends  # noqa: E402
from tests import test_oracle_vs_ref as t  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--backend", default="ref", choices=["ref", "port"])
a = ap.parse_args()
if a.backend not in available_backends():
    sys.exit(f"back end {a.backend!r} not built: run __graft_entry__.build() with SPHSM_REFERENCE_DIR set to a checkout of the reference")

out = {}
for seed, quadratic, volume in t.CLOUDS:
    d = np.zeros((t.CLOUD_STEPS, 7, len(t.FIELDS)), np.uint64)
    for sims, step, st in t.random_cloud([a.backend], seed, quadratic, volume):
        d[step, st - 1] = t.digests(sims[0])
    p = sims[0].particles()
    out.update({f"cloud{seed}.digests": d, f"cloud{seed}.pos": p["pos"].copy(), f"cloud{seed}.Vm": p["Vm"].copy()})
for key, sims in (("walls", t.walls([a.backend])), ("lifted", t.lifted_world([a.backend]))):
    p = sims[0].particles()
    out.update({f"{key}.digests": t.digests(sims[0]), f"{key}.pos": p["pos"].copy(), f"{key}.Vm": p["Vm"].copy()})
    if key == "lifted":
        out["lifted.num_cells"] = np.int64(sims[0].num_cells)
out["fields"] = np.array(t.FIELDS)
out["backend"] = np.array(a.backend)
np.savez_compressed(t.GOLDEN, **out)
print(f"{t.GOLDEN}: {os.path.getsize(t.GOLDEN) / 1e3:.0f} kB from back end {a.backend!r}")
