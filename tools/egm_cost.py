#!/usr/bin/env python
"""Cost of the on-device electrograms (sphsm_egm_*): step time with electrograms off and on with 1, 16, 64 and 256 electrodes, on
one GPU.

    python tools/egm_cost.py [--workloads 8m,cfg2] [--rounds 8] [--block 20] [--out FILE]

The settings alternate in one process on one handle (start / stop between blocks), so clocks and neighbours affect them alike;
each block is warmed by a few steps of its own setting (its CUDA graph, on the small set, is captured there) and timed with device
events around `block` steps.  The electrodes are spread over a box around the body, half of them inside it.  Prints one JSON line
with the GPU name and power limit (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from sph_sm_monodomain_b200 import Sim  # noqa: E402

SETTINGS = ("off", "egm_1", "egm_16", "egm_64", "egm_256")


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, plim = (v.strip() for v in out.split(","))
        return name, plim
    except Exception:  # (no nvidia-smi: the name from the runtime, the limit unknown)
        import torch

        return torch.cuda.get_device_name(0), None


def measure(key, rounds, block, warm):
    wl = bench.parse_workload(key)
    pos, world, fixed, stim = bench.workload_inputs(wl)
    n = len(pos)
    kw = dict(capacity=n, world=world) if "golden" not in wl else {}
    sim = Sim(diagnostics=False, **kw)
    sim.Init_Fluid(pos)
    sim.set_masks(fixed, stim)
    if wl.get("quadratic"):
        sim.flip_quadratic()
    lo, hi = pos.min(axis=0), pos.max(axis=0)
    el = (lo + (np.random.default_rng(7).random((256, 3)) * 2.0 - 0.5) * (hi - lo)).astype(np.float32)
    ms = {s: [] for s in SETTINGS}
    sim.Animation(warm)
    for r in range(rounds):
        k = r % len(SETTINGS)
        order = SETTINGS[k:] + SETTINGS[:k]  # rotate which setting goes first
        for s in order:
            sim.egm_stop()
            if s != "off":
                sim.egm_start(el[: int(s.split("_")[1])], rows=block + warm)
            sim.Animation(warm)
            sim.timer_mark(0)
            sim.Animation(block)
            sim.timer_mark(1)
            ms[s].append(sim.timer_ms() / block)
    sim.egm_stop()
    res = {"workload": key, "particles": n, "steps_per_setting": rounds * block, "block_steps": block}
    base = float(np.median(ms["off"]))
    for s in SETTINGS:
        v = np.asarray(ms[s])
        res[s] = {"median_ms_per_step": float(np.median(v)), "min_ms_per_step": float(v.min()), "max_ms_per_step": float(v.max())}
        if s != "off":
            res[s]["overhead_vs_off_pct"] = 100.0 * (float(np.median(v)) - base) / base
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="8m,cfg2")
    ap.add_argument("--rounds", type=int, default=8)
    ap.add_argument("--block", type=int, default=20)
    ap.add_argument("--warm", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, plim = gpu_info()
    line = {"egm_cost": [measure(k, a.rounds, a.block, a.warm) for k in a.workloads.split(",")], "gpu": name, "power_limit": plim,
            "timing": "device events around each block of steps; settings alternate in one process"}
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(s + "\n")


if __name__ == "__main__":
    main()
