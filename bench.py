#!/usr/bin/env python
"""bench.py — particle-steps/s of the full SPH + shape-matching + monodomain step (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 8m|8m_jitter|1m|32m|cfg1|cfg2|<nx>x<ny>x<nz>]
                    [--dump-outputs DIR]

A "step" is one Animation() of the whole particle set: neighbour search (hash, counting sort = cell table, reorder),
shape matching (moments, polar decomposition, goal positions), both neighbour passes, ionic model, integration.
Default workload: BASELINE.json configs[3], the synthetic 8M-particle elongated lattice (512x125x125) with quadratic
shape matching — the configuration the north_star's throughput target is quoted on; it fits one B200 and is
strong-scaled over 2/4/8 GPUs (slabs along x).  Inputs are synthetic (lattice generator of the reference's init_cube
rule) and far larger than L2 (8M x 68 B of persistent state = 544 MB vs 126 MB), so no L2 flush is needed between
timed steps.

One JSON line on stdout (rank 0).  `value` = device-resident throughput (CUDA events around exactly K steps, max over
ranks); `e2e` = the same metric through the C-ABI with HOST buffers: every step uploads the stimulation values of the
particles the rank owns from pinned host memory (the per-step control input of this path; 4 B per particle in total,
whatever the number of ranks) and downloads their positions (what the reference's viewer reads through Get_Paticles()
every frame), using the library's asynchronous I/O calls so that the copies of step k overlap the compute of step k+1;
the timed region ends when the last result is in host memory.  `roofline` is the dominant kernel (fused pass B) from
CUDA events on the handle's stream; `cpu_baseline` is the reference's own CPU step timed on this box (1 thread — the
reference has no threading) on a bounded sample.  With N > 1 the line also carries `mg_parity`: a small lattice stepped
through the same slab path on all ranks and compared with a single-GPU run on rank 0 before the timed region.  With
N = 1 and the default workload it carries `also`: quick measurements of the other configurations in the same process.

`--dump-outputs DIR` writes the particle state the timed path left after its last timed step (what a caller reads back
through Get_Paticles()) as DIR/<field>.npy, so that two builds run with the same arguments can be compared output for output.
Compare dumps of the same arm only: on a lattice workload the reference arm steps its bounded CPU sample
(CPU_SAMPLE_DIMS), not the workload the GPU arm steps.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "particle-steps/sec (full SPH+SM+monodomain step)"
UNIT = "particle-steps/s"
# SURVEY.md §8(d): algorithmic bytes per particle — whole fused-minimal step and the fused pass B
STEP_BYTES_PER_PARTICLE = 244
PASS_B_BYTES_PER_PARTICLE = 92
# On one GPU pass B also files the next step's counting-sort input (key 4 B + provisional rank 4 B per particle; the position
# it hashes is the one it has just integrated, so the hash stage's 12 B position read disappears): 92 + 8.  Slab mode keeps
# the separate k_cell_count (arrivals are not known yet) and the 92 B figure.
PASS_B_FUSED_HASH_BYTES = 8
PASS_B_NAME = "pass_b(cell+force+laplacian+integrate)"

WORKLOADS = {
    "1m": dict(dims=(100, 100, 100), quadratic=False, name="synthetic 1M-particle cubic lattice, linear shape matching (configs[2])"),
    "8m": dict(dims=(512, 125, 125), quadratic=True, name="synthetic 8M-particle elongated lattice 512x125x125, quadratic shape matching (configs[3])"),
    "32m": dict(dims=(800, 200, 200), quadratic=False, pacing=(50, 25),
                name="synthetic 32M-particle lattice 800x200x200, monodomain pacing: stimulus on the end slab every 50 steps, turnOffStim 25 steps later (configs[4])"),
    "8m_jitter": dict(dims=(512, 125, 125), quadratic=True, jitter=0.05,
                      name="synthetic 8M-particle lattice 512x125x125 with seeded jitter U(-0.05 s, 0.05 s) per coordinate (SURVEY 8d.3), quadratic shape matching"),
}
# BASELINE.json configs[0] / configs[1]: the reference's own particle sets (Resources/*.csv through main.cpp's loader rule,
# turnOnStim_Mesh), taken from the committed golden fixtures (tests/golden/, generated from the genuine reference by
# tools/make_golden.py) because the reference's sources are not part of this repository.  Small: latency-bound on a GPU; listed
# for the CPU-vs-GPU comparison on the reference's own inputs, not as the headline.
WORKLOADS["cfg1"] = dict(golden="cfg1_4944", quadratic=False, name="Resources/biceps_simple_out_4944.csv, main.cpp defaults (configs[0])")
WORKLOADS["cfg2"] = dict(golden="cfg2_5211", quadratic=False, name="Resources/biceps_simple_out_18475.csv subsampled to 5211 (configs[1])")
CPU_SAMPLE_DIMS = (100, 100, 100)  # bounded sample for the CPU legs: a 1M-particle lattice of the same spacing / SM mode (~0.9 s per step)
CPU_SAMPLE_STEPS = 10              # ~10 s of single-thread CPU work at ~1.2e6 particle-steps/s
FIXED_WARMUP = 400                 # untimed steps before the timed region, the same for every N (>= 0.1 s under load at N = 8, 0.6 s at N = 1)
# --dump-outputs: the state a step carries into the next one, i.e. the fields the fast path keeps current (44 B per particle);
# larger sets are cut to a seeded sample of DUMP_MAX_PARTICLES particles (44 MB)
DUMP_FIELDS = ("pos", "vel", "dens", "Vm", "Iion", "w", "stim")
DUMP_MAX_PARTICLES = 1 << 20
DUMP_SEED = 0


def parse_workload(s):
    if s in WORKLOADS:
        return dict(WORKLOADS[s], key=s)
    nx, ny, nz = (int(v) for v in s.lower().split("x"))
    return dict(dims=(nx, ny, nz), quadratic=False, name=f"synthetic {nx}x{ny}x{nz} lattice, linear shape matching", key=s)


def workload_inputs(wl):
    """(positions, world, fixed u8, stim f32) of a workload: a synthetic lattice or one of the reference's own particle sets."""
    if "golden" in wl:
        g = np.load(os.path.join(ROOT, "tests", "golden", wl["golden"] + ".npz"))
        return (np.ascontiguousarray(g["positions"], dtype=np.float32), (1.5, 1.5, 1.5), g["init.fixed"].astype(np.uint8),
                g["init.stim"].astype(np.float32))
    return make_lattice(wl["dims"], wl.get("jitter", 0.0))


def make_lattice(dims, jitter=0.0):
    from sph_sm_monodomain_b200 import inputs

    pos, world = inputs.lattice(*dims, jitter=jitter)
    fixed, stim = inputs.lattice_masks(pos, dims[0], 8)
    return pos, world, fixed.astype(np.uint8), np.where(stim, np.float32(300.0), np.float32(0.0)).astype(np.float32)


def dump_outputs(out_dir, particles):
    """DUMP_FIELDS of a Get_Paticles() array as out_dir/<field>.npy (float32, original particle order).  Above
    DUMP_MAX_PARTICLES particles only a sample is written: the same seeded indices on every run, ascending."""
    n = len(particles)
    idx = slice(None)
    if n > DUMP_MAX_PARTICLES:
        idx = np.sort(np.random.Generator(np.random.PCG64(DUMP_SEED)).permutation(n)[:DUMP_MAX_PARTICLES])
    os.makedirs(out_dir, exist_ok=True)
    for f in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f + ".npy"), np.ascontiguousarray(particles[f][idx], dtype=np.float32))


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_rate(quadratic, steps, warmup, backend=None, wl=None, dump_dir=None):
    """The reference's CPU step on this box: genuine class (oracle/_ref, built with its Makefile's -Ofast) when the
    prebuilt library travelled, else the bit-identical C restatement.  One thread: the reference has no threading.
    dump_dir: where to write the state after the timed steps (dump_outputs)."""
    from oracle import CpuSim, available_backends

    avail = available_backends()
    if backend is None:
        backend = "ref_ofast" if "ref_ofast" in avail else ("ref" if "ref" in avail else "port")
    whole = wl is not None and "golden" in wl  # the reference's own sets are small enough to run as they are
    pos, world, fixed, stim = workload_inputs(wl) if whole else make_lattice(CPU_SAMPLE_DIMS, (wl or {}).get("jitter", 0.0))
    sim = CpuSim(backend, capacity=len(pos), world=world)
    sim.Init_Fluid(pos)
    sim.set_fields(fixed=fixed, stim=stim)
    if quadratic:
        sim.flip_quadratic()
    sim.Animation(max(warmup, 1))
    t0 = time.perf_counter()
    sim.Animation(steps)
    dt = time.perf_counter() - t0
    if dump_dir:
        dump_outputs(dump_dir, sim.particles())
    kind = "reference" if backend.startswith("ref") else "port"
    flags = {"ref_ofast": "g++ -Ofast (the reference Makefile's flags)", "ref": "g++ -O2 -ffp-contract=off", "port": "gcc -O2 -ffp-contract=off"}[backend]
    d = CPU_SAMPLE_DIMS
    what = f"the whole workload ({len(pos)} particles)" if whole else f"{d[0]}x{d[1]}x{d[2]} = {len(pos)}-particle lattice of the same spacing and shape-matching mode"
    return {"value": len(pos) * steps / dt, "unit": UNIT, "cores": 1, "kind": kind, "host_cores_available": os.cpu_count(),
            "sample": f"{what}, {steps} steps, "
                      f"{flags}, 1 thread (the reference is single-threaded)", "ms_per_step": dt / steps * 1e3}


def run_reference(args, wl, rank, world_size):
    if rank != 0:
        return
    whole = "golden" in wl
    steps = args.steps  # each "step" of this arm is one CPU step of the bounded sample (~0.9 s at 1M)
    warmup = min(args.warmup, 100 if whole else 5)
    base = cpu_reference_rate(wl["quadratic"], steps, warmup, wl=wl, dump_dir=args.dump_outputs)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "sample": base["sample"]},
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
def stim_box_of(pos, dims):
    """The end slab the masks stimulate (inputs.lattice_masks: the first 8 x-layers) as an axis-aligned box."""
    from sph_sm_monodomain_b200 import inputs

    s = float(inputs.KERNEL_H) * 0.9
    x0 = float(pos[:, 0].min())
    return (-1.0, -1.0, -1.0), (x0 + 8 * s - 0.5 * s, 1e9, 1e9)


def pacing_schedule(start, nsteps, period, off_after):
    """The pacing protocol of BASELINE configs[4] as a list of actions covering steps [start, start + nsteps): ("stim",) before every
    step k with k % period == 0, ("off",) before every step with k % period == off_after, ("run", m) for m uninterrupted steps."""
    out, k, end = [], start, start + nsteps
    while k < end:
        ph = k % period
        if ph == 0:
            out.append(("stim",))
        if ph == off_after:
            out.append(("off",))
        nxt = min(end, k - ph + (off_after if ph < off_after else period))
        out.append(("run", nxt - k))
        k = nxt
    return out


def make_sim(pos, world, fixed, stim, quadratic, device, world_size, rank, dist, torch, parts=None, axis=None, **kw):
    """A handle with the workload loaded; with world_size > 1 also its NCCL communicator (id broadcast from rank 0) and slab."""
    from sph_sm_monodomain_b200 import Sim

    n_total = len(pos)
    if world_size > 1:
        sim = Sim(capacity=n_total, world=world, device=device, diagnostics=False, slab_axis=axis, **kw)
    else:
        sim = Sim(capacity=n_total, world=world, device=device, diagnostics=False, **kw)
    sim.Init_Fluid(pos)
    sim.set_masks(fixed, stim)
    if quadratic:
        sim.flip_quadratic()
    if world_size > 1:
        ident = torch.zeros(128, dtype=torch.uint8, device=f"cuda:{device}")
        if rank == 0:
            ident.copy_(torch.frombuffer(bytearray(Sim.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(ident, 0)
        sim.comm_init(world_size, rank, bytes(ident.cpu().numpy().tobytes()))
        sim.set_slab(*parts[rank])
    return sim


def mg_parity_check(device, world_size, rank, dist, torch):
    """Multi-GPU correctness inside the bench run: a ~55k-particle jittered lattice stepped 10 times through the slab path on
    all ranks (its own NCCL communicator, the same library code the timed region runs) and on rank 0's GPU alone; with the
    canonical in-cell order both runs sum in the same order, so the positions must agree bit for bit."""
    from sph_sm_monodomain_b200 import Sim, inputs, slabs

    dims, steps = (96, 24, 24), 10
    pos, world = inputs.lattice(*dims, jitter=0.05)
    fixed, stim = inputs.lattice_masks(pos, dims[0], 4)
    fixed, stim = fixed.astype(np.uint8), np.where(stim, np.float32(300), np.float32(0)).astype(np.float32)
    n = len(pos)
    axis = slabs.slab_axis_for(world)
    parts = slabs.partition_planes(slabs.plane_histogram(pos, axis, slabs.num_planes(world, axis)), world_size)

    def canonical(s):
        p = s.get_params()
        p.reserved[1] = 1
        s._ck(s.lib.sphsm_set_params(s.h, p))

    sim = Sim(capacity=n, world=world, device=device, diagnostics=False, slab_axis=axis)
    sim.Init_Fluid(pos)
    sim.set_masks(fixed, stim)
    canonical(sim)
    ident = torch.zeros(128, dtype=torch.uint8, device=f"cuda:{device}")
    if rank == 0:
        ident.copy_(torch.frombuffer(bytearray(Sim.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(ident, 0)
    sim.comm_init(world_size, rank, bytes(ident.cpu().numpy().tobytes()))
    sim.set_slab(*parts[rank])
    sim.Animation(steps)
    sim.sync()
    ids, xyz = sim.download_owned()
    cnt = torch.tensor([len(ids)], device=f"cuda:{device}")
    cnts = [torch.zeros_like(cnt) for _ in range(world_size)]
    dist.all_gather(cnts, cnt)
    cap = int(max(c.item() for c in cnts))
    pad_ids = torch.full((cap,), -1, dtype=torch.int32, device=f"cuda:{device}")
    pad_xyz = torch.zeros((cap, 3), dtype=torch.float32, device=f"cuda:{device}")
    pad_ids[: len(ids)] = torch.from_numpy(ids).to(pad_ids.device)
    pad_xyz[: len(ids)] = torch.from_numpy(xyz).to(pad_xyz.device)
    all_ids = [torch.zeros_like(pad_ids) for _ in range(world_size)]
    all_xyz = [torch.zeros_like(pad_xyz) for _ in range(world_size)]
    dist.all_gather(all_ids, pad_ids)
    dist.all_gather(all_xyz, pad_xyz)
    sim.close()
    res = None
    if rank == 0:
        got = np.full((n, 3), np.nan, np.float32)
        seen = np.zeros(n, np.int32)
        for i, x in zip(all_ids, all_xyz):
            i, x = i.cpu().numpy(), x.cpu().numpy()
            m = i >= 0
            got[i[m]] = x[m]
            seen[i[m]] += 1
        single = Sim(capacity=n, world=world, device=device, diagnostics=False, slab_axis=axis)
        single.Init_Fluid(pos)
        single.set_masks(fixed, stim)
        canonical(single)
        single.Animation(steps)
        i1, x1 = single.download_owned()
        single.close()
        ref = np.empty((n, 3), np.float32)
        ref[i1] = x1
        once = bool((seen == 1).all())
        res = {"particles": n, "steps": steps, "ranks": world_size, "every_particle_owned_once": once,
               "bit_identical": bool(once and np.array_equal(got, ref)),
               "max_rel": float(np.abs(got.astype(np.float64) - ref).max() / np.abs(ref).max()) if once else None,
               "owned_per_rank": [int(c.item()) for c in cnts]}
    dist.barrier()
    return res


def quick_measure(key, device, steps=30, warmup=60):
    """Device-resident ms/step of another configuration in this process (the `also` block of the default N = 1 line)."""
    from sph_sm_monodomain_b200 import Sim

    wl = parse_workload(key)
    pos, world, fixed, stim = workload_inputs(wl)
    sim = Sim(capacity=len(pos), world=world, device=device, diagnostics=False)
    sim.Init_Fluid(pos)
    sim.set_masks(fixed, stim)
    if wl["quadratic"]:
        sim.flip_quadratic()
    sim.Animation(warmup)
    sim.sync()
    sim.Animation(steps)
    sim.sync()
    ms = sim.last_step_ms() / steps
    groups = sim.profile_step(5)
    sim.close()
    return {"workload": wl["name"], "particles": len(pos), "steps": steps, "warmup": warmup, "ms_per_step": ms,
            "value": len(pos) / (ms * 1e-3), "unit": UNIT,
            "kernel_group_ms": {k: v for k, v in groups.items() if v > 0}}


def run_ours(args, wl, rank, world_size, local_rank):
    import torch

    from sph_sm_monodomain_b200 import _capi
    import ctypes as C

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the step has no CPU fallback")
    dist = None
    if world_size > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    device = local_rank
    mg_parity = mg_parity_check(device, world_size, rank, dist, torch) if world_size > 1 else None
    pos, world, fixed, stim = workload_inputs(wl)
    n_total = len(pos)
    parts = axis = None
    if world_size > 1:
        # slab decomposition along the longest axis (SURVEY.md §8e): every rank uploads the global set, then keeps the
        # cell planes the balanced partition gives it; halos / migrants travel by ncclSend/ncclRecv inside sphsm_step
        from sph_sm_monodomain_b200 import slabs

        axis = slabs.slab_axis_for(world)
        npl = slabs.num_planes(world, axis)
        parts = slabs.partition_planes(slabs.plane_histogram(pos, axis, npl), world_size)
    sim = make_sim(pos, world, fixed, stim, wl["quadratic"], device, world_size, rank, dist, torch, parts, axis)
    if world_size > 1:
        info = sim.comm_info()
        n_local = info["own_end"] - info["own_begin"]
    else:
        n_local = sim.n
    pacing = wl.get("pacing")
    box_lo, box_hi = stim_box_of(pos, wl["dims"]) if pacing else (None, None)

    def barrier():
        if dist is not None:
            dist.barrier()
        sim.sync()
        torch.cuda.synchronize()

    def advance(nsteps, start):
        """nsteps steps from step number `start`; a pacing workload (configs[4]) stimulates the end slab every `period` steps
        and calls turnOffStim `off_after` steps later (SURVEY.md 8d.5; reference cpp:704-717, 764-783) inside the timed region."""
        if not pacing:
            sim.Animation(nsteps)
            return
        for act in pacing_schedule(start, nsteps, *pacing):
            if act[0] == "stim":
                sim.set_stim_box(box_lo, box_hi, 300.0)
            elif act[0] == "off":
                sim.turnOffStim()
            else:
                sim.Animation(act[1])

    # ---- device-resident throughput -----------------------------------------------------------------------------
    # clocks / throttle reasons are sampled from before the warm-up until after the timed region (a strong-scaled timed
    # region can be shorter than one nvidia-smi sampling period, so the warm-up steps keep the GPU under the same load);
    # the warm-up is the same number of steps for every N
    sampler = ClockSampler(device)
    sampler.start()
    prewarm = max(args.warmup, FIXED_WARMUP)
    advance(prewarm, 0)
    barrier()
    sim.reset_launch_count()
    barrier()
    t0 = time.perf_counter()
    sim.timer_mark(0)
    advance(args.steps, prewarm)
    sim.timer_mark(1)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ev_ms = sim.timer_ms()
    clocks = sampler.stop()
    launches = sim.launch_count()
    if args.dump_outputs:  # after reading the launch count (the download is a launch), before the steps below move the state on
        dump_outputs(args.dump_outputs, sim.particles())
    t = torch.tensor([ev_ms, wall_ms], dtype=torch.float64, device=f"cuda:{device}")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ev_ms, wall_ms = float(t[0]), float(t[1])
    value = n_total * args.steps / (ev_ms * 1e-3)

    # ---- per-kernel-group device times (CUDA events on the handle's stream) -> roofline of the dominant kernel -----
    prof_steps = max(3, min(args.steps, 10))
    groups = sim.profile_step(prof_steps)
    peak, peak_src = measured_peak_gbs()
    pb_ms = groups[PASS_B_NAME]
    if world_size > 1:
        info = sim.comm_info()
        n_local = info["own_end"] - info["own_begin"]
    achieved = PASS_B_BYTES_PER_PARTICLE * n_local / (pb_ms * 1e-3) / 1e9
    roofline = {"kernel": "k_pass_b4 (fused cell model + force + Laplacian + integration"
                          + (" + next step's cell key / rank / count)" if world_size == 1 else ")"),
                "bound": "hbm", "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_particle": PASS_B_BYTES_PER_PARTICLE,
                "extra_bytes_per_particle_not_counted": {"next step's sort input filed by the same kernel (key + rank)": PASS_B_FUSED_HASH_BYTES if world_size == 1 else 0},
                "particles_per_launch": int(n_local), "ms_per_launch": pb_ms,
                "whole_step": {"achieved": STEP_BYTES_PER_PARTICLE * n_total / (ev_ms / args.steps * 1e-3) / 1e9,
                               "algorithmic_bytes_per_particle": STEP_BYTES_PER_PARTICLE, "peak": peak * world_size,
                               "peak_note": f"{world_size} x the single-GPU measured peak"},
                "kernel_group_ms": groups}
    roofline["whole_step"]["frac"] = roofline["whole_step"]["achieved"] / (peak * world_size)
    traffic_file = os.path.join(ROOT, "profiles", "pass_b_traffic.json")
    if world_size == 1 and os.path.exists(traffic_file):  # (an ncu capture of one launch at N = 1; no per-N capture exists)
        with open(traffic_file) as fh:
            tr = json.load(fh)
        if tr.get("workload") == wl["key"]:
            roofline["traffic"] = tr.get("dram_bytes_per_launch")

    # ---- end to end through the C-ABI with host buffers ---------------------------------------------------------------
    # the owned count is only known on the device, so a fixed window crosses PCIe: what the library bounds the count by
    own_cap = n_total if world_size == 1 else min(n_total, n_local + 2 * sim.comm_info()["halo_capacity"] + 4096)
    stim_by_id = stim.copy()
    stim_host = torch.zeros((own_cap,), dtype=torch.float32).pin_memory()
    pos_host = torch.empty((own_cap, 3), dtype=torch.float32).pin_memory()
    ids_host = torch.empty((own_cap,), dtype=torch.int32).pin_memory()
    cnt_host = torch.zeros((4,), dtype=torch.int32).pin_memory()
    lib = sim.lib
    FP, IP = C.POINTER(C.c_float), C.POINTER(C.c_int)
    stim_ptr = C.cast(stim_host.data_ptr(), FP)
    pos_ptr = C.cast(pos_host.data_ptr(), FP)
    ids_ptr = C.cast(ids_host.data_ptr(), IP)
    cnt_ptr = C.cast(cnt_host.data_ptr(), IP)
    e2e_steps = max(3, min(args.steps, 20))
    sent = {"n": 0}

    stim_all = torch.from_numpy(stim.copy()).pin_memory() if world_size == 1 else None
    stim_all_ptr = C.cast(stim_all.data_ptr(), FP) if world_size == 1 else None

    def e2e_step():
        # The library's asynchronous I/O calls: every step's inputs cross PCIe host -> device and every step's result
        # device -> host, on copy streams beside the compute stream (the result of step k lands while step k+1 runs).
        if world_size == 1:
            # H2D: the per-particle stimulation array (4 B / particle); D2H: positions in the caller's order (12 B / particle)
            _capi.check(lib, sim.h, lib.sphsm_set_masks_async(sim.h, None, stim_all_ptr, n_total))
            _capi.check(lib, sim.h, lib.sphsm_step(sim.h, 1))
            _capi.check(lib, sim.h, lib.sphsm_download_positions_async(sim.h, pos_ptr, n_total))
            return
        # H2D: the stimulation value of every particle the rank owns, in the order of its last download (4 B / particle)
        _capi.check(lib, sim.h, lib.sphsm_set_stim_owned_async(sim.h, stim_ptr, sent["n"]))
        _capi.check(lib, sim.h, lib.sphsm_step(sim.h, 1))
        # D2H: (id, position) of the particles the rank owns, 16 B / particle
        _capi.check(lib, sim.h, lib.sphsm_download_owned_async(sim.h, ids_ptr, pos_ptr, own_cap, cnt_ptr))

    if world_size > 1:
        # prime: one download tells the host which particles it owns and in which order; their stimulation values follow that order
        _capi.check(lib, sim.h, lib.sphsm_download_owned_async(sim.h, ids_ptr, pos_ptr, own_cap, cnt_ptr))
        _capi.check(lib, sim.h, lib.sphsm_sync(sim.h))
        sent["n"] = min(int(cnt_host[0]), own_cap)
        stim_host[: sent["n"]] = torch.from_numpy(stim_by_id[ids_host.numpy()[: sent["n"]]])
    for _ in range(2):
        e2e_step()
    _capi.check(lib, sim.h, lib.sphsm_sync(sim.h))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    _capi.check(lib, sim.h, lib.sphsm_sync(sim.h))  # the last step's result is in host memory
    barrier()
    e2e_s = time.perf_counter() - t0
    n_read = n_total if world_size == 1 else min(int(cnt_host[0]), own_cap)
    te = torch.tensor([e2e_s, float(sent["n"]), float(own_cap)], dtype=torch.float64, device=f"cuda:{device}")
    tsum = te.clone()
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    h2d = 4 * n_total if world_size == 1 else 4 * int(tsum[1])
    d2h = 12 * n_total if world_size == 1 else 16 * int(tsum[2]) + 4 * world_size
    e2e = {"value": n_total * e2e_steps / float(te[0]), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
           "protocol": ("per step: sphsm_set_masks_async(stim, 4 B per particle) from pinned host memory -> sphsm_step(1) -> "
                        "sphsm_download_positions_async (12 B per particle)" if world_size == 1 else
                        "per step and rank: sphsm_set_stim_owned_async (stimulation of the rank's own particles, 4 B each, pinned host memory) -> "
                        "sphsm_step(1) -> sphsm_download_owned_async (ids + positions of the rank's particles, 16 B each, a fixed window of the slab's "
                        "population bound because the owned count is only known on the device)")
                       + " to pinned host memory; copies overlap the next step on the library's copy streams, the timed region "
                         "ends when the last result is in host memory (sphsm_sync); bytes summed over ranks"}
    assert np.isfinite(pos_host.numpy()[:n_read]).all()
    push_exchange = push_allreduce = None
    if world_size > 1:
        push_exchange = ("push: the packing kernel stores into the neighbour's receive slot (CUDA IPC over NVLink), flag word + polling kernel"
                         if sim.push_exchange() else "ncclSend / ncclRecv of full-capacity messages")
        push_allreduce = ("push: one kernel stores the rank's sums into every rank's landing area (CUDA IPC over NVLink), waits for the others' and adds in rank order"
                          if sim.push_allreduce() else "ncclAllReduce")

    also = None
    if rank == 0 and world_size == 1 and wl["key"] == "8m" and not args.no_also:
        sim.close()
        also = {}
        for key in ("1m", "8m_jitter", "cfg1", "cfg2"):
            also[key] = quick_measure(key, device, steps=30 if key in ("1m", "8m_jitter") else 200, warmup=60 if key in ("1m", "8m_jitter") else 300)

    if rank == 0:
        cpu = cpu_reference_rate(wl["quadratic"], CPU_SAMPLE_STEPS, 1, wl=wl) if not args.no_cpu_baseline else None
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ev_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": wl["name"], "particles": n_total, "world": [round(w, 4) for w in world],
                           "shape_matching": "quadratic" if wl["quadratic"] else "linear", "parallelism": f"slab{world_size}",
                           "l2": ("inputs larger than L2 (no flush): %.0f MB of persistent state" % (n_total * 68 / 1e6)) if n_total * 68 > 126e6
                                 else ("persistent state (%.1f MB) fits the 126 MB L2: the timed steps run cache-resident, as any run of this size "
                                       "does (each step consumes the previous step's output); not the headline configuration" % (n_total * 68 / 1e6)),
                           "warmup_steps_run": prewarm},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "wall_ms_per_step": wall_ms / args.steps,
                "roofline": roofline}
        if world_size > 1:
            line["config"]["exchange1"] = push_exchange
            line["config"]["moment_allreduce"] = push_allreduce
        if pacing:
            line["config"]["pacing"] = {"stimulate_every": pacing[0], "turn_off_after": pacing[1], "inside_timed_region": True}
        if mg_parity is not None:
            line["mg_parity"] = mg_parity
        if also is not None:
            line["also"] = also
        if cpu:
            line["cpu_baseline"] = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "host_cores_available")}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="8m")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the quick measurements of the other configurations (N = 1, default workload)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the particle state after the last timed step as DIR/<field>.npy (float32; a seeded sample of "
                         f"{DUMP_MAX_PARTICLES} particles for larger sets)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world_size > 1 and args.impl == "ours":
        ap.error("--dump-outputs needs a single-GPU run: in slab mode each rank holds only its own particles")
    wl = parse_workload(args.workload)
    if args.impl == "reference":
        run_reference(args, wl, rank, world_size)
    else:
        run_ours(args, wl, rank, world_size, local_rank)


if __name__ == "__main__":
    main()
