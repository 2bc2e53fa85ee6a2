#!/usr/bin/env python
"""The electrograms on the NCCL slab path (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29542 tools/egm_mg.py

Every rank steps its slab through sphsm_step with electrograms on (8 electrodes around and inside the body, softening = h),
under the pacing protocol of tests/test_gpu_egm.py.  Before and after every step the global state is assembled from the ranks'
owned downloads (an all-reduce of the owned values).  Rank 0 sums the all-gathered per-rank rows in rank order
(slabs.merge_electrograms) and checks every row against the host formula (tests/test_egm_cpu.host_egm) on that global state:
|phi - phi_host| <= 1e-5 * A_e, with some row well above that bound.  Prints one JSON line; exits non-zero on a mismatch."""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import pacing_schedule  # noqa: E402
from sph_sm_monodomain_b200 import PARTICLE_DTYPE, Sim, inputs, slabs  # noqa: E402
from tests.test_egm_cpu import host_egm  # noqa: E402

PERIOD, OFF_AFTER, STEPS = 60, 20, 90

rank, world_size, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
dims = (96, 24, 24)
pos, world = inputs.lattice(*dims, jitter=0.05)
fixed, stim = inputs.lattice_masks(pos, dims[0], 4)
stimv = np.where(stim, np.float32(300), np.float32(0)).astype(np.float32)
n = len(pos)
axis = slabs.slab_axis_for(world)
parts = slabs.partition_planes(slabs.plane_histogram(pos, axis, slabs.num_planes(world, axis)), world_size)
sim = Sim(capacity=n, world=world, device=local, diagnostics=False, slab_axis=axis)
sim.Init_Fluid(pos)
sim.set_masks(fixed.astype(np.uint8), stimv)
ident = torch.zeros(128, dtype=torch.uint8, device=f"cuda:{local}")
if rank == 0:
    ident.copy_(torch.frombuffer(bytearray(Sim.comm_unique_id()), dtype=torch.uint8))
dist.broadcast(ident, 0)
sim.comm_init(world_size, rank, bytes(ident.cpu().numpy().tobytes()))
sim.set_slab(*parts[rank])
prm = sim.get_params()
h, cb = float(prm.kernel_h), float(prm.bspline_constant)
lo, hi = pos.min(axis=0), pos.max(axis=0)
c, ext = (lo + hi) / 2, hi - lo
el = np.array([c + [-0.6 * ext[0], 0, 0], c + [0.6 * ext[0], 0, 0], c + [0, -0.6 * ext[1] - h, 0], c + [0, 0.6 * ext[1] + h, 0],
               c + [0, 0, -0.6 * ext[2] - h], c + [0, 0, 0.6 * ext[2] + h], c, c + 20 * ext.max()], np.float32)
sim.egm_start(el, rows=STEPS)


def global_state():
    """(pos, Vm, mass, dens) of every particle from the owned downloads of every rank."""
    buf = np.zeros(n, PARTICLE_DTYPE)
    sim._ck(sim.lib.sphsm_download_aos(sim.h, buf.ctypes.data_as(C.c_void_p), n, PARTICLE_DTYPE.itemsize))
    ids, _ = sim.download_owned()
    vals = np.zeros((n, 7), np.float32)
    vals[ids, :3] = buf["pos"][ids]
    vals[ids, 3] = buf["Vm"][ids]
    vals[ids, 4] = buf["mass"][ids]
    vals[ids, 5] = buf["dens"][ids]
    vals[ids, 6] = 1.0
    t = torch.from_numpy(vals).cuda()
    dist.all_reduce(t)  # every particle is owned by exactly one rank: the sum is its value
    g = t.cpu().numpy()
    assert (g[:, 6] == 1.0).all(), "a particle is owned by no rank or by two"
    return g


pre = global_state()
refs = []
for act in pacing_schedule(0, STEPS, PERIOD, OFF_AFTER):
    if act[0] == "stim":
        sim.set_masks(None, stimv)
    elif act[0] == "off":
        sim.turnOffStim()
    else:
        for _ in range(act[1]):
            sim.Animation(1)
            post = global_state()
            if rank == 0:
                refs.append(host_egm(pre[:, :3], pre[:, 3], post[:, 4], post[:, 5], el, 1.0, h, h, world, cb))
            pre = post
        continue
    pre = global_state()

first, phi = sim.electrogram()
t = torch.from_numpy(np.concatenate([[float(first)], phi.reshape(-1)])).cuda()
ts = [torch.zeros_like(t) for _ in range(world_size)]
dist.all_gather(ts, t)
res = {"ranks": world_size, "particles": n, "steps": STEPS, "electrodes": len(el)}
if rank == 0:
    rows = [(int(a[0]), a[1:].reshape(phi.shape)) for a in (x.cpu().numpy() for x in ts)]
    f, merged = slabs.merge_electrograms(rows)
    ref = np.stack([r for r, _ in refs])
    scale = np.stack([a for _, a in refs])
    res["first_step"] = f
    res["max_err_over_scale"] = float((np.abs(merged - ref) / scale).max())
    res["max_phi_over_bound"] = float((np.abs(merged) / (1e-5 * scale)).max())
    ok = f == 1 and merged.shape == ref.shape and res["max_err_over_scale"] <= 1e-5 and res["max_phi_over_bound"] > 100
    res["egm_mg"] = "ok" if ok else "mismatch"
    print(json.dumps(res))
    sys.stdout.flush()
dist.barrier()
status = res.get("egm_mg", "ok") if rank == 0 else "ok"
dist.destroy_process_group()
sys.exit(0 if status == "ok" else 1)
