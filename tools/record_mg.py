#!/usr/bin/env python
"""The Vm recorder on the NCCL slab path (run under torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 tools/record_mg.py

Every rank steps its slab through sphsm_step with recording on, under the pacing protocol (stimulus on the end slab every 60
steps, turnOffStim 20 steps later; thresholds as in tests/test_gpu_record.py).  After every step and every call between steps the
global Vm is assembled from the ranks' owned downloads (an all-reduce of the owned values).  Each rank checks its own maps against
the host rule applied to the particles it integrated in each step (its owned set after that step); rank 0 checks the merged maps
(slabs.merge_activation over the all-gathered per-rank maps) and the merged probe traces against the whole-set reference.
Prints one JSON line; exits non-zero on a mismatch."""
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
from tests.test_record_cpu import host_crossings  # noqa: E402

VM = -94.2
PERIOD, OFF_AFTER, STEPS = 60, 20, 150

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
probes = np.unique(np.linspace(0, n - 1, 64).astype(np.int32))
sim.record_start(VM, VM, probes=probes, trace_rows=STEPS)


def global_state():
    """(global Vm, global pos, this rank's owned mask) from the owned downloads of every rank."""
    buf = np.zeros(n, PARTICLE_DTYPE)
    sim._ck(sim.lib.sphsm_download_aos(sim.h, buf.ctypes.data_as(C.c_void_p), n, PARTICLE_DTYPE.itemsize))
    ids, _ = sim.download_owned()
    mine = np.zeros(n, bool)
    mine[ids] = True
    vals = np.zeros((n, 5), np.float32)
    vals[ids, :3] = buf["pos"][ids]
    vals[ids, 3] = buf["Vm"][ids]
    vals[ids, 4] = 1.0
    t = torch.from_numpy(vals).cuda()
    dist.all_reduce(t)  # every particle is owned by exactly one rank: the sum is its value
    g = t.cpu().numpy()
    assert (g[:, 4] == 1.0).all(), "a particle is owned by no rank or by two"
    return g[:, 3].copy(), g[:, :3].copy(), mine


pre, _, _ = global_state()
mine_series, all_series, posts, owned = [], [], [], []
for act in pacing_schedule(0, STEPS, PERIOD, OFF_AFTER):
    if act[0] == "stim":
        sim.set_masks(None, stimv)
    elif act[0] == "off":
        sim.turnOffStim()
    else:
        for _ in range(act[1]):
            sim.Animation(1)
            post, p, mine = global_state()
            step = sim.total_time_steps
            all_series.append((step, pre, post))
            mine_series.append((step, np.where(mine, pre, np.nan), np.where(mine, post, np.nan)))
            posts.append((p[probes], post[probes]))
            owned.append(mine[probes])
            pre = post
        continue
    pre, _, _ = global_state()

got = sim.activation(n)
own_ref = host_crossings(mine_series, VM, VM, n)
ok_rank = all(np.array_equal(got[k], own_ref[k]) for k in slabs.ACTIVATION_KEYS)
first, xyzv, own = sim.probe_trace()
ok_rank = ok_rank and first == 1 and np.array_equal(own, np.stack(owned))

maps = torch.from_numpy(np.stack([got[k] for k in slabs.ACTIVATION_KEYS])).cuda()
gathered = [torch.zeros_like(maps) for _ in range(world_size)]
dist.all_gather(gathered, maps)
tr = torch.from_numpy(np.concatenate([xyzv.reshape(-1), own.reshape(-1).astype(np.float32)])).cuda()
trs = [torch.zeros_like(tr) for _ in range(world_size)]
dist.all_gather(trs, tr)
oks = torch.tensor([1 if ok_rank else 0], device="cuda")
dist.all_reduce(oks)
res = {"ranks": world_size, "particles": n, "steps": STEPS, "every_rank_matches_its_own_reference": int(oks.item()) == world_size}
if rank == 0:
    parts_m = [dict(zip(slabs.ACTIVATION_KEYS, g.cpu().numpy())) for g in gathered]
    merged = slabs.merge_activation(parts_m)
    ref = host_crossings(all_series, VM, VM, n)
    res["merged_maps_equal"] = all(np.array_equal(merged[k], ref[k]) for k in slabs.ACTIVATION_KEYS)
    res["n_up_total"] = int(merged["n_up"].sum())
    res["not_vacuous"] = bool((merged["n_up"] >= 2).any() and (merged["last_down"] >= 0).any() and (merged["first_up"] < 0).any())
    K, R = len(probes), len(xyzv)
    tparts = []
    for t in trs:
        a = t.cpu().numpy()
        tparts.append((1, a[: R * K * 4].reshape(R, K, 4), a[R * K * 4:].reshape(R, K) > 0))
    f, mx, mo = slabs.merge_traces(tparts)
    refx = np.concatenate([np.stack([p for p, _ in posts]), np.stack([v for _, v in posts])[..., None]], axis=2).astype(np.float32)
    res["merged_traces_equal"] = bool(mo.all() and mx.tobytes() == refx.tobytes())
    ok = res["every_rank_matches_its_own_reference"] and res["merged_maps_equal"] and res["not_vacuous"] and res["merged_traces_equal"]
    res["record_mg"] = "ok" if ok else "mismatch"
    print(json.dumps(res))
    sys.stdout.flush()
dist.barrier()
status = res.get("record_mg", "ok") if rank == 0 else ("ok" if ok_rank else "mismatch")
dist.destroy_process_group()
sys.exit(0 if status == "ok" else 1)
