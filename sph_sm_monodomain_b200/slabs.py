"""Host-side slab decomposition for the multi-GPU path (SURVEY.md §8e): which axis to cut, the cell plane of a position
(exactly as the device computes it), per-plane particle counts and the balanced partition into contiguous plane ranges, the exact merge of the per-rank results of
the Vm recorder (Sim.activation / Sim.probe_trace) and the sum of the per-rank electrograms (Sim.electrogram).  Pure numpy; per-rank values are combined by the caller (torch.distributed in
bench.py and tools/record_mg.py, LocalGroup for virtual ranks)."""
from __future__ import annotations

import numpy as np

KERNEL_H = np.float32(0.04)


def slab_axis_for(world) -> int:
    """Cut along the longest axis (ties -> the lowest axis index)."""
    return int(np.argmax(np.asarray(world, dtype=np.float64)))


def num_planes(world, axis: int, h=KERNEL_H) -> int:
    """Grid_Size along the axis, ceil(World / Cell_Size) in float like the reference ctor (cpp:32-35)."""
    return int(np.ceil(np.float32(world[axis]) / np.float32(h)))


def plane_of(pos: np.ndarray, axis: int, h=KERNEL_H) -> np.ndarray:
    """Cell plane of every position: float32 division by Cell_Size and C truncation (cpp:127-134)."""
    return (np.asarray(pos, np.float32)[:, axis] / np.float32(h)).astype(np.int64)


def plane_histogram(pos: np.ndarray, axis: int, nplanes: int, h=KERNEL_H) -> np.ndarray:
    pl = plane_of(pos, axis, h)
    pl = pl[(pl >= 0) & (pl < nplanes)]
    return np.bincount(pl, minlength=nplanes).astype(np.int64)


def partition_planes(hist: np.ndarray, nranks: int):
    """Contiguous plane ranges [(lo, hi)] covering [0, len(hist)), every rank at least one plane, particle counts as
    even as plane granularity allows (cut where the prefix sum crosses k/nranks of the total)."""
    hist = np.asarray(hist, np.int64)
    nplanes = len(hist)
    if nranks < 1 or nranks > nplanes:
        raise ValueError(f"cannot cut {nplanes} planes into {nranks} slabs")
    prefix = np.concatenate([[0], np.cumsum(hist)])
    total = int(prefix[-1])
    cuts = [0]
    for k in range(1, nranks):
        target = total * k / nranks
        c = int(np.searchsorted(prefix, target, side="left"))
        if c > 0 and abs(prefix[c - 1] - target) <= abs(prefix[min(c, nplanes)] - target):
            c -= 1
        c = max(c, cuts[-1] + 1)             # at least one plane per rank so far
        c = min(c, nplanes - (nranks - k))   # and one for each rank still to come
        cuts.append(c)
    cuts.append(nplanes)
    return [(cuts[k], cuts[k + 1]) for k in range(nranks)]


ACTIVATION_KEYS = ("first_up", "last_up", "last_down", "n_up")


def merge_activation(parts):
    """Merge per-rank activation maps (dicts of int32 arrays by original id, as Sim.activation returns them).  Each crossing is
    recorded by exactly one rank, so the merge is exact: first_up = minimum over the ranks that set it, last_up / last_down =
    maximum, n_up = sum; a step no rank set stays -1."""
    parts = list(parts)
    if not parts:
        raise ValueError("no parts to merge")
    fu = np.stack([np.asarray(p["first_up"], np.int32) for p in parts])
    big = np.iinfo(np.int32).max
    first = np.where(fu >= 0, fu, big).min(axis=0)
    out = {"first_up": np.where(first == big, -1, first).astype(np.int32)}
    for k in ("last_up", "last_down"):
        out[k] = np.stack([np.asarray(p[k], np.int32) for p in parts]).max(axis=0).astype(np.int32)
    out["n_up"] = np.stack([np.asarray(p["n_up"], np.int32) for p in parts]).sum(axis=0, dtype=np.int64).astype(np.int32)
    return out


def merge_traces(parts):
    """Merge per-rank probe traces (first_step, xyzv (rows, K, 4), owned (rows, K)) as Sim.probe_trace returns them: every entry
    comes from the rank that integrated that probe in that step.  All parts must cover the same steps; an entry owned by two ranks
    is an error.  Returns (first_step, xyzv, owned)."""
    parts = list(parts)
    if not parts:
        raise ValueError("no parts to merge")
    first = int(parts[0][0])
    xyzv = np.zeros(np.shape(parts[0][1]), np.float32)
    owned = np.zeros(xyzv.shape[:2], bool)
    for f, x, o in parts:
        x, o = np.asarray(x, np.float32), np.asarray(o, bool)
        if int(f) != first or x.shape != xyzv.shape or o.shape != owned.shape:
            raise ValueError("probe traces of different steps or shapes")
        if (owned & o).any():
            raise ValueError("a probe entry is owned by two ranks")
        xyzv[o] = x[o]
        owned |= o
    return first, xyzv, owned


def merge_electrograms(parts):
    """Sum per-rank electrograms (first_step, phi (rows, E)) as Sim.electrogram returns them, in rank order: each rank holds the
    sum over the particles it integrated.  All parts must cover the same steps and electrodes.  Returns (first_step, phi)."""
    parts = list(parts)
    if not parts:
        raise ValueError("no parts to merge")
    first = int(parts[0][0])
    phi = np.zeros(np.shape(parts[0][1]), np.float64)
    for f, p in parts:
        p = np.asarray(p, np.float64)
        if int(f) != first or p.shape != phi.shape:
            raise ValueError("electrograms of different steps or shapes")
        phi += p
    return first, phi
