"""CPU: the electrograms' host-side pieces — the electrogram restated on the host in float64 (the reference the GPU tests compare
the device rows with) and the sum of per-rank rows (slabs.merge_electrograms)."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

from sph_sm_monodomain_b200 import slabs


def host_pairs(pos, h, world):
    """The pairs (i, j), i != j, pass B sums over: j in the 27-cell stencil of i (cell = float32 pos / h, truncated, inside the
    grid of ceil(world / h) cells per axis), r2 > 1e-12 and r / h < 2 in float32 as the strict branch of k_pass_b evaluates them.
    Returns i, j and the B_spline_2 factor without its constant (float32 q)."""
    pos = np.asarray(pos, np.float32)
    h32 = np.float32(h)
    g = np.ceil(np.asarray(world, np.float32) / h32).astype(np.int64)
    cell = np.trunc(pos / h32).astype(np.int64)
    inside = ((cell >= 0) & (cell < g)).all(axis=1)
    pairs = cKDTree(pos.astype(np.float64)).query_pairs(2.0 * float(h) * (1 + 1e-5), output_type="ndarray")
    i = np.concatenate([pairs[:, 0], pairs[:, 1]])
    j = np.concatenate([pairs[:, 1], pairs[:, 0]])
    d = pos[i] - pos[j]  # float32 differences, r2 = (dx dx + dy dy) + dz dz in float32
    r2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    q = np.sqrt(r2) / h32
    keep = inside[i] & inside[j] & (np.abs(cell[i] - cell[j]) <= 1).all(axis=1) & (r2 > np.float32(1e-12)) & (q < np.float32(2.0))
    i, j, q = i[keep], j[keep], q[keep].astype(np.float64)
    b2 = np.where(q < 1.0, -3.0 + 4.5 * q, 1.5 * (2.0 - q))
    return i, j, b2


def host_egm(pos, vm, mass, dens, electrodes, gain, softening, h, world, c_bspline):
    """phi_e = gain * sum_i vol_i L_i / sqrt(|x_i - e|^2 + eps^2), L_i = sum_j vol_j (Vm_j - Vm_i) B2(r_ij), in float64.
    pos / vm: the state the step started from; mass / dens: the step's (vol = mass / dens in float32, as the device forms it).
    Also returns A_e = gain * sum_i sum_j |vol_i vol_j (Vm_j - Vm_i) B2| / sqrt(...), the scale for tolerances."""
    vol = (np.asarray(mass, np.float32) / np.asarray(dens, np.float32)).astype(np.float64)
    vm = np.asarray(vm, np.float32).astype(np.float64)
    i, j, b2 = host_pairs(pos, h, world)
    term = vol[i] * vol[j] * (vm[j] - vm[i]) * (float(c_bspline) * b2)
    n = len(vol)
    q = np.bincount(i, weights=term, minlength=n)
    a = np.bincount(i, weights=np.abs(term), minlength=n)
    x = np.asarray(pos, np.float32).astype(np.float64)
    el = np.asarray(electrodes, np.float64).reshape(-1, 3)
    w = 1.0 / np.sqrt(((x[None, :, :] - el[:, None, :]) ** 2).sum(axis=2) + float(softening) ** 2)  # (E, n)
    return gain * (w @ q), abs(gain) * (w @ a)


def _b2(q):
    return -3.0 + 4.5 * q if q < 1 else (1.5 * (2.0 - q) if q < 2 else 0.0)


WORLD, H, CB = (4.0, 4.0, 4.0), 1.0, 0.5


def test_two_particles_by_hand():
    pos = np.array([[1.0, 1.0, 1.0], [1.5, 1.0, 1.0]], np.float32)  # r = h / 2: B2 = c (-3 + 4.5 / 2) = -0.75 c
    vm = np.array([0.0, 1.0], np.float32)
    mass = np.array([2.0, 1.0], np.float32)
    dens = np.array([1.0, 4.0], np.float32)  # vol = 2, 0.25
    e = np.array([[3.0, 1.0, 1.0]])
    phi, a = host_egm(pos, vm, mass, dens, e, 3.0, 1.0, H, WORLD, CB)
    b = CB * -0.75
    q0 = 2.0 * 0.25 * (1.0 - 0.0) * b  # vol_0 * vol_1 (Vm_1 - Vm_0) B2
    q1 = 0.25 * 2.0 * (0.0 - 1.0) * b
    ref = 3.0 * (q0 / np.sqrt(2.0**2 + 1.0) + q1 / np.sqrt(1.5**2 + 1.0))
    assert phi[0] == pytest.approx(ref, rel=1e-12) and ref != 0.0
    assert a[0] == pytest.approx(3.0 * (abs(q0) / np.sqrt(5.0) + abs(q1) / np.sqrt(3.25)), rel=1e-12)


def test_three_particles_by_hand():
    pos = np.array([[1.0, 1.0, 1.0], [1.5, 1.0, 1.0], [1.0, 2.5, 1.0]], np.float32)
    vm = np.array([-1.0, 2.0, 5.0], np.float32)
    ones = np.ones(3, np.float32)
    e = np.array([[1.0, 1.0, 3.0], [-2.0, 0.0, 0.0]])
    phi, _ = host_egm(pos, vm, ones, ones, e, 1.0, 0.5, H, WORLD, CB)
    r = {(0, 1): 0.5, (0, 2): 1.5, (1, 2): np.sqrt(0.25 + 2.25)}
    q = np.zeros(3)
    for (a, b), d in r.items():  # every pair is within 2h and in adjacent cells
        q[a] += (vm[b] - vm[a]) * CB * _b2(d / H)
        q[b] += (vm[a] - vm[b]) * CB * _b2(d / H)
    assert abs(q.sum()) < 1e-12  # the Laplacian conserves: no monopole
    for k in range(2):
        ref = sum(q[m] / np.sqrt(((pos[m] - e[k]) ** 2).sum() + 0.25) for m in range(3))
        assert phi[k] == pytest.approx(ref, rel=1e-6)


def test_pairs_follow_the_cell_stencil():
    # r = 1.02 h < 2h, but the cells (0 and 2 along x) are not neighbours: pass B never sees the pair
    pos = np.array([[0.99, 1.0, 1.0], [2.01, 1.0, 1.0]], np.float32)
    phi, a = host_egm(pos, [0.0, 1.0], [1, 1], [1, 1], [[0.0, 0.0, 0.0]], 1.0, 1.0, H, WORLD, CB)
    assert phi[0] == 0.0 and a[0] == 0.0
    pos[1, 0] = 1.99  # cells 0 and 1
    phi, _ = host_egm(pos, [0.0, 1.0], [1, 1], [1, 1], [[0.0, 0.0, 0.0]], 1.0, 1.0, H, WORLD, CB)
    assert phi[0] != 0.0


def _cloud(seed=3, n=400):
    rng = np.random.default_rng(seed)
    pos = (rng.random((n, 3)) * 2.5 + 0.7).astype(np.float32)
    vm = rng.normal(size=n).astype(np.float32)
    mass = (1 + 0.1 * rng.random(n)).astype(np.float32)
    dens = (1 + 0.1 * rng.random(n)).astype(np.float32)
    e = np.array([[0.0, 0.0, 0.0], [2.0, 2.0, 2.0], [9.0, -3.0, 1.0]])
    return pos, vm, mass, dens, e


def test_sign_flips_with_vm():
    pos, vm, mass, dens, e = _cloud()
    phi, a = host_egm(pos, vm, mass, dens, e, 2.0, 0.3, H, WORLD, CB)
    phi2, a2 = host_egm(pos, -vm, mass, dens, e, 2.0, 0.3, H, WORLD, CB)
    assert np.array_equal(phi2, -phi) and np.array_equal(a2, a) and (np.abs(phi) > 1e-6 * a).all()


def test_translation_invariance():
    pos, vm, mass, dens, e = _cloud()
    phi, a = host_egm(pos, vm, mass, dens, e, 1.0, 0.3, H, (8.0, 8.0, 8.0), CB)
    shift = np.array([3.0, 2.0, 1.0], np.float32)  # whole cells: the stencil stays the same
    phi2, a2 = host_egm(pos + shift, vm, mass, dens, e + shift, 1.0, 0.3, H, (8.0, 8.0, 8.0), CB)
    # (the shifted positions are rounded to float32 again: agreement to float32 precision of the terms)
    assert (np.abs(phi2 - phi) <= 1e-6 * a).all() and np.allclose(a2, a, rtol=1e-6) and (np.abs(phi) > 1e-4 * a).all()


def test_merge_electrograms():
    a = (5, np.array([[1.0, 2.0], [3.0, 4.0]]))
    b = (5, np.array([[0.5, -2.0], [1.0, 1.0]]))
    first, phi = slabs.merge_electrograms([a, b])
    assert first == 5 and np.array_equal(phi, a[1] + b[1]) and phi.dtype == np.float64
    first, phi = slabs.merge_electrograms([a])
    assert first == 5 and np.array_equal(phi, a[1])
    with pytest.raises(ValueError):
        slabs.merge_electrograms([a, (6, b[1])])  # different steps
    with pytest.raises(ValueError):
        slabs.merge_electrograms([a, (5, b[1][:1])])  # different row counts
    with pytest.raises(ValueError):
        slabs.merge_electrograms([a, (5, b[1][:, :1])])  # different electrodes
    with pytest.raises(ValueError):
        slabs.merge_electrograms([])
