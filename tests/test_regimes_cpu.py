"""CPU: the cases of tests/test_gpu_regimes.py reach the branches they are named for — on the restatement and in numpy —
so that a GPU test that passes on them has compared something: the mirror trips the flip guard, the compressions the volume
clamp, the sheets the invert3 failure path and its near-singular neighbour, and the sort worlds have the padded cell counts
and radix pass counts that select the path each case names."""
import numpy as np
import pytest

from oracle import CpuSim
from tests import regimes as R


def solve(name, **kw):
    st = R.body_state(name)
    s, cm, ocm, x = R.solve_state(st, **kw)
    return st, s, cm, ocm, x


def det(m):
    return float(np.linalg.det(np.asarray(m, np.float64).reshape(3, 3)))


@pytest.mark.parametrize("name", ["cube_mirror_x", "lattice_mirror_x"])
def test_mirror_reaches_the_flip_guard(name):
    st, s, cm, ocm, x = solve(name, dbl=False)
    assert det(R.restatement_apq(st, cm, ocm)) < 0.0
    assert det(x[:9]) < 0.0  # the guard keeps the mirror: T is not a rotation


@pytest.mark.parametrize("name,factor", [("cube_compress_0.5", 0.5), ("cube_compress_0.3", 0.3), ("lattice_compress_0.3", 0.3)])
def test_compressions_reach_the_volume_clamp(name, factor):
    st, s, cm, ocm, x = solve(name, dbl=False)
    a = R.restatement_apq(st, cm, ocm).astype(np.float64) @ np.linalg.inv(R.restatement_aqq(st, ocm).astype(np.float64))
    assert 1.0 / np.sqrt(abs(np.linalg.det(a))) > 2.0
    beta = float(s.constants()["beta"])
    clamped = (1.0 - beta) + beta * 2.0 * factor  # T = (1 - beta) R + beta * 2 A with R = I, A = factor * I
    assert np.allclose(x[:9].reshape(3, 3), clamped * np.eye(3), atol=1e-4)
    _, _, _, _, x_off = solve(name, dbl=False, volume=False)
    assert np.allclose(x_off[:9].reshape(3, 3), ((1.0 - beta) + beta * factor) * np.eye(3), atol=1e-4)


def test_sheets_reach_the_invert3_failure_path_and_its_neighbour():
    # float restatement (the reference's sums): the z = 0.5 sheet's centre is exact, Aqq's z row is zero and invert3 fails;
    # at z = 0.45 the centre is an ulp off, Aqq is nearly singular and is inverted
    st, s, cm, ocm, x = solve("sheet_z0.5", dbl=False)
    assert ocm[2] == np.float32(0.5)
    aqq = R.restatement_aqq(st, ocm)
    assert not aqq[2].any() and not s.invert3(aqq)[0]
    st, s, cm, ocm, x = solve("sheet_z0.45", dbl=False)
    assert ocm[2] != np.float32(0.45)
    aqq = R.restatement_aqq(st, ocm)
    ok, _ = s.invert3(aqq)
    assert ok and np.linalg.cond(aqq.astype(np.float64)) > 1e6
    # with double sums (the fast path's order of record) both centres are exact: both sheets take the failure path
    for name, z in (("sheet_z0.5", 0.5), ("sheet_z0.45", 0.45)):
        st, s, cm, ocm, x = solve(name, dbl=True)
        assert ocm[2] == np.float32(z) and not s.invert3(R.restatement_aqq(st, ocm))[0], name


def test_degenerate_bodies_are_degenerate():
    for name, (_, _, _, degenerate) in R.BODIES.items():
        st, s, cm, ocm, x = solve(name)
        cond = np.linalg.cond(R.restatement_aqq(st, ocm).astype(np.float64))
        assert (cond > 1e6) == degenerate, (name, cond)


@pytest.mark.parametrize("name", list(R.RADIX_CASES))
def test_radix_worlds_select_the_radix_path(name):
    world, pos, mode, passes = R.radix_case(name)
    g = R.grid_dims(world)
    assert CpuSim("port", capacity=len(pos), world=world).num_cells == g[0] * g[1] * g[2]
    assert R.sort_passes(world) == passes
    lo, hi = 1 << (8 * (passes - 1)), 1 << (8 * passes)
    assert lo <= R.padded_cells(world) + 1 <= hi
    # forced cases would take the counting sort on their own; automatic ones are a small body in a large world
    assert R.counting_sort_auto(world, len(pos)) == (mode == 1)
    assert pos.min() >= 0 and (pos < np.float32(world)).all()


@pytest.mark.parametrize("name", list(R.TILE_CASES))
def test_tile_worlds_have_the_intended_cell_tables(name):
    world, pos, m = R.tile_case(name)
    g = R.grid_dims(world)
    assert g == R.TILE_CASES[name][0]
    assert R.padded_cells(world) + 1 == m
    assert R.counting_sort_auto(world, len(pos))
    assert CpuSim("port", capacity=len(pos), world=world).num_cells == g[0] * g[1] * g[2]
    assert pos.min() > 0 and (pos < np.float32(world)).all() and len(pos) > 100


def test_boundary_sets():
    for n in R.BOUNDARY_COUNTS:
        pos = R.boundary_set(n)
        assert len(pos) == n == len(np.unique(pos, axis=0))
        assert pos.min() > 0 and pos.max() < 1.5
