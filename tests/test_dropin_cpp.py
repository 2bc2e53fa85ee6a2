"""The C++ drop-in class (include/dropin/SPH_SM_monodomain.h + libsphsm_dropin.so) behind the reference's main.cpp.

CPU part: the headers keep the reference's source-level API (the UNMODIFIED reference main.cpp compiles against them and
every SPH_SM_monodomain:: symbol it references is exported by libsphsm_dropin.so; an in-repo translation unit that makes the
same calls is always checked, main.cpp itself as well where $SPHSM_REFERENCE_DIR names a checkout of the reference), and the
Particle layout is the reference's 132 bytes.
GPU part: the headless replay of main.cpp's run protocol (sphsm_headless) against the oracle driven the same way.
"""
import os
import subprocess
import tempfile

import numpy as np
import pytest

from sph_sm_monodomain_b200 import build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INC = os.path.join(ROOT, "include", "dropin")
STUBS = os.path.join(ROOT, "tests", "stubs")
REF_MAIN = os.path.join(os.environ["SPHSM_REFERENCE_DIR"], "main.cpp") if os.environ.get("SPHSM_REFERENCE_DIR") else None

# every call main.cpp (and the survey's boundary list, SURVEY.md §8b) makes on the class, as a stand-alone unit
API_USER = r"""
#include <SPH_SM_monodomain.h>
#include <iostream>
int use_api() {
    SPH_SM_monodomain *sph = new SPH_SM_monodomain();
    std::vector<m3Vector> pos; pos.push_back(m3Vector(0.5f, 0.5f, 0.5f));
    sph->Init_Fluid(pos); sph->Init_Particle(m3Vector(0.6f, 0.5f, 0.5f), m3Vector(0.f, 0.f, 0.f));
    sph->turnOnStim_Cube(pos); sph->turnOnStim_Mesh(pos); sph->set_stim(m3Vector(0.5f, 0.5f, 0.5f), 0.01f, 300.0f); sph->turnOffStim();
    sph->Animation(); sph->compute_SPH_SM_monodomain();
    sph->Find_neighbors(); sph->calculate_corrected_velocity(); sph->apply_external_forces(); sph->projectPositions();
    sph->calculate_intermediate_velocity(); sph->Compute_Density_SingPressure(); sph->calculate_cell_model(); sph->Compute_Force();
    sph->Update_Properties();
    Particle *p = sph->Get_Paticles(); Cell *c = sph->Get_Cells();
    float s = p[0].pos.x + p[0].getDisplacement() + p[0].Vm + (float)c[0].contained_particles.size();
    s += sph->Get_Particle_Number() + sph->Get_World_Size().x + sph->Get_stand_dens() + sph->max_voltage + sph->voltage_constant + sph->max_pressure;
    s += sph->Poly6(0.f) + sph->Spiky(0.01f) + sph->Visco(0.01f) + sph->B_spline(0.01f) + sph->B_spline_1(0.01f) + sph->B_spline_2(0.01f);
    s += sph->Calculate_Cell_Hash(sph->Calculate_Cell_Position(p[0].pos)) + sph->pow2roundup(5);
    bool q = sph->flip_quadratic(), v = sph->flip_volume(); sph->add_viscosity(1.0f);
    duration_d d = sph->d_find_neighbors + sph->d_compute_Force; tpoint t = sph->t_start_cell_model; (void)t;
    sph->print_report(1.0, d.count()); int steps = sph->total_time_steps;
    delete sph;
    return (int)s + q + v + steps;
}
"""


def run(cmd, **kw):
    return subprocess.run(cmd, capture_output=True, text=True, **kw)


def test_api_user_compiles_against_dropin_headers(tmp_path):
    src = tmp_path / "api_user.cpp"
    src.write_text(API_USER)
    r = run(["g++", "-std=c++11", "-Wall", "-fsyntax-only", "-I", INC, str(src)])
    assert r.returncode == 0, r.stderr


def test_particle_layout_is_the_reference_layout(tmp_path):
    src = tmp_path / "layout.cpp"
    src.write_text(r"""
#include <Particle.h>
#include <cstddef>
#include <cstdio>
int main() { printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(Particle), offsetof(Particle, vel), offsetof(Particle, mass),
    offsetof(Particle, mOriginalPos), offsetof(Particle, mFixed), offsetof(Particle, dens), offsetof(Particle, stim), offsetof(Particle, w)); }
""")
    exe = tmp_path / "layout"
    r = run(["g++", "-std=c++11", "-Wno-invalid-offsetof", "-I", INC, str(src), "-o", str(exe)])
    assert r.returncode == 0, r.stderr
    assert run([str(exe)]).stdout.split() == ["132", "12", "72", "76", "100", "104", "124", "128"]  # Particle.h:7-35


def _class_symbols_needed(obj):
    out = run(["nm", "-C", "--undefined-only", obj]).stdout
    return sorted({ln.split(None, 1)[1].strip() for ln in out.splitlines() if "SPH_SM_monodomain::" in ln})


def _exported(lib):
    out = run(["nm", "-C", "-D", "--defined-only", lib]).stdout
    return {ln.split(None, 2)[2].strip() for ln in out.splitlines() if len(ln.split(None, 2)) == 3}


def test_dropin_library_exports_what_main_cpp_links_against(tmp_path):
    build.build()
    lib = build.build_dropin()
    exported = _exported(lib)
    units = []
    user = tmp_path / "api_user.cpp"
    user.write_text(API_USER)
    units.append((str(user), []))
    if REF_MAIN and os.path.exists(REF_MAIN):  # the genuine, unmodified viewer source (GL calls stubbed as declarations)
        units.append((REF_MAIN, ["-I", STUBS]))
    for k, (src, extra) in enumerate(units):
        obj = str(tmp_path / f"unit{k}.o")
        r = run(["g++", "-std=c++11", "-c", "-I", INC] + extra + [src, "-o", obj])
        assert r.returncode == 0, r.stderr
        needed = _class_symbols_needed(obj)
        assert needed, "no class symbols referenced?"
        missing = [s for s in needed if s not in exported]
        assert not missing, missing


# ------------------------------------------------------------------------------------------------------------------
def _headless(args, cwd, env=None):
    build.build()
    build.build_dropin()
    r = run([build.HEADLESS] + args, cwd=cwd, timeout=600, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    return r


def _load_dump(path):
    from sph_sm_monodomain_b200.sim import PARTICLE_DTYPE

    return np.fromfile(path, dtype=PARTICLE_DTYPE)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["staged", "fused", "strict"])
def test_headless_cube_protocol_matches_oracle(mode):
    """main.cpp's protocol on init_cube: 10 steps, stimulation switched off when half are left, Get_Paticles() each frame.
    SPHSM_STRICT=1 (reference-order arithmetic): every field of every particle is BIT-IDENTICAL to the oracle after
    the whole run.  Fast path: the pressure sums cancel to ~1e-4 of their terms, so summation-order rounding shows up as
    ~1e-2 velocity noise per step in the reference itself; trajectory bounds as in test_gpu_parity.py (pos / goal 5e-4
    of the field scale, density 5e-3, Vm 1e-4 after 10 steps)."""
    from oracle import CpuSim
    from sph_sm_monodomain_b200 import inputs
    from tests.common import bits_equal, rel_err

    steps = 10
    env = dict(os.environ, SPHSM_STRICT="1" if mode == "strict" else "0")
    with tempfile.TemporaryDirectory() as d:
        dump = os.path.join(d, "out.bin")
        r = _headless(["--cube", "--steps", str(steps), "--dump", dump] + (["--staged"] if mode == "staged" else []), d, env=env)
        got = _load_dump(dump)
    report = [ln for ln in r.stdout.splitlines() if ln.count(";") == 22]
    assert len(report) == 1, r.stdout  # the 23-field report line, cpp:785-792
    fields = report[0].split(";")
    assert int(fields[2]) == steps and float(fields[10]) == 0.5 and float(fields[13]) == 100.0
    if mode == "staged":
        assert all(float(x) > 0 for x in fields[3:10])  # per-stage device seconds per step
    elif mode == "fused":  # the default: sampled kernel-group timers in the slots of the dominating stages
        assert all(float(fields[k]) > 0 for k in (3, 4, 5, 8)) and all(float(fields[k]) == 0 for k in (6, 7, 9))
    assert "Turning stimulation off" in r.stdout and "Number of Paticles : 4913" in r.stdout

    pos = inputs.init_cube_positions()
    ora = CpuSim("port")
    ora.Init_Fluid(pos)
    ora.turnOnStim_Cube(pos)
    for left in range(steps, 0, -1):
        if left == steps // 2:
            ora.turnOffStim()
        ora.Animation(1)
    ref = ora.particles()
    assert len(got) == len(ref) == 4913
    assert np.array_equal(got["fixed"], ref["fixed"]) and np.array_equal(got["stim"], ref["stim"])
    if mode == "strict":
        bad = [f for f in ref.dtype.names if f != "_pad" and not bits_equal(got[f], ref[f])]
        assert bad == [], bad
    else:
        for f, tol in (("pos", 5e-4), ("dens", 5e-3), ("Vm", 1e-4), ("goal", 5e-4)):
            assert rel_err(got[f], ref[f]) <= tol, (f, rel_err(got[f], ref[f]))


@pytest.mark.gpu
def test_headless_mesh_from_raw_positions_and_host_writes():
    """init_mesh on cfg1's point set fed as raw xyz; 10 steps; every field of every particle present and finite."""
    from tests.common import load_golden

    g, _ = load_golden("cfg1_4944")
    with tempfile.TemporaryDirectory() as d:
        xyz = os.path.join(d, "p.xyz")
        g["positions"].astype("<f4").tofile(xyz)
        dump = os.path.join(d, "out.bin")
        _headless(["--xyz", xyz, "--steps", "10", "--no-stim-off", "--dump", dump], d)
        got = _load_dump(dump)
    assert len(got) == 4944 and got["fixed"].sum() == 1675 and (got["stim"] == 300.0).all()
    for f in ("pos", "vel", "acc", "dens", "pres", "Vm", "Inter_Vm", "goal", "corrected_vel", "inter_vel"):
        assert np.isfinite(got[f]).all(), f
    assert np.array_equal(got["orig"], g["positions"])
