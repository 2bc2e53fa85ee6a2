"""GPU: the on-device Vm recorder (activation / recovery maps and probe traces, include/sphsm_b200.h sphsm_record_*).

The reference of every case is built from the same run: Vm is downloaded (particles()) after every step, after every call that
changes state between steps, and the host rule (tests/test_record_cpu.host_crossings) is applied to the (pre, post) pairs.  The
device maps must equal it as integers and the probe traces must be bit-equal to the downloaded pos / Vm.

Protocol: the pacing of BASELINE configs[4] (bench.pacing_schedule) with period 60 and turnOffStim 20 steps after each stimulus,
the golden case's own stimulated set re-applied at every stimulus.  Stimulated particles rise by ~0.071 per step; turnOffStim zeroes
Vm and its stim = -10000 drives every particle down by ~2.37 per step, to ~-94.8 after 40 steps; the next stimulus lifts only the
stimulated particles back to ~-93.4 in 20 steps.  Thresholds vm_up = vm_down = -94.2 therefore give: an upstroke per later stimulus
of every stimulated particle (n_up = 2 in 150 steps), a real downstroke (made by a step, not by turnOffStim's reset) of every
particle in each off phase, and unstimulated particles that never activate.  (Values read off the CPU oracle of the same model.)"""
import numpy as np
import pytest

from bench import pacing_schedule
from sph_sm_monodomain_b200 import inputs, slabs
from tests.common import load_golden, setup_from_golden
from tests.test_record_cpu import host_crossings

pytestmark = pytest.mark.gpu

VM_UP = VM_DOWN = -94.2
PERIOD, OFF_AFTER, STEPS = 60, 20, 150
CASES = ["cfg2_5211_wave", "cube_4913", "lattice_24x10x12"]  # warp-per-particle + graph replay; thread-per-particle
MODES = ["graph", "no_graph", "strict", "diagnostics", "stage_timing", "profile_step"]


def make(name, mode):
    from sph_sm_monodomain_b200 import Sim

    g, kw = load_golden(name)
    s = Sim(diagnostics=(mode == "diagnostics"), strict=(mode == "strict"), **kw)
    setup_from_golden(s, g, False)
    if mode == "no_graph":
        p = s.get_params()
        p.reserved[4] = 1
        s._ck(s.lib.sphsm_set_params(s.h, p))
    if mode == "stage_timing":
        s.enable_stage_timing(True)
    return s, np.asarray(g["init.stim"], np.float32)


def probe_ids(n):
    return np.unique(np.linspace(0, n - 1, 24).astype(np.int32))


def run(s, stim, steps, mode="graph", start=0, download=True):
    """Pacing protocol over `steps` steps; returns the reference series and the post-step particles of every step."""
    series, posts = [], []
    pre = s.particles()["Vm"].copy() if download else None

    def one():
        nonlocal pre
        if mode == "profile_step":
            s.profile_step(1)
        else:
            s.Animation(1)
        if download:
            p = s.particles()
            series.append((s.total_time_steps, pre, p["Vm"].copy()))
            posts.append(p)
            pre = p["Vm"].copy()

    for act in pacing_schedule(start, steps, PERIOD, OFF_AFTER):
        if act[0] == "stim":
            s.set_masks(None, stim)
        elif act[0] == "off":
            s.turnOffStim()
        else:
            for _ in range(act[1]):
                one()
            continue
        if download:
            pre = s.particles()["Vm"].copy()  # pre = Vm after the call made between steps
    return series, posts


def check_trace(s, posts, ids, first_expected):
    first, xyzv, owned = s.probe_trace()
    assert first == first_expected and len(xyzv) == len(posts) and owned.all()
    ref = np.concatenate([np.stack([p["pos"][ids] for p in posts]), np.stack([p["Vm"][ids] for p in posts])[..., None]], axis=2)
    assert xyzv.tobytes() == ref.astype(np.float32).tobytes()


def check_maps(got, ref):
    for k in slabs.ACTIVATION_KEYS:
        assert got[k].dtype == np.int32 and np.array_equal(got[k], ref[k]), k


def not_vacuous(m):
    assert (m["n_up"] >= 2).any(), "no particle with two upstrokes"
    assert (m["last_down"] >= 0).any(), "no downstroke"
    assert (m["first_up"] < 0).any(), "every particle activated"


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", CASES)
def test_maps_and_traces_match_host_rule(name, mode):
    s, stim = make(name, mode)
    ids = probe_ids(s.n)
    s.record_start(VM_UP, VM_DOWN, probes=ids, trace_rows=STEPS)
    series, posts = run(s, stim, STEPS, mode)
    ref = host_crossings(series, VM_UP, VM_DOWN, s.n)
    got = s.activation()
    check_maps(got, ref)
    not_vacuous(got)
    check_trace(s, posts, ids, 1)


def test_recording_does_not_perturb_and_needs_no_downloads():
    name = "cube_4913"
    finals, maps, traces = [], [], []
    for variant in ("off", "on", "on_no_download", "started_then_stopped"):
        s, stim = make(name, "graph")
        ids = probe_ids(s.n)
        if variant != "off":
            s.record_start(VM_UP, VM_DOWN, probes=ids, trace_rows=STEPS)
        if variant == "started_then_stopped":
            run(s, stim, 70, download=False)
            s.record_stop()
            run(s, stim, STEPS - 70, start=70, download=False)
        else:
            run(s, stim, STEPS, download=(variant == "on"))
        if variant.startswith("on"):
            maps.append(s.activation())
            traces.append(s.probe_trace())
        p = s.particles()
        finals.append((p["pos"].tobytes(), p["Vm"].tobytes()))
    assert finals[1] == finals[0] and finals[2] == finals[0] and finals[3] == finals[0]
    check_maps(maps[1], maps[0])  # the per-step downloads neither cause nor hide a crossing
    assert traces[0][0] == traces[1][0] and traces[0][1].tobytes() == traces[1][1].tobytes() and (traces[1][2] == traces[0][2]).all()


def test_recording_off_adds_no_launches():
    def per_step(s):
        s.Animation(5)  # steady state (graphs captured)
        s.reset_launch_count()
        s.Animation(10)
        return s.launch_count()

    for name in ("cfg2_5211_wave", "lattice_24x10x12"):
        never, _ = make(name, "graph")
        was, _ = make(name, "graph")
        was.record_start(VM_UP, probes=[0, 1], trace_rows=4)
        was.Animation(3)
        was.record_stop()
        assert per_step(never) == per_step(was)
        on, _ = make(name, "graph")
        on.record_start(VM_UP)
        assert per_step(on) == per_step(never) + 10  # one k_record launch per step while on


def test_start_stop_restart_after_graph_capture():
    s, stim = make("cfg2_5211_wave", "graph")
    ids = probe_ids(s.n)
    run(s, stim, 30, download=False)  # graphs of the unrecorded step are captured
    s.record_start(VM_UP, VM_DOWN, probes=ids, trace_rows=200)
    series, posts = run(s, stim, 60, start=30)
    check_maps(s.activation(), host_crossings(series, VM_UP, VM_DOWN, s.n))
    check_trace(s, posts, ids, 31)
    s.record_stop()
    with pytest.raises(Exception):
        s.activation()
    run(s, stim, 20, start=90, download=False)
    s.record_start(VM_UP, VM_DOWN, probes=ids, trace_rows=200)
    series, posts = run(s, stim, 70, start=110)
    got = s.activation()
    check_maps(got, host_crossings(series, VM_UP, VM_DOWN, s.n))
    check_trace(s, posts, ids, 111)
    assert (got["n_up"] >= 1).any() and (got["last_down"] >= 0).any()


def test_ring_buffer_keeps_the_last_rows_in_order():
    s, stim = make("lattice_24x10x12", "graph")
    ids = probe_ids(s.n)
    s.record_start(VM_UP, VM_DOWN, probes=ids, trace_rows=37)
    series, posts = run(s, stim, 100)
    check_trace(s, posts[-37:], ids, 64)
    s.record_reset()  # data cleared, configuration kept
    assert (s.activation()["first_up"] == -1).all() and len(s.probe_trace()[1]) == 0
    series, posts = run(s, stim, 10, start=100)
    check_trace(s, posts, ids, 101)
    check_maps(s.activation(), host_crossings(series, VM_UP, VM_DOWN, s.n))


def test_snapshot_continues_numbering(tmp_path):
    s, stim = make("cube_4913", "graph")
    run(s, stim, 40, download=False)
    path = tmp_path / "k40.snap"
    s.save_state(path)
    t, _ = make("cube_4913", "graph")
    ids = probe_ids(t.n)
    t.record_start(VM_UP, VM_DOWN, probes=ids, trace_rows=100)
    t.Animation(3)
    t.load_state(path)  # the recorded data of the replaced set is cleared; numbering continues at 41
    assert t.total_time_steps == 40
    series, posts = run(t, stim, 50, start=40)
    assert series[0][0] == 41
    got = t.activation()
    check_maps(got, host_crossings(series, VM_UP, VM_DOWN, t.n))
    check_trace(t, posts, ids, 41)
    assert (got["last_down"] >= 41).any()


def test_single_stages_record_nothing():
    s, stim = make("lattice_24x10x12", "graph")
    s.record_start(0.01, 0.01, probes=[3], trace_rows=4)  # (stage 7 alone lifts the stimulated particles' Vm through 0.01)
    for st in range(1, 8):
        s.stage(st)
    assert s.total_time_steps == 0
    assert (s.activation()["n_up"] == 0).all() and len(s.probe_trace()[1]) == 0
    s.Animation(1)
    first, x, o = s.probe_trace()
    assert first == 1 and len(x) == 1 and o.all()


def test_invalid_arguments():
    from sph_sm_monodomain_b200 import SphsmError

    s, _ = make("lattice_24x10x12", "graph")
    n = s.n
    with pytest.raises(SphsmError):
        s.activation()  # recording is off
    with pytest.raises(SphsmError):
        s.probe_trace()
    with pytest.raises(SphsmError):
        s.record_reset()
    bad = [dict(vm_up=1.0, vm_down=2.0), dict(vm_up=float("nan")), dict(vm_up=1.0, vm_down=float("-inf")),
           dict(vm_up=1.0, probes=[1, 1], trace_rows=4), dict(vm_up=1.0, probes=[n], trace_rows=4), dict(vm_up=1.0, probes=[-1], trace_rows=4),
           dict(vm_up=1.0, probes=[0], trace_rows=0), dict(vm_up=1.0, probes=np.arange(70000) % n, trace_rows=1),
           dict(vm_up=1.0, probes=np.arange(2000), trace_rows=1 << 14)]
    for kw in bad:
        with pytest.raises(SphsmError):
            s.record_start(**kw)
    with pytest.raises(SphsmError):
        s.activation()  # a rejected start leaves recording off
    s.record_start(1.0, probes=[0, n - 1], trace_rows=2)
    with pytest.raises(SphsmError):
        s.activation(n=s.get_params().capacity + 1)
    s.record_stop()
    s.record_stop()  # (idempotent)


# ---- slab mode: virtual ranks ---------------------------------------------------------------------------------------------------
def _owned_download(sims, n):
    """Global Vm / pos assembled from every rank's download_aos (owned particles only) and the owner of every particle."""
    from sph_sm_monodomain_b200 import PARTICLE_DTYPE
    import ctypes as C

    out = np.zeros(n, PARTICLE_DTYPE)
    owner = np.full(n, -1, np.int32)
    for r, s in enumerate(sims):
        buf = np.zeros(n, PARTICLE_DTYPE)
        s._ck(s.lib.sphsm_download_aos(s.h, buf.ctypes.data_as(C.c_void_p), n, PARTICLE_DTYPE.itemsize))
        ids, _ = s.download_owned()
        assert (owner[ids] == -1).all()
        owner[ids] = r
        out[ids] = buf[ids]
    assert (owner >= 0).all()
    return out, owner


@pytest.mark.parametrize("nranks", [3, 4])
def test_virtual_ranks_merge_exactly(nranks):
    from sph_sm_monodomain_b200 import LocalGroup, Sim

    dims = (40, 9, 8)
    pos, world = inputs.lattice(*dims, jitter=0.05)
    fixed, stim = inputs.lattice_masks(pos, dims[0], 4)
    stimv = np.where(stim, np.float32(300), np.float32(0)).astype(np.float32)
    n = len(pos)
    parts = slabs.partition_planes(slabs.plane_histogram(pos, 0, slabs.num_planes(world, 0)), nranks)
    sims = []
    for _ in range(nranks):
        s = Sim(capacity=n, world=world, diagnostics=False, slab_axis=0)
        s.Init_Fluid(pos)
        s.set_masks(fixed.astype(np.uint8), stimv)
        sims.append(s)
    grp = LocalGroup(sims)
    for s, (lo, hi) in zip(sims, parts):
        s.set_slab(lo, hi)
    ids = np.unique(np.linspace(0, n - 1, 40).astype(np.int32))
    for s in sims:
        s.record_start(VM_UP, VM_DOWN, probes=ids, trace_rows=STEPS)
    series, posts, owners = [], [], []
    pre = _owned_download(sims, n)[0]["Vm"].copy()
    for act in pacing_schedule(0, STEPS, PERIOD, OFF_AFTER):
        if act[0] in ("stim", "off"):
            for s in sims:  # collective: every rank alike
                if act[0] == "stim":
                    s.set_masks(None, stimv)
                else:
                    s.turnOffStim()
            pre = _owned_download(sims, n)[0]["Vm"].copy()
            continue
        for _ in range(act[1]):
            grp.step(1)
            p, owner = _owned_download(sims, n)
            series.append((sims[0].total_time_steps, pre, p["Vm"].copy()))
            posts.append(p)
            owners.append(owner[ids])
            pre = p["Vm"].copy()
    ref = host_crossings(series, VM_UP, VM_DOWN, n)
    got = grp.activation(n)
    check_maps(got, ref)  # n_up summed over ranks == reference: each crossing counted once
    not_vacuous(got)
    parts_tr = [s.probe_trace() for s in sims]
    for r, (f, x, o) in enumerate(parts_tr):  # each rank owns exactly the probes it integrated
        assert f == 1 and np.array_equal(o, np.stack(owners) == r)
    first, xyzv, owned = grp.probe_trace()
    assert first == 1 and owned.all()
    refx = np.concatenate([np.stack([p["pos"][ids] for p in posts]), np.stack([p["Vm"][ids] for p in posts])[..., None]], axis=2)
    assert xyzv.tobytes() == refx.astype(np.float32).tobytes()


# ---- NCCL slab path (2+ GPUs) ---------------------------------------------------------------------------------------------------
def test_nccl_ranks_record_and_merge():
    import json
    import os
    import subprocess
    import sys

    import torch

    ngpu = torch.cuda.device_count() if torch.cuda.is_available() else 0
    if ngpu < 2:
        pytest.skip("needs at least 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    nproc = 2 if ngpu < 4 else 4
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(root, "tools", "record_mg.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert r.returncode == 0 and lines, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(lines[-1])
    assert res["record_mg"] == "ok", res
