"""GPU: extracellular electrograms at virtual electrodes (include/sphsm_b200.h sphsm_egm_*).

The reference of every case is built from the same run: the particles are downloaded before every step (after any call made
between steps) and after it, and the host formula (tests/test_egm_cpu.host_egm) is applied to the pre-step positions and Vm and
the step's mass and density.  Every device row must agree with it within 1e-5 * A_e, A_e being the sum of the absolute values of
the elementary terms, and some rows must exceed that bound a hundredfold (the pacing protocol of tests/test_gpu_record.py makes
Vm gradients; on the sets as main.cpp runs them the Laplacian vanishes and so does the electrogram)."""
import numpy as np
import pytest

from bench import pacing_schedule
from sph_sm_monodomain_b200 import inputs, slabs
from tests.common import rel_err
from tests.test_egm_cpu import host_egm, host_pairs
from tests.test_gpu_record import CASES, MODES, OFF_AFTER, PERIOD, STEPS, VM_DOWN, VM_UP, make, probe_ids

pytestmark = pytest.mark.gpu

TOL, VACUOUS = 1e-5, 100.0


def electrodes(pos, h):
    """8 electrodes: six outside the body's box, one at its centre (inside the tissue: softening h keeps it finite), one far away."""
    lo, hi = pos.min(axis=0), pos.max(axis=0)
    c, ext = (lo + hi) / 2, hi - lo
    out = [c + s * np.eye(3)[a] * (0.6 * ext[a] + h) for a in range(3) for s in (-1, 1)]
    return np.array(out + [c, c + 20 * ext.max() * np.array([1.0, 0.5, 0.25])], np.float32)


def geometry(s):
    p = s.get_params()
    return float(p.kernel_h), tuple(float(w) for w in p.world), float(p.bspline_constant)


def run(s, stim, steps, mode="graph", start=0, download=True):
    """Pacing protocol over `steps` steps; returns (step, pre particles, post particles) of every step when downloading."""
    recs = []
    pre = s.particles() if download else None

    def one():
        nonlocal pre
        if mode == "profile_step":
            s.profile_step(1)
        else:
            s.Animation(1)
        if download:
            post = s.particles()
            recs.append((s.total_time_steps, pre, post))
            pre = post

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
            pre = s.particles()
    return recs


def host_rows(recs, el, gain, eps, geo):
    h, world, cb = geo
    out = [host_egm(pre["pos"], pre["Vm"], post["mass"], post["dens"], el, gain, eps, h, world, cb) for _, pre, post in recs]
    return np.stack([r for r, _ in out]), np.stack([a for _, a in out])


def check_rows(phi, ref, scale, tol=TOL):
    assert phi.shape == ref.shape
    err = np.abs(phi - ref)
    assert (err <= tol * scale).all(), float((err / scale).max())
    assert (np.abs(phi) > VACUOUS * TOL * scale).any(), "every row is within the tolerance of zero"


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", CASES)
def test_rows_match_host_formula(name, mode):
    s, stim = make(name, mode)
    geo = geometry(s)
    el = electrodes(s.particles()["pos"], geo[0])
    if mode == "graph":  # the host pair rule is pass B's candidate rule
        p = s.particles()
        s.stage(1)
        q = np.arange(0, s.n, 7, dtype=np.int32)
        got = s.neighbor_sets(q, kind=3)
        i, j, _ = host_pairs(p["pos"], *geo[:2])
        for k, qi in enumerate(q):
            assert np.array_equal(np.sort(got[k]), np.sort(j[i == qi])), qi
    s.egm_start(el, gain=2.5, rows=STEPS)
    recs = run(s, stim, STEPS, mode)
    first, phi = s.electrogram()
    assert first == 1 and len(phi) == STEPS and [r[0] for r in recs] == list(range(1, STEPS + 1))
    ref, scale = host_rows(recs, el, 2.5, geo[0], geo)
    check_rows(phi, ref, scale)


def test_large_lattice_many_blocks():
    from sph_sm_monodomain_b200 import Sim

    dims = (128, 96, 86)  # 1,056,768 particles
    pos, world = inputs.lattice(*dims, jitter=0.05)
    fixed, stim = inputs.lattice_masks(pos, dims[0], 4)
    s = Sim(capacity=len(pos), world=world, diagnostics=False)
    s.Init_Fluid(pos)
    s.set_masks(fixed.astype(np.uint8), np.where(stim, np.float32(300), np.float32(0)).astype(np.float32))
    s.Animation(4)  # stimulated particles rise: a Vm front at the end of the lattice
    geo = geometry(s)
    rng = np.random.default_rng(5)
    lo, hi = pos.min(axis=0), pos.max(axis=0)
    el = (lo + (rng.random((16, 3)) * 1.6 - 0.3) * (hi - lo)).astype(np.float32)
    s.egm_start(el, rows=8)
    recs = []
    for _ in range(3):
        pre = s.particles()
        s.Animation(1)
        recs.append((s.total_time_steps, pre, s.particles()))
    first, phi = s.electrogram()
    assert first == 5 and len(phi) == 3
    ref, scale = host_rows(recs, el, 1.0, geo[0], geo)
    check_rows(phi, ref, scale)


def test_deterministic_and_non_interfering():
    name = "cube_4913"
    finals, rows = {}, {}
    for variant in ("off", "on", "on_again", "no_graph", "started_then_stopped", "recorder", "recorder+egm"):
        s, stim = make(name, "no_graph" if variant == "no_graph" else "graph")
        el = electrodes(s.particles()["pos"], geometry(s)[0])
        if variant not in ("off", "recorder"):
            s.egm_start(el, rows=STEPS)
        if variant.startswith("recorder"):
            s.record_start(VM_UP, VM_DOWN, probes=probe_ids(s.n), trace_rows=STEPS)
        if variant == "started_then_stopped":
            run(s, stim, 70, download=False)
            s.egm_stop()
            run(s, stim, STEPS - 70, start=70, download=False)
        else:
            run(s, stim, STEPS, download=False)
        if variant not in ("off", "recorder", "started_then_stopped"):
            rows[variant] = s.electrogram()
        if variant.startswith("recorder"):
            rows[variant + ".maps"] = s.activation()
            rows[variant + ".trace"] = s.probe_trace()
        p = s.particles()
        finals[variant] = (p["pos"].tobytes(), p["Vm"].tobytes(), p["dens"].tobytes())
    assert all(f == finals["off"] for f in finals.values())
    for v in ("on_again", "no_graph", "recorder+egm"):  # bit for bit: the same run twice, graph replay or eager steps
        assert rows[v][0] == rows["on"][0] == 1 and rows[v][1].tobytes() == rows["on"][1].tobytes(), v
    for k in slabs.ACTIVATION_KEYS:
        assert np.array_equal(rows["recorder.maps"][k], rows["recorder+egm.maps"][k]), k
    a, b = rows["recorder.trace"], rows["recorder+egm.trace"]
    assert a[0] == b[0] == rows["recorder+egm"][0] and a[1].tobytes() == b[1].tobytes() and np.array_equal(a[2], b[2])
    assert len(a[1]) == len(rows["recorder+egm"][1])  # both number the same steps


def test_launches_off_and_on():
    def per_step(s):
        s.Animation(5)  # steady state (graphs captured)
        s.reset_launch_count()
        s.Animation(10)
        return s.launch_count()

    for name in ("cfg2_5211_wave", "lattice_24x10x12"):
        never, _ = make(name, "graph")
        el = electrodes(never.particles()["pos"], geometry(never)[0])
        was, _ = make(name, "graph")
        was.egm_start(el)
        was.Animation(3)
        was.egm_stop()
        base = per_step(never)
        assert per_step(was) == base
        on, _ = make(name, "graph")
        on.egm_start(el)
        assert per_step(on) == base + 10  # one k_egm launch per step
        both, _ = make(name, "graph")
        both.egm_start(el)
        both.record_start(VM_UP)
        assert per_step(both) == base + 20


def test_start_stop_restart_after_graph_capture():
    s, stim = make("cfg2_5211_wave", "graph")
    geo = geometry(s)
    el = electrodes(s.particles()["pos"], geo[0])
    run(s, stim, 30, download=False)  # graphs of the plain step are captured
    s.egm_start(el, rows=200)
    recs = run(s, stim, 60, start=30)
    first, phi = s.electrogram()
    assert first == 31
    check_rows(phi, *host_rows(recs, el, 1.0, geo[0], geo))
    s.egm_stop()
    with pytest.raises(Exception):
        s.electrogram()
    run(s, stim, 20, start=90, download=False)
    s.egm_start(el[:3], gain=-1.0, softening=0.5 * geo[0], rows=200)
    recs = run(s, stim, 70, start=110)
    first, phi = s.electrogram()
    assert first == 111
    check_rows(phi, *host_rows(recs, el[:3], -1.0, 0.5 * geo[0], geo))


def test_ring_keeps_the_last_rows_in_order():
    s, stim = make("lattice_24x10x12", "graph")
    geo = geometry(s)
    el = electrodes(s.particles()["pos"], geo[0])
    s.egm_start(el, rows=37)
    recs = run(s, stim, 100)
    ref, scale = host_rows(recs, el, 1.0, geo[0], geo)
    first, phi = s.electrogram()
    assert first == 64 and len(phi) == 37
    check_rows(phi, ref[-37:], scale[-37:])
    s.egm_reset()  # rows cleared, configuration kept
    assert len(s.electrogram()[1]) == 0
    recs = run(s, stim, 10, start=100)
    first, phi = s.electrogram()
    assert first == 101 and len(phi) == 10
    ref, scale = host_rows(recs, el, 1.0, geo[0], geo)
    assert (np.abs(phi - ref) <= TOL * scale).all()


def test_snapshot_continues_numbering(tmp_path):
    s, stim = make("cube_4913", "graph")
    run(s, stim, 40, download=False)
    path = tmp_path / "k40.snap"
    s.save_state(path)
    t, _ = make("cube_4913", "graph")
    geo = geometry(t)
    el = electrodes(t.particles()["pos"], geo[0])
    t.egm_start(el, rows=100)
    t.record_start(VM_UP, VM_DOWN, probes=probe_ids(t.n), trace_rows=100)
    t.Animation(3)
    t.load_state(path)  # the rows of the replaced set are cleared; numbering continues at 41
    assert t.total_time_steps == 40 and len(t.electrogram()[1]) == 0
    recs = run(t, stim, 50, start=40)
    first, phi = t.electrogram()
    assert first == 41 and len(phi) == 50 and t.probe_trace()[0] == 41
    check_rows(phi, *host_rows(recs, el, 1.0, geo[0], geo))


def test_single_stages_produce_nothing():
    s, _ = make("lattice_24x10x12", "graph")
    s.egm_start(electrodes(s.particles()["pos"], geometry(s)[0]), rows=4)
    for st in range(1, 8):
        s.stage(st)
    assert s.total_time_steps == 0 and len(s.electrogram()[1]) == 0
    s.Animation(1)
    first, phi = s.electrogram()
    assert first == 1 and len(phi) == 1


def test_invalid_arguments():
    from sph_sm_monodomain_b200 import SphsmError

    s, _ = make("lattice_24x10x12", "graph")
    with pytest.raises(SphsmError):
        s.electrogram()  # off
    with pytest.raises(SphsmError):
        s.egm_reset()
    ok = np.zeros((2, 3), np.float32)
    bad = [dict(electrodes=np.zeros((0, 3), np.float32)), dict(electrodes=np.zeros((257, 3), np.float32)),
           dict(electrodes=np.array([[0, np.nan, 0]], np.float32)), dict(electrodes=np.array([[np.inf, 0, 0]], np.float32)),
           dict(electrodes=ok, gain=float("nan")), dict(electrodes=ok, gain=float("inf")), dict(electrodes=ok, softening=0.0),
           dict(electrodes=ok, softening=-1.0), dict(electrodes=ok, softening=float("nan")), dict(electrodes=ok, softening=float("inf")),
           dict(electrodes=ok, rows=0), dict(electrodes=ok, rows=-3), dict(electrodes=np.zeros((256, 3), np.float32), rows=(1 << 16) + 1)]
    for kw in bad:
        with pytest.raises(SphsmError):
            s.egm_start(**kw)
    with pytest.raises(SphsmError):
        s.electrogram()  # a rejected start leaves electrograms off
    s.egm_start(np.zeros((256, 3), np.float32), rows=1 << 16)  # the largest ring
    s.egm_stop()
    s.egm_stop()  # (idempotent)


# ---- slab mode: virtual ranks ---------------------------------------------------------------------------------------------------
def _slab_group(nranks, pos, world, fixed, stimv, canonical=False):
    from sph_sm_monodomain_b200 import LocalGroup, Sim
    from tests.test_gpu_slabs import canonical_everywhere

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
        if canonical:
            canonical_everywhere(s)
        s.set_slab(lo, hi)
    return sims, grp


def _jittered(dims=(40, 9, 8)):
    pos, world = inputs.lattice(*dims, jitter=0.05)
    fixed, stim = inputs.lattice_masks(pos, dims[0], 4)
    return pos, world, fixed, np.where(stim, np.float32(300), np.float32(0)).astype(np.float32)


@pytest.mark.parametrize("nranks", [3, 4])
def test_virtual_ranks_merge(nranks):
    from tests.test_gpu_record import _owned_download

    pos, world, fixed, stimv = _jittered()
    n = len(pos)
    sims, grp = _slab_group(nranks, pos, world, fixed, stimv)
    geo = geometry(sims[0])
    el = electrodes(pos, geo[0])
    for s in sims:
        s.egm_start(el, rows=STEPS)
    recs = []
    pre = _owned_download(sims, n)[0]
    for act in pacing_schedule(0, STEPS, PERIOD, OFF_AFTER):
        if act[0] in ("stim", "off"):
            for s in sims:  # every rank alike
                if act[0] == "stim":
                    s.set_masks(None, stimv)
                else:
                    s.turnOffStim()
            pre = _owned_download(sims, n)[0]
            continue
        for _ in range(act[1]):
            grp.step(1)
            post = _owned_download(sims, n)[0]
            recs.append((sims[0].total_time_steps, pre, post))
            pre = post
    first, phi = grp.electrogram()
    assert first == 1 and all(s.electrogram()[0] == 1 for s in sims)
    check_rows(phi, *host_rows(recs, el, 1.0, geo[0], (geo[0], world, geo[2])))


def test_canonical_order_slabs_match_single_gpu():
    """With the canonical in-cell order every neighbour sum of the slab run visits its candidates as the single-GPU run does, but
    not every sum of the step is grouped alike (tests/test_gpu_slabs.py): the two states agree to a few ulps, not bit for bit (this
    holds with shape matching switched off too).  The electrograms then agree within 1e-6 of the summed absolute terms."""
    from sph_sm_monodomain_b200 import Sim
    from tests.test_gpu_record import _owned_download
    from tests.test_gpu_slabs import canonical_everywhere

    pos, world, fixed, stimv = _jittered()
    n = len(pos)
    sims, grp = _slab_group(3, pos, world, fixed, stimv, canonical=True)
    one = Sim(capacity=n, world=world, diagnostics=False)
    one.Init_Fluid(pos)
    one.set_masks(fixed.astype(np.uint8), stimv)
    canonical_everywhere(one)
    geo = geometry(one)
    el = electrodes(pos, geo[0])
    one.egm_start(el, rows=STEPS)
    for s in sims:
        s.egm_start(el, rows=STEPS)
    recs = []
    pre = one.particles()
    for act in pacing_schedule(0, STEPS, PERIOD, OFF_AFTER):
        if act[0] in ("stim", "off"):
            for s in sims + [one]:
                if act[0] == "stim":
                    s.set_masks(None, stimv)
                else:
                    s.turnOffStim()
            pre = one.particles()
            continue
        for _ in range(act[1]):
            grp.step(1)
            one.Animation(1)
            post = one.particles()
            recs.append((one.total_time_steps, pre, post))
            pre = post
    slab = _owned_download(sims, n)[0]
    assert rel_err(slab["pos"], pre["pos"]) <= 2e-6 and rel_err(slab["Vm"], pre["Vm"]) <= 2e-6  # the same trajectory
    f1, phi1 = one.electrogram()
    fs, phis = grp.electrogram()
    ref, scale = host_rows(recs, el, 1.0, geo[0], (geo[0], world, geo[2]))
    assert f1 == fs == 1
    check_rows(phi1, ref, scale)
    assert (np.abs(phis - phi1) <= 1e-6 * scale).all(), float((np.abs(phis - phi1) / scale).max())


# ---- NCCL slab path (2+ GPUs) ---------------------------------------------------------------------------------------------------
def test_nccl_ranks_merge():
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
           "--master-port", "29542", os.path.join(root, "tools", "egm_mg.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert r.returncode == 0 and lines, r.stdout[-2000:] + r.stderr[-2000:]
    res = json.loads(lines[-1])
    assert res["egm_mg"] == "ok", res
