"""GPU: bench.py --dump-outputs on the CUDA path — the files, their dtype, the seeded sample above DUMP_MAX_PARTICLES, the same
bytes from run to run, and the state they hold is the state after exactly the warm-up and the --steps timed steps."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WORKLOAD = "110x100x100"  # 1.1M particles: above DUMP_MAX_PARTICLES, so the sample path is taken


def test_dump_outputs_of_the_timed_path(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    from sph_sm_monodomain_b200 import Sim

    steps, warmup = 7, 3
    dumps = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", WORKLOAD, "--steps", str(steps), "--warmup",
                            str(warmup), "--no-cpu-baseline", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        dumps.append({f.name: np.load(f) for f in sorted(out.iterdir())})
    assert sorted(dumps[0]) == sorted(f + ".npy" for f in bench.DUMP_FIELDS)
    for name, a in dumps[0].items():
        assert a.dtype == np.float32 and len(a) == bench.DUMP_MAX_PARTICLES and np.isfinite(a).all(), name
        assert a.tobytes() == dumps[1][name].tobytes(), name

    # the same steps outside bench.py: warm-up, then the timed steps, then Get_Paticles()
    pos, world, fixed, stim = bench.workload_inputs(bench.parse_workload(WORKLOAD))
    sim = Sim(capacity=len(pos), world=world, diagnostics=False)
    sim.Init_Fluid(pos)
    sim.set_masks(fixed, stim)
    sim.Animation(max(warmup, bench.FIXED_WARMUP))
    sim.Animation(steps)
    ref = tmp_path / "direct"
    bench.dump_outputs(str(ref), sim.particles())
    sim.close()
    for name, a in dumps[0].items():
        assert a.tobytes() == np.load(ref / name).tobytes(), name
