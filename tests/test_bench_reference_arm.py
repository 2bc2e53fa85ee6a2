"""bench.py --impl reference runs without a GPU: it times the reference's own CPU implementation (oracle/_ref when the
genuine reference was compiled here, else the C restatement) and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("workload", ["cfg1", "8m"])
def test_reference_arm_prints_the_contract_line(workload):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload, "--steps", "3",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["unit"] == "particle-steps/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 3
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] == 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    if workload == "cfg1":
        assert "4944" in line["cpu_baseline"]["sample"]


def test_reference_arm_dumps_the_same_outputs_every_run(tmp_path):
    """--dump-outputs: the state after the timed steps as float32 .npy files, identical from run to run with the same arguments;
    --steps sets the number of timed steps, also above 100."""
    dumps = []
    for k in range(2):
        out = tmp_path / f"run{k}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "101",
                            "--warmup", "1", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])["steps"] == 101
        dumps.append({f.name: np.load(f) for f in sorted(out.iterdir())})
    sys.path.insert(0, ROOT)
    import bench

    assert sorted(dumps[0]) == sorted(f + ".npy" for f in bench.DUMP_FIELDS)
    for name, a in dumps[0].items():
        assert a.dtype == np.float32 and len(a) == 4944 and np.isfinite(a).all(), name
        assert a.tobytes() == dumps[1][name].tobytes(), name
    assert not np.array_equal(dumps[0]["pos.npy"], np.load(os.path.join(ROOT, "tests", "golden", "cfg1_4944.npz"))["positions"])


def test_pacing_schedule_of_the_32m_workload():
    """configs[4]: stimulus on the end slab every 50 steps, turnOffStim 25 steps later (SURVEY.md 8d.5), wherever the window starts."""
    sys.path.insert(0, ROOT)
    import bench

    def events(start, n):
        k, ev = start, []
        for a in bench.pacing_schedule(start, n, 50, 25):
            if a[0] == "run":
                assert a[1] > 0
                k += a[1]
            else:
                ev.append((a[0], k))
        assert k == start + n
        return ev

    assert events(0, 120) == [("stim", 0), ("off", 25), ("stim", 50), ("off", 75), ("stim", 100)]
    assert events(400, 100) == [("stim", 400), ("off", 425), ("stim", 450), ("off", 475)]
    assert events(410, 30) == [("off", 425)]
    assert events(26, 10) == []
    assert bench.WORKLOADS["32m"]["pacing"] == (50, 25)
