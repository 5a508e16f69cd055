"""bench.py contract on the CPU-runnable arm: `--impl reference` (the oracle on the host cores) must print ONE JSON line
with the keys the driver reads.  The CUDA arm is exercised on the GPU box by the driver itself."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--workload", "vlp16"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "scans/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and abs(d["value"] - 1e3 / d["ms_per_step"]) < 1e-6 * d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_reference_arm_dumps_the_same_outputs_every_run(tmp_path):
    """--dump-outputs writes the last timed scan's window states and stage-A clouds; the same arguments give the same inputs, so
    two runs of the (deterministic) oracle write identical files."""
    import numpy as np
    names = ["states", "corner_points_sharp", "corner_points_less_sharp", "surface_points_flat", "surface_points_less_flat"]
    dumps = []
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                              "--workload", "vlp16", "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=600,
                             cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
        assert sorted(os.listdir(tmp_path / run)) == sorted(n + ".npy" for n in names)
        dumps.append({n: np.load(tmp_path / run / (n + ".npy")) for n in names})
    a, b = dumps
    assert a["states"].dtype == np.float64 and a["states"].shape == (11, 16)
    assert a["surface_points_less_flat"].dtype == np.float32 and a["surface_points_less_flat"].shape[0] > 1000
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for n in names:
        assert np.array_equal(a[n], b[n]), n


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1", "--workload", "vlp16"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
