"""CPU side of the pre-initialisation chain: the hand-off the device chain relies on (PointMapping fed the odometry's clouds and
transform_sum_ directly == fed the decoded /compact_data payload), and the contract of scripts/premap_bench.py."""
import json
import os
import subprocess
import sys

import numpy as np

from tests.test_oracle_point_odometry import sweeps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT = os.path.join(ROOT, "scripts", "premap_bench.py")


def test_mapping_on_the_odometry_clouds_equals_mapping_on_the_payload(oracle):
    fr = sweeps(oracle, "vlp16", 5)
    po = oracle.PointOdometryOracle(0.1, 2, 25)
    via_payload, direct = oracle.PointMappingOracle(), oracle.PointMappingOracle()
    mapped = 0
    for s in fr:
        ts, _, info = po.process(s["sharp"], s["less_sharp"], s["flat"], s["less_flat"], s["full"])
        if not info["published"]:
            continue
        tf7, c, sf, _ = oracle.compact_decode(po.cloud("compact"))
        a = via_payload.process(c, sf, tf7)
        b = direct.process(po.cloud("last_corner"), po.cloud("last_surf"), ts)
        assert np.array_equal(tf7, ts) and np.array_equal(a[0], b[0]) and a[1] == b[1]
        assert via_payload.centre() == direct.centre()
        for which in ("corner", "surf"):
            sa, sb = via_payload.cube_sizes(which), direct.cube_sizes(which)
            assert np.array_equal(sa, sb)
            for idx in np.nonzero(sa)[0]:
                assert np.array_equal(via_payload.cube(idx, which), direct.cube(idx, which))
        mapped += 1
    assert mapped == 2


def _run(*args):
    return subprocess.run([sys.executable, SCRIPT, *args], capture_output=True, text=True, cwd=ROOT, timeout=900)


def test_premap_bench_reference_arm_prints_one_json_line():
    p = _run("--impl", "reference", "--workload", "vlp16", "--sweeps", "3", "--warmup", "1")
    assert p.returncode == 0, p.stderr
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    r = json.loads(lines[0])
    for k in ("impl", "workload", "sweeps", "warmup", "median_ms", "p95_ms", "max_ms", "sweeps_per_s", "stage_median_ms", "per_sweep", "gpu",
              "note", "parity"):
        assert k in r, k
    assert r["impl"] == "reference" and r["workload"] == "vlp16" and r["sweeps"] == 3
    assert set(r["stage_median_ms"]) == {"stage_a", "odometry", "mapping"} and r["median_ms"] > 0
    assert set(r["per_sweep"]) == {"launches", "syncs", "h2d_bytes", "d2h_bytes"}


def test_premap_bench_gpu_arm_without_a_device_fails_clearly():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is visible here")
    p = _run("--impl", "device", "--workload", "vlp16", "--sweeps", "2", "--warmup", "0")
    assert p.returncode != 0 and "needs a CUDA device" in p.stderr and not p.stdout.strip()
