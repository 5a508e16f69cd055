"""Pre-initialisation pipeline benchmark: stage A -> PointOdometry -> PointMapping, one sweep per timed unit.

Workload: a seeded, motion-distorted synthetic drive (lio_mapping_b200.synth, `hdl64` or `vlp16`), generated before timing.
One timed unit is one sweep through stage A and the odometry, plus the mapping when the odometry's io_ratio gate publishes
(every second sweep).  Arms:
  --impl device     raw sweeps resident in HBM, the chain through the _dev entries (no host copy of a cloud)
  --impl host       the same chain through the _host entries: every hand-off goes through host buffers (stage-A clouds
                    downloaded and uploaded again, the /compact_data payload downloaded and decoded, then uploaded again)
  --impl reference  the oracle chain on the CPU (stage_a -> PointOdometryOracle -> compact encode / decode ->
                    PointMappingOracle): the CPU baseline
The two GPU arms always run together in one process, alternating sweep by sweep on two independent chains; --impl picks the
arm reported at the top level, the other one is reported under "other_arm", and "parity" compares them (final pose, every
odometry pose, cube sizes: array_equal).  A GPU arm without a device exits non-zero; there is no fallback.

Prints one JSON line.  Writes nothing unless --out is given.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PP_NAMES = ("corner_points_sharp", "corner_points_less_sharp", "surface_points_flat", "surface_points_less_flat", "laser_scans")
NOTE = ("the map working set (cube segments, pulled maps, last clouds) is a few MB and stays L2-resident across sweeps, as in the "
        "real pipeline; the raw sweeps of the device arm are resident in HBM, the host arm starts from host arrays")


def make_drive(kind, n, seed0=70, t0=1.0):
    from lio_mapping_b200 import synth
    sensor, scene, traj = synth.default_config(kind)
    raw = [np.ascontiguousarray(synth.make_sweep(sensor, scene, traj, t0 + 0.1 * f, seed=seed0 + f, distort=True), np.float32) for f in range(n)]
    return sensor, raw


def summarise(ms):
    a = np.asarray(ms, np.float64)
    med = float(np.median(a))
    return dict(median_ms=med, p95_ms=float(np.percentile(a, 95)), max_ms=float(a.max()), sweeps_per_s=1000.0 / med if med > 0 else None)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = [x.strip() for x in out[0].split(",")]
        return dict(name=name, power_limit_w=float(power))
    except Exception as e:   # the record still carries torch's device name
        import torch
        return dict(name=torch.cuda.get_device_name(0), power_limit_w=None, nvidia_smi_error=str(e))


def run_reference(kind, sweeps, warmup):
    from oracle import oracle_py as O
    O.build()
    sensor, raw = make_drive(kind, warmup + sweeps)
    po = O.PointOdometryOracle(0.1, 2, 25)
    pm = O.PointMappingOracle()
    total, st_a, st_o, st_m = [], [], [], []
    for f, sw in enumerate(raw):
        t0 = time.perf_counter()
        r = O.stage_a(sw, sensor.lower_deg, sensor.upper_deg, sensor.rings)
        t1 = time.perf_counter()
        ts, _, info = po.process(r["sharp"], r["less_sharp"], r["flat"], r["less_flat"], r["laser_scans"])
        t2 = time.perf_counter()
        if info["published"]:
            tf7, c, s, _ = O.compact_decode(po.cloud("compact"))
            pm.process(c, s, tf7)
        t3 = time.perf_counter()
        if f >= warmup:
            total.append(1e3 * (t3 - t0)); st_a.append(1e3 * (t1 - t0)); st_o.append(1e3 * (t2 - t1))
            if info["published"]:
                st_m.append(1e3 * (t3 - t2))
    res = dict(impl="reference", workload=kind, sweeps=sweeps, warmup=warmup, **summarise(total),
               stage_median_ms=dict(stage_a=float(np.median(st_a)), odometry=float(np.median(st_o)),
                                    mapping=float(np.median(st_m)) if st_m else None),
               per_sweep=dict(launches=0, syncs=0, h2d_bytes=0, d2h_bytes=0), gpu=None, note="CPU oracle chain (single thread)", parity=None)
    return res


class GpuChain:
    def __init__(self, sensor, device_arm, max_points):
        from lio_mapping_b200.point_mapping import PointMapping
        from lio_mapping_b200.point_odometry import PointOdometry
        from lio_mapping_b200.point_processor import PointProcessor
        self.device_arm = device_arm
        self.pp = PointProcessor(sensor.lower_deg, sensor.upper_deg, sensor.rings, max_points=max_points)
        self.po = PointOdometry(0.1, 2, 25)
        self.pm = PointMapping(max_points=1 << 17)
        self.poses, self.tobe = [], None

    def step(self, raw_host, raw_dev, ev):
        """One sweep; ev = 4 CUDA events recorded at the stage boundaries.  Returns {launches, syncs, h2d, d2h} of the sweep."""
        from lio_mapping_b200 import wire
        c = dict(launches=0, syncs=0, h2d=0, d2h=0)
        ev[0].record()
        if self.device_arm:
            self.pp.process_device(raw_dev.data_ptr(), raw_dev.shape[0])
            c["d2h"] += 24                                            # stage A's asynchronous count read-back
        else:
            self.pp.SetInputCloud(raw_host); self.pp.Process()
            c["h2d"] += 16 * raw_host.shape[0]; c["syncs"] += 1
        c["launches"] += self.pp.last_launches()
        ev[1].record()
        if self.device_arm:
            ts, _, info = self.po.process_device(self.pp)
        else:
            clouds = [self.pp.cloud(k) for k in PP_NAMES]
            c["d2h"] += sum(16 * x.shape[0] for x in clouds); c["syncs"] += sum(1 for x in clouds if x.shape[0])
            ts, _, info = self.po.Process(*clouds)
        s = self.po.stats()
        c["launches"] += s["launches"]; c["syncs"] += s["syncs"]; c["h2d"] += s["h2d_bytes"]; c["d2h"] += s["d2h_bytes"]
        self.poses.append(ts)
        ev[2].record()
        if info["published"]:
            if self.device_arm:
                self.tobe, _ = self.pm.process_device(self.po, ts)
            else:
                payload = self.po.compact_data()
                c["d2h"] += 16 * payload.shape[0]; c["syncs"] += 1
                tf7, corner, surf, _ = wire.compact_decode(payload)
                self.tobe, _ = self.pm.Process(corner, surf, tf7)
            s = self.pm.stats()
            c["launches"] += s["launches"]; c["syncs"] += s["syncs"]; c["h2d"] += s["h2d_bytes"]; c["d2h"] += s["d2h_bytes"]
        ev[3].record()
        return info["published"], c


def run_gpu(impl, kind, sweeps, warmup):
    import torch
    from lio_mapping_b200 import _lib
    if not torch.cuda.is_available() or _lib.lib().lio_device_count() <= 0:
        print(f"premap_bench: --impl {impl} needs a CUDA device and none is usable (no CPU fallback; use --impl reference for the CPU baseline)",
              file=sys.stderr)
        sys.exit(2)
    sensor, raw = make_drive(kind, warmup + sweeps)
    max_points = max(r.shape[0] for r in raw)
    dev_raw = [torch.from_numpy(r).cuda() for r in raw]
    torch.cuda.synchronize()
    arms = {"device": GpuChain(sensor, True, max_points), "host": GpuChain(sensor, False, max_points)}
    rec = {a: dict(total=[], stage_a=[], odometry=[], mapping=[], counts=[]) for a in arms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    for f in range(len(raw)):
        order = ("device", "host") if f % 2 == 0 else ("host", "device")   # alternate which arm goes first
        for a in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            published, c = arms[a].step(raw[f], dev_raw[f], ev)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if f < warmup:
                continue
            r = rec[a]
            r["total"].append(1e3 * (t1 - t0))
            r["stage_a"].append(ev[0].elapsed_time(ev[1])); r["odometry"].append(ev[1].elapsed_time(ev[2]))
            if published:
                r["mapping"].append(ev[2].elapsed_time(ev[3]))
            r["counts"].append(c)

    def arm_result(a):
        r = rec[a]
        cnt = {k: float(np.mean([c[k] for c in r["counts"]])) for k in ("launches", "syncs", "h2d", "d2h")}
        return dict(impl=a, **summarise(r["total"]),
                    stage_median_ms=dict(stage_a=float(np.median(r["stage_a"])), odometry=float(np.median(r["odometry"])),
                                         mapping=float(np.median(r["mapping"])) if r["mapping"] else None),
                    per_sweep=dict(launches=cnt["launches"], syncs=cnt["syncs"], h2d_bytes=cnt["h2d"], d2h_bytes=cnt["d2h"]))

    d, h = arms["device"], arms["host"]
    parity = dict(final_pose=bool(np.array_equal(d.tobe, h.tobe)),
                  odometry_poses=bool(all(np.array_equal(x, y) for x, y in zip(d.poses, h.poses))),
                  cube_sizes=bool(all(np.array_equal(d.pm.cube_sizes(w), h.pm.cube_sizes(w)) for w in ("corner", "surf"))))
    parity["all"] = all(parity.values())
    other = "host" if impl == "device" else "device"
    res = dict(arm_result(impl), workload=kind, sweeps=sweeps, warmup=warmup, points_per_sweep=int(np.median([r.shape[0] for r in raw])),
               timing="host clock around each sweep ending in a device synchronise; stage medians from CUDA events; mapping median over "
                      "the published sweeps",
               gpu=gpu_info(), note=NOTE, parity=parity, other_arm=arm_result(other))
    res["device_over_host_median"] = res["median_ms"] / res["other_arm"]["median_ms"] if impl == "device" else res["other_arm"]["median_ms"] / res["median_ms"]
    return res


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--impl", choices=("device", "host", "reference"), default="device")
    ap.add_argument("--workload", choices=("hdl64", "vlp16"), default="hdl64")
    ap.add_argument("--sweeps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--out", default=None, help="also write the JSON record to this path")
    a = ap.parse_args(argv)
    if a.sweeps < 1 or a.warmup < 0:
        ap.error("--sweeps must be >= 1 and --warmup >= 0")
    res = run_reference(a.workload, a.sweeps, a.warmup) if a.impl == "reference" else run_gpu(a.impl, a.workload, a.sweeps, a.warmup)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
