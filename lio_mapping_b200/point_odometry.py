"""Host-side mirror of lio::PointOdometry (scan-to-scan odometry of the pre-initialisation phase and the /compact_data
pass-through) over the C-ABI: clouds, matching and the 6 x 6 Gauss-Newton live in the library (csrc/podom.cu).

Method names follow the reference (include/point_processor/PointOdometry.h): Process, EnableOdom; the topic handlers
collapse into the arguments of Process (one synchronised set of the five feature topics)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

_WHICH = {"last_corner": 0, "last_surf": 1, "full": 2}


class PointOdometry:
    def __init__(self, scan_period: float = 0.1, io_ratio: int = 2, num_max_iterations: int = 25, max_feature_points: int = 1 << 17,
                 max_full_points: int = 1 << 20, device: int = 0, stream: int = 0):
        _lib.require_device()
        self.max_feature_points, self.max_full_points = int(max_feature_points), int(max_full_points)
        self.h = C.c_void_p()
        _lib.check(_lib.lib().lio_po_create(scan_period, int(io_ratio), int(num_max_iterations), int(max_feature_points), int(max_full_points),
                                            device, C.c_void_p(stream), C.byref(self.h)), "lio_po_create")

    def close(self):
        if getattr(self, "h", None):
            _lib.lib().lio_po_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def EnableOdom(self, enable: bool):
        """The /enable_odom service (PointOdometry.cc:126-131)."""
        _lib.check(_lib.lib().lio_po_set_enable_odom(self.h, int(bool(enable))), "lio_po_set_enable_odom")

    def Process(self, corner_points_sharp, corner_points_less_sharp, surf_points_flat, surf_points_less_flat, full_cloud):
        """PointOdometry::Process + PublishResults: returns (transform_sum tf7, transform_es tf7, info dict)."""
        args = []
        for c in (corner_points_sharp, corner_points_less_sharp, surf_points_flat, surf_points_less_flat, full_cloud):
            c = np.ascontiguousarray(c, np.float32).reshape(-1, 4)
            args += [c if c.shape[0] else np.zeros((1, 4), np.float32), c.shape[0]]
        ts = np.zeros(7, np.float32); te = np.zeros(7, np.float32); info = np.zeros(4, np.int32)
        _lib.check(_lib.lib().lio_po_process_host(self.h, *args, ts, te, info), "lio_po_process_host")
        return ts, te, dict(iterations=int(info[0]), published=int(info[1]), frame_count=int(info[2]), matches=int(info[3]))

    def process_device(self, pp, n_max=None):
        """Process on the five stage-A clouds of `pp` (a PointProcessor) where they lie on the device, with their device counts:
        no host copy of a cloud.  n_max (optional, 5 ints) bounds the counts (a larger device count is clamped to it); default:
        pp.output_bounds() capped at this context's capacities.  Returns what Process returns.  The clouds that outlive the
        call are copied into this context, so `pp` may process the next sweep right away."""
        L = _lib.lib()
        names = ("corner_points_sharp", "corner_points_less_sharp", "surface_points_flat", "surface_points_less_flat", "laser_scans")
        if n_max is None:
            b = pp.output_bounds()
            n_max = [min(b[k], self.max_feature_points) for k in names[:4]] + [min(b["laser_scans"], self.max_full_points)]
        clouds = (_lib.DevCloud * 5)()
        for k, name in enumerate(names):
            clouds[k] = _lib.DevCloud(pp.cloud_dev(name), pp.count_dev(name), int(n_max[k]))
        ts = np.zeros(7, np.float32); te = np.zeros(7, np.float32); info = np.zeros(4, np.int32)
        _lib.check(L.lio_po_process_dev(self.h, clouds, ts, te, info), "lio_po_process_dev")
        return ts, te, dict(iterations=int(info[0]), published=int(info[1]), frame_count=int(info[2]), matches=int(info[3]))

    def cloud_dev(self, which: str):
        """(device pointer, device count pointer) of last_corner / last_surf / full; valid until the next process call."""
        p, n = C.c_void_p(), C.c_void_p()
        _lib.check(_lib.lib().lio_po_cloud_dev(self.h, _WHICH[which], C.byref(p), C.byref(n)), "lio_po_cloud_dev")
        return p.value, n.value

    def stats(self) -> dict:
        """What the last process call cost the host."""
        out = np.zeros(4, np.int64)
        _lib.check(_lib.lib().lio_po_last_stats(self.h, out), "lio_po_last_stats")
        return dict(launches=int(out[0]), syncs=int(out[1]), h2d_bytes=int(out[2]), d2h_bytes=int(out[3]))

    def cloud(self, which: str):
        w = _WHICH[which]
        n = C.c_int()
        _lib.check(_lib.lib().lio_po_cloud_size(self.h, w, C.byref(n)), "lio_po_cloud_size")
        out = np.zeros((max(n.value, 1), 4), np.float32)
        _lib.check(_lib.lib().lio_po_cloud_download(self.h, w, out, out.shape[0]), "lio_po_cloud_download")
        return out[:n.value]

    def compact_data(self):
        """The /compact_data payload of the sweep just processed as (3 + nc + ns + nf, 4) float32."""
        n = sum(self.cloud_size(w) for w in _WHICH) + 3
        out = np.zeros((n, 4), np.float32)
        m = C.c_int()
        _lib.check(_lib.lib().lio_po_compact_data(self.h, out, n, C.byref(m)), "lio_po_compact_data")
        return out[:m.value]

    def cloud_size(self, which: str) -> int:
        n = C.c_int()
        _lib.check(_lib.lib().lio_po_cloud_size(self.h, _WHICH[which], C.byref(n)), "lio_po_cloud_size")
        return n.value

    def matches(self, kind: str, n_queries: int):
        k = 0 if kind == "corner" else 1
        out = np.zeros((max(n_queries, 1), 2 + k), np.int32)
        _lib.check(_lib.lib().lio_po_matches(self.h, k, out, n_queries), "lio_po_matches")
        return out[:n_queries]

    def last_launches(self) -> int:
        return int(_lib.lib().lio_po_last_launches(self.h))
