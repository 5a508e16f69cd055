"""Host-side mirror of lio::PointMapping (pre-initialisation scan-to-map path) over the C-ABI: the rolling cube map
lives in HBM inside the library (csrc/cubemap.cu), the Python layer only moves arrays.

Method names follow the reference (include/point_processor/PointMapping.h): Process, and accessors for the cube arrays
laser_cloud_corner_array_ / laser_cloud_surf_array_."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

NUM_CUBES = 21 * 21 * 11


class PointMapping:
    def __init__(self, max_points: int = 1 << 17, corner_filter_size: float = 0.2, surf_filter_size: float = 0.4,
                 min_match_sq_dis: float = 1.0, min_plane_dis: float = 0.2, max_iterations: int = 10, device: int = 0, stream: int = 0):
        _lib.require_device()
        self.max_points = int(max_points)
        self.h = C.c_void_p()
        _lib.check(_lib.lib().lio_pm_create(int(max_points), corner_filter_size, surf_filter_size, min_match_sq_dis, min_plane_dis,
                                            int(max_iterations), device, C.c_void_p(stream), C.byref(self.h)), "lio_pm_create")

    def close(self):
        if getattr(self, "h", None):
            _lib.lib().lio_pm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def Process(self, corner_last, surf_last, transform_sum7):
        """PointMapping::Process: returns (transform_tobe_mapped tf7, info dict)."""
        c = np.ascontiguousarray(corner_last, np.float32).reshape(-1, 4); s = np.ascontiguousarray(surf_last, np.float32).reshape(-1, 4)
        tobe = np.zeros(7, np.float32); info = np.zeros(3, np.int32)
        _lib.check(_lib.lib().lio_pm_process_host(self.h, c if c.shape[0] else np.zeros((1, 4), np.float32), c.shape[0],
                                                  s if s.shape[0] else np.zeros((1, 4), np.float32), s.shape[0],
                                                  np.ascontiguousarray(transform_sum7, np.float32), tobe, info), "lio_pm_process_host")
        return tobe, dict(iterations=int(info[0]), corner_from_map=int(info[1]), surf_from_map=int(info[2]))

    def process_device(self, po, transform_sum7):
        """Process on the odometry's last_corner / last_surf clouds (a PointOdometry) where they lie on the device; transform_sum7
        as po's Process / process_device returned it.  The bound of each count is the size po read back with its last call."""
        L = _lib.lib()
        clouds = []
        for which in ("last_corner", "last_surf"):
            p, n = po.cloud_dev(which)
            clouds.append(_lib.DevCloud(p, n, po.cloud_size(which)))
        tobe = np.zeros(7, np.float32); info = np.zeros(3, np.int32)
        _lib.check(L.lio_pm_process_dev(self.h, C.byref(clouds[0]), C.byref(clouds[1]), np.ascontiguousarray(transform_sum7, np.float32), tobe, info),
                   "lio_pm_process_dev")
        return tobe, dict(iterations=int(info[0]), corner_from_map=int(info[1]), surf_from_map=int(info[2]))

    def process_dev_clouds(self, corner, surf, transform_sum7):
        """Process on explicit device clouds: corner / surf = (device pointer, device count pointer, n_max)."""
        tobe = np.zeros(7, np.float32); info = np.zeros(3, np.int32)
        c, s = _lib.DevCloud(*corner), _lib.DevCloud(*surf)
        _lib.check(_lib.lib().lio_pm_process_dev(self.h, C.byref(c), C.byref(s), np.ascontiguousarray(transform_sum7, np.float32), tobe, info),
                   "lio_pm_process_dev")
        return tobe, dict(iterations=int(info[0]), corner_from_map=int(info[1]), surf_from_map=int(info[2]))

    def stats(self) -> dict:
        """What the last process call cost the host."""
        out = np.zeros(4, np.int64)
        _lib.check(_lib.lib().lio_pm_last_stats(self.h, out), "lio_pm_last_stats")
        return dict(launches=int(out[0]), syncs=int(out[1]), h2d_bytes=int(out[2]), d2h_bytes=int(out[3]))

    def centre(self):
        out = np.zeros(3, np.int32)
        _lib.check(_lib.lib().lio_pm_map_centre(self.h, out), "lio_pm_map_centre")
        return tuple(out.tolist())

    def cube_sizes(self, which):
        w = 0 if which == "corner" else 1
        n = C.c_int()
        out = np.zeros(NUM_CUBES, np.int64)
        L = _lib.lib()
        for i in range(NUM_CUBES):
            L.lio_pm_cube_size(self.h, i, w, C.byref(n))
            out[i] = n.value
        return out

    def cube(self, index, which):
        w = 0 if which == "corner" else 1
        n = C.c_int()
        _lib.check(_lib.lib().lio_pm_cube_size(self.h, int(index), w, C.byref(n)), "lio_pm_cube_size")
        out = np.zeros((max(n.value, 1), 4), np.float32)
        _lib.check(_lib.lib().lio_pm_cube_download(self.h, int(index), w, out, out.shape[0]), "lio_pm_cube_download")
        return out[:n.value]
