"""Host-side mirror of lio::PointProcessor over the C-ABI (stage A).

Same method names and meaning as the reference class (include/point_processor/PointProcessor.h:
122-229): SetupConfig, SetInputCloud, PointToRing, ExtractFeaturePoints, Process; results are the
reference's member clouds.  All compute happens in liblio_b200.so on the GPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

CLOUDS = {"laser_scans": 0, "cloud_in_rings": 1, "corner_points_sharp": 2, "corner_points_less_sharp": 3,
          "surface_points_flat": 4, "surface_points_less_flat": 5}
INDICES = {"sharp": 0, "less_sharp": 1, "flat": 2, "orig": 3}


class PointProcessor:
    def __init__(self, lower_bound: float = -15.0, upper_bound: float = 15.0, num_rings: int = 16,
                 max_points: int = 1 << 20, device: int = 0, stream: int = 0, **config):
        L = _lib.lib()
        _lib.require_device()
        cfg = _lib.PPConfig()
        L.lio_pp_default_config(C.byref(cfg))
        cfg.lower_bound, cfg.upper_bound, cfg.num_rings = lower_bound, upper_bound, num_rings
        for k, v in config.items():
            if not hasattr(cfg, k):
                raise AttributeError(f"PointProcessorConfig has no field {k}")
            setattr(cfg, k, v)
        self.cfg = cfg
        self.max_points = max_points
        self._h = C.c_void_p()
        _lib.check(L.lio_pp_create(C.byref(cfg), max_points, device, C.c_void_p(stream), C.byref(self._h)), "lio_pp_create")
        self._cloud = None
        self.last_input_size = 0

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            _lib.lib().lio_pp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference-shaped API -----------------------------------------------------------------
    def SetInputCloud(self, cloud_in: np.ndarray):
        self._cloud = np.ascontiguousarray(cloud_in, dtype=np.float32).reshape(-1, 4)

    def Process(self):
        """PointToRing + ExtractFeaturePoints (PointProcessor.cc:96-100); host buffers in/out."""
        if self._cloud is None:
            raise _lib.LioError("SetInputCloud first")
        _lib.check(_lib.lib().lio_pp_process_host(self._h, self._cloud, self._cloud.shape[0]), "lio_pp_process_host")
        self.last_input_size = self._cloud.shape[0]

    def ProcessWithRingField(self, rings):
        """PointToRing for PointXYZIR input (ring index per point, PointProcessor.cc:428-536) + ExtractFeaturePoints."""
        if self._cloud is None:
            raise _lib.LioError("SetInputCloud first")
        r = np.ascontiguousarray(rings, np.uint16)
        if r.shape[0] != self._cloud.shape[0]:
            raise ValueError("one ring index per point")
        _lib.check(_lib.lib().lio_pp_process_host_ring(self._h, self._cloud, r, self._cloud.shape[0]), "lio_pp_process_host_ring")
        self.last_input_size = self._cloud.shape[0]

    def process_device(self, dev_ptr: int, n: int):
        """Device-resident input (float4 array); asynchronous on the processor's stream."""
        _lib.check(_lib.lib().lio_pp_process_dev(self._h, C.c_void_p(dev_ptr), n), "lio_pp_process_dev")
        self.last_input_size = int(n)

    def output_bounds(self) -> dict:
        """Upper bounds of the feature cloud sizes of the last process call, known without reading the counts back: at most
        max_corner_sharp / max_corner_less_sharp / max_surf_flat points per ring and subregion (ExtractFeaturePoints),
        and never more points than the sweep had."""
        c, n = self.cfg, self.last_input_size
        rs = c.num_rings * c.num_scan_subregions
        return {"corner_points_sharp": min(n, rs * c.max_corner_sharp), "corner_points_less_sharp": min(n, rs * c.max_corner_less_sharp),
                "surface_points_flat": min(n, rs * c.max_surf_flat), "surface_points_less_flat": n, "laser_scans": n}

    # -- results ------------------------------------------------------------------------------
    def sizes(self) -> dict:
        s = np.zeros(6, np.int32)
        _lib.check(_lib.lib().lio_pp_cloud_sizes(self._h, s), "lio_pp_cloud_sizes")
        return {k: int(s[v]) for k, v in CLOUDS.items()}

    def cloud(self, name: str) -> np.ndarray:
        w = CLOUDS[name]
        n = self.sizes()[name]
        out = np.zeros((max(n, 1), 4), np.float32)
        got = C.c_int()
        _lib.check(_lib.lib().lio_pp_download_cloud(self._h, w, out, out.shape[0], C.byref(got)), "lio_pp_download_cloud")
        return out[:got.value].copy()

    def cloud_dev(self, name: str) -> int:
        p = C.c_void_p()
        _lib.check(_lib.lib().lio_pp_cloud_dev(self._h, CLOUDS[name], C.byref(p)), "lio_pp_cloud_dev")
        return p.value

    def count_dev(self, name: str) -> int:
        """Device pointer of the point count of one output cloud (lio_pp_cloud_count_dev), to chain stage A on the device."""
        p = C.c_void_p()
        _lib.check(_lib.lib().lio_pp_cloud_count_dev(self._h, CLOUDS[name], C.byref(p)), "lio_pp_cloud_count_dev")
        return p.value

    def index(self, name: str) -> np.ndarray:
        cap = self.sizes()["laser_scans"] + 1
        out = np.zeros(cap, np.int32)
        got = C.c_int()
        _lib.check(_lib.lib().lio_pp_download_index(self._h, INDICES[name], out, cap, C.byref(got)), "lio_pp_download_index")
        return out[:got.value].copy()

    def scan_ranges(self) -> np.ndarray:
        out = np.zeros(2 * self.cfg.num_rings, np.int32)
        _lib.check(_lib.lib().lio_pp_download_scan_ranges(self._h, out), "lio_pp_download_scan_ranges")
        return out.reshape(-1, 2)

    def mask_labels(self):
        n = self.sizes()["laser_scans"]
        m = np.zeros(max(n, 1), np.uint8)
        lab = np.zeros(max(n, 1), np.int8)
        _lib.check(_lib.lib().lio_pp_download_mask_labels(self._h, m, lab, m.shape[0]), "lio_pp_download_mask_labels")
        return m[:n], lab[:n]

    def start_ori(self) -> float:
        v = C.c_float()
        _lib.check(_lib.lib().lio_pp_start_ori(self._h, C.byref(v)), "lio_pp_start_ori")
        return v.value

    def last_launches(self) -> int:
        return int(_lib.lib().lio_pp_last_launches(self._h))
