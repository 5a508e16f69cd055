"""The pre-initialisation chain on the device: stage A -> PointOdometry -> PointMapping through the _dev entries (no host copy of a
cloud), against the same chain through the _host entries (bit for bit) and against the oracle chain; lifetime of the inputs, the
pass-through into the estimator, the transfer bound of one call, argument handling and the growth of the re-filter workspace."""
import numpy as np
import pytest

from lio_mapping_b200 import synth
from tests import helpers

pytestmark = pytest.mark.gpu

PP_NAMES = ("corner_points_sharp", "corner_points_less_sharp", "surface_points_flat", "surface_points_less_flat", "laser_scans")
WHICH = ("last_corner", "last_surf", "full")


def _drive(kind, n, seed0=70, t0=1.0):
    sensor, scene, traj = synth.default_config(kind)
    raw, poses = [], []
    for f in range(n):
        t_end = t0 + 0.1 * f
        raw.append(np.ascontiguousarray(synth.make_sweep(sensor, scene, traj, t_end, seed=seed0 + f, distort=True), np.float32))
        p, R, _, _, _ = traj.state(np.array(t_end))
        poses.append((R, p))
    return sensor, raw, poses


def _cubes(pm):
    out = {}
    for which in ("corner", "surf"):
        sizes = pm.cube_sizes(which)
        out[which] = (sizes, {int(i): pm.cube(int(i), which) for i in np.nonzero(sizes)[0]})
    return out


def _assert_maps_equal(a, b, tag):
    for which in ("corner", "surf"):
        assert np.array_equal(a[which][0], b[which][0]), (tag, which)
        for i, c in a[which][1].items():
            assert np.array_equal(c, b[which][1][i]), (tag, which, i)


class Chain:
    """One stage A -> odometry -> mapping chain on the GPU, through the _dev entries (device=True) or the _host entries."""

    def __init__(self, sensor, device, io_ratio=2, pm_max_points=1 << 17):
        from lio_mapping_b200.point_mapping import PointMapping
        from lio_mapping_b200.point_odometry import PointOdometry
        from lio_mapping_b200.point_processor import PointProcessor
        self.device = device
        self.pp = PointProcessor(sensor.lower_deg, sensor.upper_deg, sensor.rings, max_points=1 << 18)
        self.po = PointOdometry(0.1, io_ratio, 25)
        self.pm = PointMapping(max_points=pm_max_points)

    def step(self, raw):
        import torch
        if self.device:
            t = torch.from_numpy(raw).cuda()
            self.pp.process_device(t.data_ptr(), t.shape[0])
            ts, te, info = self.po.process_device(self.pp)
            del t
        else:
            self.pp.SetInputCloud(raw); self.pp.Process()
            ts, te, info = self.po.Process(*[self.pp.cloud(k) for k in PP_NAMES])
        out = dict(ts=ts, te=te, info=info, payload=None, tobe=None, info3=None)
        if info["published"]:
            if self.device:
                out["tobe"], out["info3"] = self.pm.process_device(self.po, ts)
            else:
                from lio_mapping_b200 import wire
                payload = self.po.compact_data()
                tf7, c, s, _ = wire.compact_decode(payload)
                out["tobe"], out["info3"] = self.pm.Process(c, s, tf7)
        return out


@pytest.mark.parametrize("kind", ["hdl64", "vlp16"])
def test_device_chain_equals_host_chain(kind):
    sensor, raw, _ = _drive(kind, 8)
    dev, host = Chain(sensor, True), Chain(sensor, False)
    mapped = 0
    for f, sw in enumerate(raw):
        a, b = dev.step(sw), host.step(sw)
        assert np.array_equal(a["ts"], b["ts"]) and np.array_equal(a["te"], b["te"]) and a["info"] == b["info"], (f, a, b)
        for w in WHICH:
            assert np.array_equal(dev.po.cloud(w), host.po.cloud(w)), (f, w)
        if a["info"]["published"]:
            assert np.array_equal(dev.po.compact_data(), host.po.compact_data()), f
            assert np.array_equal(a["tobe"], b["tobe"]) and a["info3"] == b["info3"], (f, a["tobe"], b["tobe"], a["info3"], b["info3"])
            assert dev.pm.centre() == host.pm.centre()
            mapped += 1
    assert mapped == 4 and a["info3"]["iterations"] >= 1
    _assert_maps_equal(_cubes(dev.pm), _cubes(host.pm), kind)


@pytest.mark.parametrize("kind", ["hdl64", "vlp16"])
def test_device_chain_against_the_oracle_chain(oracle, kind):
    sensor, raw, poses = _drive(kind, 8)
    dev = Chain(sensor, True)
    po = oracle.PointOdometryOracle(0.1, 2, 25)
    pm = oracle.PointMappingOracle()
    worst, anchor = (0.0, 0.0), None
    for f, sw in enumerate(raw):
        g = dev.step(sw)
        r = oracle.stage_a(sw, sensor.lower_deg, sensor.upper_deg, sensor.rings)
        to, eo, io = po.process(r["sharp"], r["less_sharp"], r["flat"], r["less_flat"], r["laser_scans"])
        tg, eg, ig = g["ts"], g["te"], g["info"]
        assert ig["published"] == io["published"] and ig["frame_count"] == io["frame_count"]
        if f > 0:   # the tolerances of test_point_odometry_gpu.py
            assert abs(ig["iterations"] - io["iterations"]) <= 1 and abs(ig["matches"] - io["matches"]) <= 2 + 0.01 * io["matches"]
            scale = max(1.0, float(np.abs(to[4:]).max()))
            assert np.abs(eg[4:] - eo[4:]).max() <= 2e-4 and min(np.abs(eg[:4] - eo[:4]).max(), np.abs(eg[:4] + eo[:4]).max()) <= 2e-5, (f, eg, eo)
            assert np.abs(tg[4:] - to[4:]).max() <= 3e-4 * scale and min(np.abs(tg[:4] - to[:4]).max(), np.abs(tg[:4] + to[:4]).max()) <= 5e-5, (f, tg, to)
        if not io["published"]:
            continue
        tf7, c, s, _ = oracle.compact_decode(po.cloud("compact"))
        tobe_o, _ = pm.process(c, s, tf7)
        tobe_g = g["tobe"]
        for which in ("corner", "surf"):
            assert np.array_equal(pm.cube_sizes(which) > 0, dev.pm.cube_sizes(which) > 0), (f, which)
        # against the truth: the map is anchored at the odometry's pose of the first published sweep (no map yet, nothing to
        # correct; the reference's HDL-64 odometry is 0.15 m off there on this drive, the oracle chain alike), so the mapped
        # trajectory is compared with the true one from that anchor on
        _, _, tf_true = helpers.rel_transform(poses[0], poses[f])
        if anchor is None:
            anchor = (tobe_g[4:].copy(), tobe_o[4:].copy(), tf_true[4:].copy())
        else:
            moved = tf_true[4:] - anchor[2]
            assert np.linalg.norm(tobe_g[4:] - anchor[0] - moved) < 0.08 and np.linalg.norm(tobe_o[4:] - anchor[1] - moved) < 0.08, (f, tobe_g, tobe_o, tf_true)
        dp = float(np.abs(tobe_g[4:] - tobe_o[4:]).max())
        dq = float(min(np.abs(tobe_g[:4] - tobe_o[:4]).max(), np.abs(tobe_g[:4] + tobe_o[:4]).max()))
        worst = (max(worst[0], dp), max(worst[1], dq))
        assert dp <= 1e-3 and dq <= 1e-4, f"sweep {f}: mapped pose differs from the oracle chain by {dp:.3g} m, {dq:.3g} per quaternion component"
    print(kind, "largest mapped-pose difference to the oracle chain: %.3g m, %.3g (quaternion)" % worst)


def test_inputs_are_only_read_during_the_call():
    import torch
    sensor, raw, _ = _drive("vlp16", 4)
    ch = Chain(sensor, True, io_ratio=1)
    for sw in raw[:3]:
        ch.step(sw)
    before = {w: ch.po.cloud(w) for w in WHICH}
    t = torch.from_numpy(raw[3]).cuda()
    ch.pp.process_device(t.data_ptr(), t.shape[0])              # the producer moves on to the next sweep
    ch.pp.sizes()
    for w in WHICH:
        assert before[w].shape[0] > 0 and np.array_equal(ch.po.cloud(w), before[w]), w


def test_pass_through_feeds_the_estimator():
    """After /enable_odom false the odometry's last_surf cloud is stage A's less-flat cloud: handing it to the estimator on the
    device gives the same window as handing it stage A's cloud directly."""
    import torch
    from lio_mapping_b200 import estimator, ops, scenario
    from lio_mapping_b200.point_odometry import PointOdometry
    from lio_mapping_b200.point_processor import PointProcessor
    W = 4
    scn = scenario.Scenario("vlp16", n_total=W + 3)
    sensor = scn.sensor
    pp = PointProcessor(sensor.lower_deg, sensor.upper_deg, sensor.rings, max_points=max(s.shape[0] for s in scn.raw))
    cfg = dict(scenario.EST_CFG["vlp16"], odom_max_iterations=1)
    ests = [estimator.Estimator(window_size=W, opt_window_size=W, max_frame_points=1 << 15, max_scan_points=1 << 16, **cfg) for _ in range(2)]

    def surf_ds(k):
        pp.SetInputCloud(scn.raw[k]); pp.Process()
        return ops.voxel_grid(pp.cloud("surface_points_less_flat"), 0.4)

    for e in ests:
        scenario.warm_start(e, scn, W, surf_ds, lambda a, g: estimator.Pim(a, g, np.zeros(3), np.zeros(3), acc_n=0.2, gyr_n=0.02))
    po = PointOdometry(0.1, 2, 25)
    po.EnableOdom(False)
    for k in range(W, W + 2):
        t = torch.from_numpy(np.ascontiguousarray(scn.raw[k], np.float32)).cuda()
        pp.process_device(t.data_ptr(), t.shape[0])
        po.process_device(pp)
        p, n = po.cloud_dev("last_surf")
        scenario.feed_imu(ests[0], scn, k); ests[0].process_scan_dev(p, n, 1 << 16)
        scenario.feed_imu(ests[1], scn, k); ests[1].process_scan_dev(pp.cloud_dev("surface_points_less_flat"), pp.count_dev("surface_points_less_flat"), 1 << 16)
        assert np.array_equal(ests[0].states(), ests[1].states()), k


def test_transfer_bound_of_one_call():
    """A _dev odometry call: one synchronisation and under 1 KiB each way.  A _dev mapping call: at most 256 KiB of copies whatever
    the point count, and at most 4 synchronisations when it re-allocates no workspace.  Growing a cube segment is stream-ordered
    and costs none, so over a drive that grows the map every call stays within 4 + the two workspace re-allocations (scan-to-map,
    re-filter); a repeat of the last call, which grows nothing, stays within 4."""
    sensor, raw, _ = _drive("hdl64", 8)
    dev, host = Chain(sensor, True), Chain(sensor, False)
    for f, sw in enumerate(raw):
        a = dev.step(sw); host.step(sw)
        so = dev.po.stats()
        assert so["syncs"] <= 1 and so["h2d_bytes"] <= 1024 and so["d2h_bytes"] <= 1024, (f, so)
        ho = host.po.stats()
        given = 16 * sum(host.pp.sizes()[k] for k in PP_NAMES)
        assert ho["h2d_bytes"] >= given, (f, ho, given)
        if a["info"]["published"]:
            sm, hm = dev.pm.stats(), host.pm.stats()
            n_in = dev.po.cloud_size("last_corner") + dev.po.cloud_size("last_surf")
            assert hm["h2d_bytes"] >= 16 * n_in, (f, hm)
            assert sm["h2d_bytes"] + sm["d2h_bytes"] <= 256 * 1024, (f, sm)
            assert sm["syncs"] <= 4 + 2, (f, sm)
    for _ in range(2):   # the last sweep's clouds again, at the same pose
        dev.pm.process_device(dev.po, a["ts"])
    sm = dev.pm.stats()
    assert sm["syncs"] <= 4 and sm["h2d_bytes"] + sm["d2h_bytes"] <= 256 * 1024, sm


def test_arguments():
    import torch
    from lio_mapping_b200 import _lib
    from lio_mapping_b200.point_mapping import PointMapping
    from lio_mapping_b200.point_odometry import PointOdometry
    sensor, raw, _ = _drive("vlp16", 3)
    ch = Chain(sensor, True, io_ratio=1)
    ch.step(raw[0])
    L = _lib.lib()
    import ctypes as C
    ts = np.zeros(7, np.float32); te = np.zeros(7, np.float32); info = np.zeros(4, np.int32)
    clouds = (_lib.DevCloud * 5)()
    for k, name in enumerate(PP_NAMES):
        clouds[k] = _lib.DevCloud(ch.pp.cloud_dev(name), ch.pp.count_dev(name), 64)
    bad = (_lib.DevCloud * 5)(*clouds)
    bad[2] = _lib.DevCloud(None, ch.pp.count_dev(PP_NAMES[2]), 64)
    assert L.lio_po_process_dev(ch.po.h, bad, ts, te, info) == -2                      # NULL cloud with n_max > 0
    bad = (_lib.DevCloud * 5)(*clouds)
    bad[1] = _lib.DevCloud(ch.pp.cloud_dev(PP_NAMES[1]), ch.pp.count_dev(PP_NAMES[1]), (1 << 17) + 1)
    assert L.lio_po_process_dev(ch.po.h, bad, ts, te, info) == -3                      # n_max above the capacity
    tobe = np.zeros(7, np.float32); info3 = np.zeros(3, np.int32)
    c = _lib.DevCloud(None, None, 5)
    assert L.lio_pm_process_dev(ch.pm.h, C.byref(c), C.byref(c), ts, tobe, info3) == -2
    c = _lib.DevCloud(ch.pp.cloud_dev(PP_NAMES[1]), ch.pp.count_dev(PP_NAMES[1]), (1 << 17) + 1)
    assert L.lio_pm_process_dev(ch.pm.h, C.byref(c), C.byref(c), ts, tobe, info3) == -3

    # after the refused calls the contexts behave like fresh ones on the rest of the drive
    fresh = Chain(sensor, True, io_ratio=1)
    fresh.step(raw[0])
    for sw in raw[1:]:
        a, b = ch.step(sw), fresh.step(sw)
        assert np.array_equal(a["ts"], b["ts"]) and np.array_equal(a["tobe"], b["tobe"]) and a["info3"] == b["info3"]

    # a device count above n_max is clamped: the result equals the host call on the first n_max points
    pp = ch.pp
    t = torch.from_numpy(raw[2]).cuda()
    pp.process_device(t.data_ptr(), t.shape[0])
    host = {k: pp.cloud(k) for k in PP_NAMES}
    n_max = [max(1, host[k].shape[0] // 2) for k in PP_NAMES]
    pd, ph = PointOdometry(0.1, 1, 25), PointOdometry(0.1, 1, 25)
    for _ in range(2):
        a = pd.process_device(pp, n_max=n_max)
        b = ph.Process(*[host[k][:n_max[i]] for i, k in enumerate(PP_NAMES)])
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and a[2] == b[2]
        for w in WHICH:
            assert np.array_equal(pd.cloud(w), ph.cloud(w)), w
    md, mh = PointMapping(), PointMapping()
    lc = host["corner_points_less_sharp"]; lf = host["surface_points_less_flat"]
    nc, ns = max(1, lc.shape[0] // 3), max(1, lf.shape[0] // 3)
    tf = np.array([0, 0, 0, 1, 0, 0, 0], np.float32)
    a = md.process_dev_clouds((pp.cloud_dev(PP_NAMES[1]), pp.count_dev(PP_NAMES[1]), nc), (pp.cloud_dev(PP_NAMES[3]), pp.count_dev(PP_NAMES[3]), ns), tf)
    b = mh.Process(lc[:nc], lf[:ns], tf)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]
    _assert_maps_equal(_cubes(md), _cubes(mh), "clamped")


def test_refilter_workspace_grows_with_the_cubes(oracle):
    """A cube that outgrows max_points after the insert: the per-cube VoxelGrid workspace grows before anything moves, every call
    succeeds and the map follows the oracle (the first call bit for bit)."""
    from lio_mapping_b200.point_mapping import PointMapping
    from tests.test_point_mapping_gpu import _frames
    corner, surf, _, tf_true = _frames(oracle, "vlp16", 1)[0]
    max_points = 1024
    # one sweep fed in chunks of at most max_points points at the true pose: the cubes accumulate the whole sweep
    chunks = [(corner[i * 64:(i + 1) * 64], surf[i * max_points:(i + 1) * max_points]) for i in range((surf.shape[0] + max_points - 1) // max_points)]
    pg = PointMapping(max_points=max_points)
    po = oracle.PointMappingOracle()
    for f, (c, s) in enumerate(chunks):
        tg, ig = pg.Process(c, s, tf_true)
        to, io = po.process(c, s, tf_true)
        assert pg.centre() == po.centre()
        if f == 0:
            assert ig == io and np.array_equal(tg, to)
            for which in ("corner", "surf"):
                so = po.cube_sizes(which)
                assert np.array_equal(so, pg.cube_sizes(which))
                for idx in np.nonzero(so)[0]:
                    assert np.array_equal(pg.cube(idx, which), po.cube(idx, which)), (which, idx)
        else:
            assert abs(ig["iterations"] - io["iterations"]) <= 1
            assert np.abs(tg[4:] - to[4:]).max() <= 2e-4 and np.abs(tg[:4] - to[:4]).max() <= 2e-5, (f, tg, to)
            for which in ("corner", "surf"):
                so, sg = po.cube_sizes(which), pg.cube_sizes(which)
                assert np.array_equal(so > 0, sg > 0)
                assert np.abs(so - sg).sum() <= 2 + 0.005 * so.sum()
    assert pg.cube_sizes("surf").max() > max_points
