"""Occupancy-fusion parity: fuelgpu_map_input_point_cloud (C ABI) vs the CPU oracle of
SDFMap::inputPointCloud (plan_env/src/sdf_map.cpp:259-345).  Log-odds are fp64 sums of the same constants
in both, so the bar is bit-exact: log-odds, tri-state, local bounds and the updated box."""
import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests import ref_pins as RP
from tests.helpers import orc_grid, sdf_map_geometry

pytestmark = pytest.mark.gpu


def pair(fuel, orc, g, **kw):
    m = fuel.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max)
    m.setFusionParams(**kw)
    f = orc.Fusion(orc_grid(orc, g), orc.fusion_params(**kw))
    return m, f


def check_frame(m, f, pts, cam):
    lo, hi = f.input_point_cloud(pts, cam)
    m.inputPointCloud(pts, pts.shape[0], cam)
    got = m.getLogOdds().reshape(-1)
    assert np.array_equal(got, f.logodds), "log-odds differ in %d voxels" % int((got != f.logodds).sum())
    if pts.shape[0]:
        assert np.array_equal(m.local_bound_min_, lo) and np.array_equal(m.local_bound_max_, hi)
    tri = np.empty(m.shape, np.uint8)
    inf = np.empty(m.shape, np.int8)
    from fuel_b200._lib import check, lib, ptr
    check(lib().fuelgpu_map_download_occupancy(m._h, ptr(inf), ptr(tri)), m._h)
    assert np.array_equal(tri.reshape(-1), f.tristate())


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_clouds(fuel, orc, seed):
    """Random clouds around a random camera: in-map hits, over-range points, points outside the map,
    points under z = 0.2, duplicates in one voxel, exact-integer coordinates."""
    rng = np.random.default_rng(seed)
    g = W.Grid((70, 60, 30), (-3.5, -3.0, -0.5), 0.1)
    m, f = pair(fuel, orc, g, max_ray_length=2.5)
    for frame in range(4):
        cam = np.array([rng.uniform(-2, 2), rng.uniform(-2, 2), rng.uniform(0.5, 2.0)])
        pts = cam + rng.normal(size=(3000, 3)) * np.array([2.0, 2.0, 0.8])
        pts[:50] = np.round(pts[:50])                      # coordinates on voxel faces
        pts[50:100] = pts[50]                              # many points in one voxel
        pts[100:130] *= 8.0                                # far outside the map
        check_frame(m, f, pts.astype(np.float32), cam)
    lo, hi = f.updated_box(reset=True)
    glo, ghi = m.getUpdatedBox(reset=True)
    assert np.array_equal(lo, glo) and np.array_equal(hi, ghi)
    cam = np.array([0.3, 0.1, 1.0])
    pts = (cam + rng.normal(size=(200, 3))).astype(np.float32)
    check_frame(m, f, pts, cam)
    assert np.array_equal(np.concatenate(f.updated_box()), np.concatenate(m.getUpdatedBox()))
    m.close()


def test_pcl_point_stride(fuel, orc):
    """pcl::PointXYZ is 16 bytes (xyz + padding): stride 4 must give the same map as packed xyz."""
    rng = np.random.default_rng(9)
    g = W.Grid((40, 40, 20), (-2.0, -2.0, -0.5), 0.1)
    m, f = pair(fuel, orc, g)
    cam = np.array([0.1, -0.2, 0.8])
    pts = (cam + rng.normal(size=(500, 3))).astype(np.float32)
    f.input_point_cloud(pts, cam)
    p4 = np.full((500, 4), np.nan, np.float32)
    p4[:, :3] = pts
    m.inputPointCloud(p4, 500, cam)
    assert np.array_equal(m.getLogOdds().reshape(-1), f.logodds)
    m.close()


def test_empty_cloud(fuel, orc):
    g = W.Grid((20, 20, 20), (-1.0, -1.0, -0.5), 0.1)
    m, f = pair(fuel, orc, g)
    m.inputPointCloud(np.zeros((0, 3), np.float32), 0, np.array([0.0, 0.0, 0.5]))
    check_frame(m, f, np.array([[0.5, 0.2, 0.7]], np.float32), np.array([0.0, 0.0, 0.5]))
    m.close()


def test_office_depth_frames_then_inflate_and_esdf(fuel, orc):
    """The MapROS::depthPoseCallback chain (map_ros.cpp:121-154 + updateESDFCallback :105-119) on the office map:
    inputPointCloud -> clearAndInflateLocalMap -> updateESDF3d, every stage on the device, against the oracle chain."""
    g, inflate_truth = W.office_map()
    og = orc_grid(orc, g)
    m, f = pair(fuel, orc, g)
    tri_o = None
    inf_o = np.zeros(g.n, np.int8)
    poses = [((0.0, 0.0, 1.0), 0.0), ((0.3, 0.1, 1.0), 0.8), ((0.8, 0.4, 1.1), 1.7), ((1.0, 1.0, 1.2), 3.0)]
    for cam, yaw in poses:
        cam = np.array(cam)
        pts = W.depth_frame(g, inflate_truth, cam, yaw)
        check_frame(m, f, pts, cam)
        lo, hi = m.local_bound_min_.copy(), m.local_bound_max_.copy()
        # oracle chain
        tri_o = f.tristate().reshape(g.n).copy()
        orc.clear_and_inflate(og, tri_o, inf_o, lo, hi, 2, -1)
        ref = orc.update_esdf3d(og, inf_o, tri_o, lo, hi, False, False)
        # device chain
        m.clearAndInflateLocalMap(obstacles_inflation=0.199)
        assert np.array_equal(m.occupancy_buffer_inflate_, inf_o)
        m.updateESDF3d()
        got = m.download(lo, hi).copy()
        sl = tuple(slice(lo[i], hi[i] + 1) for i in range(3))
        r, q = ref[sl], got[sl]
        fin = r < 1e150
        assert np.array_equal(np.isinf(q), ~fin)
        assert np.all(np.abs(q[fin] - r[fin]) <= 1e-4 * np.abs(r[fin]))
    m.close()


def test_depth_image_path(fuel, orc):
    """fuelgpu_map_input_depth_image == oracle proessDepthImage -> inputPointCloud, bit for bit."""
    g, inflate_truth = W.office_map()
    m, f = pair(fuel, orc, g)
    cp = orc.camera_params()
    rng = np.random.default_rng(4)
    for k, (cam, yaw, pitch) in enumerate([((0.0, 0.0, 1.0), 0.3, 0.0), ((0.4, 0.2, 1.2), 1.1, -0.2), ((0.4, 0.2, 1.2), 2.5, 0.15)]):
        cam = np.array(cam)
        img, R = W.depth_image(g, inflate_truth, cam, yaw, pitch)
        if k == 1:   # sensor drop-outs and too-close returns
            img[rng.integers(0, 480, 4000), rng.integers(0, 640, 4000)] = 0
            img[rng.integers(0, 480, 3000), rng.integers(0, 640, 3000)] = 150
        pts = orc.process_depth_image(cp, img, R, cam)
        lo, hi = f.input_point_cloud(pts, cam)
        cnt = m.inputDepthImage(img, R, cam)
        assert cnt == pts.shape[0]
        got = m.getLogOdds().reshape(-1)
        assert np.array_equal(got, f.logodds), "log-odds differ in %d voxels" % int((got != f.logodds).sum())
        assert np.array_equal(m.local_bound_min_, lo) and np.array_equal(m.local_bound_max_, hi)
    assert np.array_equal(np.concatenate(f.updated_box()), np.concatenate(m.getUpdatedBox()))
    # an all-too-close image projects nothing and changes nothing
    before = m.getLogOdds()
    assert m.inputDepthImage(np.full((480, 640), 50, np.uint16), np.eye(3), np.array([0.0, 0.0, 1.0])) == 0
    assert np.array_equal(before, m.getLogOdds())
    m.close()


CEILING_MAP = dict(resolution=0.1, map_size_x=8.0, map_size_y=6.0, map_size_z=3.0, ground_height=-0.5, obstacles_inflation=0.199,
                   local_bound_inflate=0.5, local_map_margin=50, default_dist=0.0, optimistic=0, signed_dist=0, p_hit=0.65,
                   p_miss=0.35, p_min=0.12, p_max=0.90, p_occ=0.80, max_ray_length=4.5, virtual_ceil_height=1.5)


def _ceiling_clouds():
    """rays that go up through the ceiling plane (misses on ceiling voxels) and hits below it"""
    ceil_h = CEILING_MAP["virtual_ceil_height"]
    rng = np.random.default_rng(21)
    for cycle in range(4):
        cam = np.array([rng.uniform(-2, 2), rng.uniform(-1.5, 1.5), rng.uniform(0.3, 1.2)])
        pts = cam + rng.normal(size=(4000, 3)) * np.array([2.0, 2.0, 1.5])
        pts[:1500, 2] = np.abs(pts[:1500, 2]) + ceil_h + 0.3
        yield cycle, cam, pts.astype(np.float32)


def ref_virtual_ceiling():
    """the reference's side, run by tools/make_ref_pins.py: its own sdf_map.cpp (oracle/_ref)"""
    import oracle
    ref = oracle.RefSDFMap(**CEILING_MAP)
    out = {}
    for cycle, cam, pts in _ceiling_clouds():
        ref.input_point_cloud(pts, cam)
        out["bound%d" % cycle] = np.concatenate(ref.get_local_bound())
        ref.clear_and_inflate()
        out["logodds%d" % cycle] = ref.occupancy.copy()
        out["inflate%d" % cycle] = ref.inflate.copy()
    ref.close()
    return out


def test_virtual_ceiling_survives_later_frames(fuel):
    """Several fuse -> clearAndInflateLocalMap cycles with a virtual ceiling (virtual_ceil_height 1.5, as the
    kino/topo launch files set 2.5-3.2) against the reference's own sdf_map.cpp (stored outputs, tests/ref_pins.py):
    the reference writes occupancy_buffer_[ceiling] = clamp_max_log_ (sdf_map.cpp:462-470), so the ceiling voxels stay
    occupied when later frames register misses on them; log-odds, tri-state and inflation must stay bit-exact after
    every cycle."""
    P = RP.load("test_gpu_fusion", "virtual_ceiling", REF_PINS)
    n, origin, _ = sdf_map_geometry(CEILING_MAP)
    g = W.Grid(n, tuple(origin), CEILING_MAP["resolution"])
    m = fuel.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max)
    m.setFusionParams(max_ray_length=4.5)
    for cycle, cam, pts in _ceiling_clouds():
        m.inputPointCloud(pts, pts.shape[0], cam)
        P.check("bound%d" % cycle, np.concatenate([m.local_bound_min_, m.local_bound_max_]), "cycle %d" % cycle)
        m.clearAndInflateLocalMap(obstacles_inflation=CEILING_MAP["obstacles_inflation"],
                                  virtual_ceil_height=CEILING_MAP["virtual_ceil_height"])
        P.check("logodds%d" % cycle, m.getLogOdds().reshape(-1), "cycle %d" % cycle)
        P.check("inflate%d" % cycle, m.occupancy_buffer_inflate_.reshape(-1), "cycle %d: inflation" % cycle)
    m.close()


def test_first_frame_respects_uploaded_occupancy(fuel, orc):
    """A map whose occupancy was uploaded as tri-state (setOccupancyBuffer + upload) and then receives its first fused
    frame: the device log-odds are seeded from the resident byte (UNKNOWN / FREE / OCCUPIED -> clamp_min - 0.01 /
    clamp_min / clamp_max), so one miss does not turn an uploaded OCCUPIED voxel into FREE."""
    g = W.Grid((40, 30, 20), (-2.0, -1.5, -0.5), 0.1)
    tri = np.full(g.n, W.FREE, dtype=np.uint8)
    tri[25, 15, 10] = W.OCCUPIED
    tri[:, :, 15:] = W.UNKNOWN
    m = fuel.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max)
    m.setOccupancyBuffer(tristate=tri)
    m.upload()
    m.setFusionParams(max_ray_length=4.5)
    cam = np.array([-1.0, 0.05, 0.55])
    # one ray through the occupied voxel (a miss on it), ending well behind it
    target = np.array([[1.5, 0.05, 0.55]], dtype=np.float32)
    m.inputPointCloud(target, 1, cam)
    lo = m.getLogOdds()
    lg = lambda p: np.log(p / (1 - p))  # noqa: E731
    assert lo[25, 15, 10] == lg(0.90) + lg(0.35)     # clamp_max + one miss: still above min_occupancy_log
    assert lo[0, 0, 0] == lg(0.12) and lo[0, 0, 18] == lg(0.12) - 0.01
    tri2 = np.empty(m.shape, np.uint8)
    inf = np.empty(m.shape, np.int8)
    from fuel_b200._lib import check, lib, ptr
    check(lib().fuelgpu_map_download_occupancy(m._h, ptr(inf), ptr(tri2)), m._h)
    assert tri2[25, 15, 10] == W.OCCUPIED
    m.close()


REF_PINS = {"virtual_ceiling": (ref_virtual_ceiling, [()])}
