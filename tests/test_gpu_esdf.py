"""ESDF parity: libfuelgpu (C ABI) vs the CPU oracle of SDFMap::updateESDF3d
(plan_env/src/sdf_map.cpp:152-241), to the exact squared voxel distance (tests.helpers.assert_esdf_exact: every
finite distance is res*sqrt(N) with N an integer, and the device's N must equal the reference's wherever N <= 2^20)."""
import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests.helpers import ESDF_SENTINEL as SENTINEL
from tests.helpers import assert_esdf_exact, make_sdf_map, orc_grid, random_scene

pytestmark = pytest.mark.gpu


def compare(dist_gpu, dist_ref, res, box=None):
    assert_esdf_exact(dist_gpu, dist_ref, res, box)


@pytest.mark.parametrize("n,seed", [((17, 23, 11), 1), ((64, 48, 40), 2), ((33, 1, 7), 3), ((1, 1, 1), 4),
                                    ((40, 40, 70), 5)])
@pytest.mark.parametrize("optimistic", [True, False])
def test_random_full_box(fuel, orc, n, seed, optimistic):
    g = W.Grid(n, (-1.0, -2.0, -0.5), 0.1)
    inflate, tri = random_scene(n, seed)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=optimistic)
    m.updateESDF3d()
    got = m.download().copy()
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(n) - 1, optimistic, False)
    compare(got, ref, g.res)
    m.close()


def test_signed(fuel, orc):
    n = (40, 36, 28)
    g = W.Grid(n, (0, 0, 0), 0.1)
    rng = np.random.default_rng(9)
    inflate = np.zeros(n, dtype=np.int8)
    for _ in range(5):
        c = rng.integers(4, 24, 3)
        inflate[c[0]:c[0] + 6, c[1]:c[1] + 7, c[2]:c[2] + 4] = 1
    tri = np.full(n, W.FREE, dtype=np.uint8)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True, signed=True)
    m.updateESDF3d()
    got = m.download().copy()
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(n) - 1, True, True)
    assert np.any(ref < 0)
    assert_esdf_exact(got, ref, g.res, signed=True)
    m.close()


def test_local_box_ignores_outside_sites(fuel, orc):
    """SURVEY H2: the transform is restricted to [local_bound_min_, local_bound_max_] and voxels
    outside keep their previous value."""
    n = (48, 40, 32)
    g = W.Grid(n, (-2.4, -2.0, -1.0), 0.1)
    inflate, tri = random_scene(n, 11, p_site=0.01, p_unknown=0)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()  # whole map first
    full = m.download().copy()
    bmin, bmax = np.array([5, 7, 3]), np.array([30, 33, 20])
    # change occupancy inside the box only, re-run on the box
    inflate2 = inflate.copy()
    inflate2[10:14, 10:12, 5:9] = 1
    m.occupancy_buffer_inflate_[...] = inflate2
    m.upload()
    m.local_bound_min_, m.local_bound_max_ = bmin, bmax
    m.updateESDF3d()
    got = m.download().copy()
    ref_full = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(n) - 1, True, False)
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate2, tri, bmin, bmax, True, False, dist=ref_full.copy())
    compare(got, ref, g.res, (bmin, bmax))
    outside = np.ones(n, dtype=bool)
    outside[bmin[0]:bmax[0] + 1, bmin[1]:bmax[1] + 1, bmin[2]:bmax[2] + 1] = False
    assert np.array_equal(got[outside], full[outside])
    m.close()


def test_empty_box_is_sentinel(fuel, orc):
    n = (12, 9, 10)
    g = W.Grid(n, (0, 0, 0), 0.1)
    inflate = np.zeros(n, dtype=np.int8)
    tri = np.full(n, W.FREE, dtype=np.uint8)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    got = m.download()
    assert np.all(np.isinf(got))
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(n) - 1, True, False)
    assert np.all(ref > SENTINEL)
    d64 = m.download(dtype=np.float64)
    assert np.allclose(d64, ref, rtol=1e-12)  # f64 download restores the reference's finite value
    m.close()


def test_office_fixture(fuel, orc):
    """BASELINE config 1/2 map: office.pcd on 200x120x40, both ESDF variants."""
    g, inflate = W.office_map()
    tri = W.office_known(g, inflate)
    for optimistic in (True, False):
        m = make_sdf_map(fuel, g, inflate, tri, optimistic=optimistic)
        m.updateESDF3d()
        got = m.download().copy()
        ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(g.n) - 1, optimistic, False,
                                threads=8)
        compare(got, ref, g.res)
        m.close()


def test_sample_matches_getDistWithGrad(fuel, orc):
    """SDFMap::getDistWithGrad (sdf_map.cpp:497-536) incl. the H6 edge cases: out-of-map
    positions, stencils poking outside the map (-1 samples), the 1e-4 isInMap margin."""
    g, inflate = W.office_map()
    tri = W.office_known(g, inflate)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    d32 = m.download().copy()
    rng = np.random.default_rng(5)
    pos = rng.uniform(g.origin - 0.3, g.map_max + 0.3, size=(20000, 3))
    edge = rng.uniform(g.origin, g.map_max, size=(3000, 3))
    edge[:1000, 0] = g.origin[0] + rng.uniform(0, 0.06, 1000)
    edge[1000:2000, 2] = g.map_max[2] - rng.uniform(0, 0.06, 1000)
    edge[2000:, 1] = g.origin[1] + 1e-4 + rng.uniform(-2e-5, 2e-5, 1000)
    pos = np.concatenate([pos, edge])
    dg, gg = m.getDistWithGrad(pos)
    # the oracle samples the same fp32 field widened to fp64: the sampler itself is then exact
    dr, gr = orc.dist_with_grad(orc_grid(orc, g), d32.astype(np.float64), pos)
    assert np.allclose(dg, dr, rtol=1e-12, atol=1e-12)
    assert np.allclose(gg, gr, rtol=1e-12, atol=1e-10)
    m.close()


@pytest.mark.parametrize("n", [(1024, 6, 5), (5, 1024, 6), (6, 5, 1024), (1024, 3, 1024)])
def test_maximum_axis_extent(fuel, orc, n):
    """1024 voxels per axis is the ABI limit (hull entries pack v in 10 bits, h in 22): distances up to
    sqrt(2*1023^2 + ...) voxels must still be exact."""
    g = W.Grid(n, (0, 0, 0), 0.1)
    inflate = np.zeros(n, dtype=np.int8)
    inflate[0, 0, 0] = 1
    inflate[n[0] - 1, n[1] - 1, n[2] // 2] = 1
    tri = np.full(n, W.FREE, dtype=np.uint8)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    got = m.download().copy()
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(n) - 1, True, False, threads=8)
    compare(got, ref, g.res)
    m.close()


@pytest.mark.parametrize("n,p_site", [((700, 40, 33), 0.004), ((37, 1000, 64), 0.002), ((600, 520, 32), 0.0005),
                                      ((1024, 70, 32), 0.02), ((513, 545, 40), 0.3)])
def test_long_lines_cluster_tiles(fuel, orc, n, p_site):
    """Lines of 513..1024 samples: the tile is shared by the two CTAs of a cluster and the hulls of the two halves are
    joined over distributed shared memory.  Dense and sparse hulls, partial last bands, then a box that starts off the
    grid origin (box-relative rows)."""
    g = W.Grid(n, (0.3, -1.0, 0.0), 0.1)
    inflate, tri = random_scene(n, 1000 + n[0], p_site=p_site, p_unknown=0.2, blobs=5)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    got = m.download().copy()
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(n) - 1, True, False, threads=16)
    compare(got, ref, g.res)
    lo = np.array([3, 2, 1])
    hi = np.array(n) - np.array([2, 4, 1])
    m.local_bound_min_, m.local_bound_max_ = lo.copy(), hi.copy()
    m.updateESDF3d()
    got2 = m.download().copy()
    ref2 = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, lo, hi, True, False, dist=ref.copy(), threads=16)
    compare(got2, ref2, g.res)
    m.close()


def test_rejects_bad_arguments(fuel):
    with pytest.raises(fuel.FuelGpuError):
        fuel.SDFMap((1025, 4, 4), 0.1, (0, 0, 0))  # beyond the 1024-per-axis limit
    with pytest.raises(fuel.FuelGpuError):
        fuel.SDFMap((8, 8, 8), -0.1, (0, 0, 0))
    m = fuel.SDFMap((8, 8, 8), 0.1, (0, 0, 0))
    m.local_bound_min_, m.local_bound_max_ = np.array([0, 0, 0]), np.array([8, 7, 7])  # outside the map
    with pytest.raises(fuel.FuelGpuError):
        m.updateESDF3d()
    m.local_bound_min_, m.local_bound_max_ = np.array([3, 3, 3]), np.array([2, 7, 7])  # empty box
    with pytest.raises(fuel.FuelGpuError):
        m.updateESDF3d()
    m.close()
