"""BASELINE.json full sizes (configs 3 and 5) through size-independent properties and thin-slab oracle
comparisons: the 512^3 pillar map for the ESDF, a 4096-trajectory batch on office3 for the cost."""
import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests.helpers import assert_esdf_exact, make_sdf_map, orc_grid

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pillar(fuel):
    g, inflate = W.pillar_map("V1")
    tri = np.where(inflate == 1, W.OCCUPIED, W.FREE).astype(np.uint8)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    yield g, inflate, tri, m
    m.close()


def test_esdf_512_properties(fuel, pillar):
    g, inflate, tri, m = pillar
    m.updateESDF3d()
    d = m.download().copy()
    assert np.all(np.isfinite(d))
    assert np.all(d[inflate == 1] == 0.0) and np.all(d[inflate == 0] >= np.float32(g.res) * (1 - 1e-6))
    # an exact Euclidean distance field is 1-Lipschitz: neighbours differ by at most one voxel
    tol = g.res * (1 + 1e-5)
    for ax in range(3):
        assert np.max(np.abs(np.diff(d, axis=ax))) <= tol
    # d^2/res^2 is an integer (sum of three squares) everywhere
    q = (d.astype(np.float64) / g.res) ** 2
    assert np.max(np.abs(q - np.rint(q))) < 2e-3 * np.maximum(1.0, q.max() ** 0.5)
    # idempotence
    m.updateESDF3d()
    assert np.array_equal(m.download(), d)


def test_esdf_512_slab_matches_oracle(fuel, orc, pillar):
    """box = full x and y extent (512 x 512), 24 planes in z: the same box semantics on both sides."""
    g, inflate, tri, m = pillar
    bmin, bmax = np.array([0, 0, 200]), np.array([511, 511, 223])
    m.local_bound_min_, m.local_bound_max_ = bmin, bmax
    m.updateESDF3d()
    d = m.download()[:, :, 200:224].copy()
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, bmin, bmax, True, False, threads=16)[:, :, 200:224]
    assert_esdf_exact(d, ref, g.res)
    m.local_bound_min_, m.local_bound_max_ = np.zeros(3, dtype=np.int32), np.array(g.n) - 1


@pytest.mark.parametrize("variant", ["V1", "V0"])
def test_esdf_512_full_box_matches_oracle(fuel, orc, variant):
    """The update bench.py times as roofline_esdf512 (box = the whole 512^3 map), voxel for voxel against the
    oracle: V1 (tiled, every line has sites) and V0 (file as is: most lines have none -> the +inf sentinel)."""
    g, inflate = W.pillar_map(variant)
    tri = np.where(inflate == 1, W.OCCUPIED, W.FREE).astype(np.uint8)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    d = m.download().copy()
    m.close()
    ref = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(g.n) - 1, True, False, threads=16)
    assert_esdf_exact(d, ref, g.res)
    del ref


def test_frontier_512_matches_oracle(fuel, orc):
    """BASELINE config 3, second half: the frontier sweep + clustering + split over the 512^3 pillar map (the large
    multi-kernel path), bit-exact against the oracle: cluster count, order, cell sets, frontier_flag_."""
    g, inflate = W.pillar_map("V1")
    tri = W.known_region(g, inflate, seed=7, n_poses=64, radius=4.5)
    m = fuel.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max)
    m.occupancy_buffer_inflate_[...] = inflate
    m.setOccupancyBuffer(tristate=tri)
    m.upload()
    env = fuel.EDTEnvironment()
    env.setMap(m)
    ff = fuel.FrontierFinder(env)
    out = ff.search_box(g.origin, g.map_max)
    fl = ff.download_flags()
    allc = np.concatenate([c.cells_addr_ for c in out])
    assert len(out) > 100 and np.unique(allc).size == allc.size and np.all(fl.ravel()[allc] == 1)
    assert ff.search_box(g.origin, g.map_max) == [] and np.array_equal(ff.download_flags(), fl)  # idempotent
    og = orc_grid(orc, g)
    ofl = np.zeros(g.n, dtype=np.int8)
    ref = orc.frontier_search(og, tri, ofl, g.origin, g.map_max, orc.frontier_params(cell_order=1))
    assert len(ref) == len(out)
    for a, b in zip(out, ref):
        assert np.array_equal(a.cells_addr_, b["addr"])
        assert np.array_equal(a.filtered_cells_, b["filtered"])  # third-party VoxelGrid restated on both sides (unpinned)
        assert np.allclose(a.average_, b["average"], rtol=0, atol=1e-12)
    assert np.array_equal(fl, ofl)
    m.close()


def test_bspline_4096_batch_office3(fuel, orc):
    """BASELINE config 5: office3.pcd 200x300x40, 4096 trajectories."""
    g, inflate = W.office3_map()
    tri = W.office_known(g, inflate)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    env = fuel.EDTEnvironment()
    env.setMap(m)
    opt = fuel.BsplineOptimizer()
    opt.setEnvironment(env)
    B, N = 4096, 20
    tr = W.make_trajectories(g, inflate, B=B, n_pts=N, seed=100)
    mask = opt.NORMAL_PHASE | opt.MINTIME
    x = W.pack_x(tr["ctrl"], tr["dt"])
    f, gr = opt.combineCostBatch(x, opt.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"]), N, mask)
    og = orc_grid(orc, g)
    d64 = orc.update_esdf3d(og, inflate, tri, [0, 0, 0], np.array(g.n) - 1, True, False, threads=16)
    tcs = orc.traj_consts(B)
    for b in range(B):
        orc.fill_traj_const(tcs[b], tr["pt_dist"][b], tr["dt"][b], tr["start"][b], tr["end_pos"][b][None, :])
    fr, grr = orc.combine_cost_batch(og, d64, orc.opt_params(), tcs, N, mask, x, threads=16)
    assert np.all(np.abs(f - fr) <= 1e-4 * np.abs(fr))
    sc = np.max(np.abs(grr), axis=1, keepdims=True)
    assert np.all(np.abs(gr - grr) <= 1e-4 * np.maximum(np.abs(grr), 1e-3 * sc))
    m.close()
