"""The host-side mirror of FrontierFinder (fuel_b200/frontier_finder.py: the list bookkeeping of searchFrontiers /
computeFrontiersToVisit / isFrontierCovered around the device calls) against the REFERENCE's own compiled
frontier_finder.cpp over a multi-frame exploration episode.  The device calls of the mirror are replaced by the oracle
here (no GPU needed), so what is compared is exactly the host logic: which stored clusters are removed when the map
changes (haveOverlap + isFrontierChanged), removed_ids_, the dormant list, id assignment, viewpoint filtering / order.
The reference's side of the episode, ref_episode(), is recorded by tools/make_ref_pins.py into
tests/golden/ref_pins.npz (tests/ref_pins.py); the test compares the mirror with those stored lists."""
import numpy as np

import oracle as O
from fuel_b200 import workloads as W
from fuel_b200.frontier_finder import Frontier, FrontierFinder
from tests import ref_pins as RP
from tests.helpers import sdf_map_geometry, viewpoint_rows

O.build()
MODULE = "test_host_frontier_bookkeeping"

MAP = dict(resolution=0.1, map_size_x=8.0, map_size_y=6.0, map_size_z=3.0, ground_height=-0.5, obstacles_inflation=0.199,
           local_bound_inflate=0.5, local_map_margin=50, default_dist=0.0, optimistic=0, signed_dist=0, p_hit=0.65, p_miss=0.35,
           p_min=0.12, p_max=0.90, p_occ=0.80, max_ray_length=4.5, virtual_ceil_height=-10.0, box_min_x=-3.6, box_min_y=-2.6,
           box_min_z=-0.3, box_max_x=3.6, box_max_y=2.6, box_max_z=2.2)
FF = dict(cluster_min=15, cluster_size_xy=1.2, cluster_size_z=10.0, min_candidate_dist=0.75, min_candidate_clearance=0.21,
          candidate_dphi=15 * 3.1415926 / 180.0, candidate_rmax=2.5, candidate_rmin=1.5, candidate_rnum=3, down_sample=3,
          min_visib_num=6, min_view_finish_fraction=0.2)
PU = dict(top_angle=0.56125, left_angle=0.69222, right_angle=0.68901, max_dist=4.5, vis_dist=1.0)


def logit(p):
    return np.log(p / (1 - p))


class FakeMap:
    """what the mirror needs from SDFMap, without a device"""

    def __init__(self, n, res, origin):
        self.shape, self.resolution_, self.map_origin_ = n, res, origin
        self.handle = None
        self.update_min_, self.update_max_ = np.zeros(3), np.zeros(3)

    def getUpdatedBox(self, reset=False):
        return self.update_min_.copy(), self.update_max_.copy()


class OracleBackedFinder(FrontierFinder):
    """fuel_b200.FrontierFinder with every libfuelgpu call answered by the oracle (BFS cell order, like the reference)"""

    def __init__(self, fmap, g, tri_ref, inflate, **kw):
        class Env:
            sdf_map_ = fmap
        super().__init__(Env(), cluster_min=kw["cluster_min"], cluster_size_xy=kw["cluster_size_xy"], down_sample=kw["down_sample"])
        self.g, self.tri, self.inflate = g, tri_ref, inflate
        self.flag = np.zeros(fmap.shape, np.int8)

    def _changed(self, ftrs):
        return np.array([O.frontier_changed_count(self.g, self.tri, f.cells_addr_) > 0 for f in ftrs], np.uint8)

    def _clear_flags(self, addr):
        self.flag.reshape(-1)[addr] = 0

    def search_box(self, update_min, update_max):
        p = O.frontier_params(cluster_min=self.cluster_min_, cluster_size_xy=self.cluster_size_xy_, down_sample=self.down_sample_,
                              cell_order=0)
        res = O.frontier_search(self.g, self.tri, self.flag, update_min, update_max, p)
        return [Frontier(self._map, r["addr"], r["filtered"], r["average"], r["box_min"], r["box_max"]) for r in res]

    def sampleViewpointsRaw(self, ftrs):
        vp = O.view_params()
        out = [O.sample_viewpoints(self.g, self.tri, self.inflate, vp, f.average_, f.filtered_cells_) for f in ftrs]
        if not out:
            return np.zeros((0, 100, 3)), np.zeros((0, 100)), np.zeros((0, 100), np.int32)
        return np.stack([o["pos"] for o in out]), np.stack([o["yaw"] for o in out]), np.stack([o["visib"] for o in out])


def list_arrays(prefix, addrs, averages):
    """a frontier list as flat arrays: cells (BFS order) and averages"""
    return {prefix + "offsets": np.cumsum([0] + [len(a) for a in addrs]),
            prefix + "addr": np.concatenate(addrs) if addrs else np.zeros(0, np.int64),
            prefix + "average": np.reshape(averages, (-1, 3))}


def mirror_arrays(prefix, ftrs):
    return list_arrays(prefix, [f.cells_addr_ for f in ftrs], [f.average_ for f in ftrs])


def ref_arrays(prefix, ftrs):
    return list_arrays(prefix, [f["addr"] for f in ftrs], [f["average"] for f in ftrs])


# the robot reveals one ball of space per frame, moving through the room
PATH = [(18, 20, 12), (28, 24, 12), (38, 30, 13), (48, 32, 12), (58, 36, 12), (60, 22, 12), (46, 16, 12), (30, 40, 14)]
BOX = ((-3.6, -2.6, -0.3), (3.6, 2.6, 2.2))


class Episode:
    """the map state of the episode: tri-state and known inflation, updated in place frame by frame"""

    def __init__(self):
        self.n, self.origin, _ = sdf_map_geometry(MAP)
        rng = np.random.default_rng(12)
        self.inflate = (rng.random(self.n) < 0.003).astype(np.int8)
        self.XYZ = np.meshgrid(*[np.arange(k) for k in self.n], indexing="ij")
        self.tri = np.full(self.n, W.UNKNOWN, np.uint8)
        self.inf_known = np.zeros(self.n, np.int8)

    def reveal(self, k, c):
        """-> the newly known voxels and the updated box of frame k"""
        X, Y, Z = self.XYZ
        ball = ((X - c[0]) ** 2 + (Y - c[1]) ** 2 + 3.0 * (Z - c[2]) ** 2) < (11 + (k % 3)) ** 2
        newly = ball & (self.tri == W.UNKNOWN)
        self.tri[newly] = np.where(self.inflate[newly] == 1, W.OCCUPIED, W.FREE)
        self.inf_known[newly] = self.inflate[newly]
        idx = np.argwhere(newly)
        assert len(idx)
        res = MAP["resolution"]
        return newly, self.origin + idx.min(axis=0) * res, self.origin + (idx.max(axis=0) + 1) * res


def ref_episode():
    ref = O.RefSDFMap(**MAP)
    ep = Episode()
    ref.inflate[:] = 0
    ref.occupancy[:] = logit(0.12) - 0.01
    rff = O.RefFrontierFinder(ref, PU, **FF)
    occ = ref.occupancy.reshape(ref.n)
    out = {}
    for k, c in enumerate(PATH):
        newly, umin, umax = ep.reveal(k, c)
        occ[newly] = np.where(ep.inflate[newly] == 1, logit(0.90), logit(0.12))
        ref.inflate[:] = ep.inf_known.reshape(-1)
        ref.R.ref_map_set_updated_box(ref.h, O._p(umin), O._p(umax))
        # searchFrontiers(); computeFrontiersToVisit()
        out.update(ref_arrays("f%d_tmp_" % k, rff.search_frontiers()))
        out["f%d_removed" % k] = np.asarray(rff.removed_ids(), np.int64)
        out["f%d_flags" % k] = rff.flags.copy()
        visit, dormant = rff.compute_to_visit()
        out.update(ref_arrays("f%d_visit_" % k, visit))
        out.update(ref_arrays("f%d_dormant_" % k, dormant))
        out["f%d_ids" % k] = [v["id"] for v in visit]
        for i, v in enumerate(visit):
            out["f%d_vp%d" % (k, i)] = viewpoint_rows(v["view_visib"], v["view_yaw"], v["view_pos"])
    rff.close()
    ref.close()
    return out


def test_exploration_episode_matches_reference():
    P = RP.load(MODULE, "episode", REF_PINS)
    ep = Episode()
    g = O.make_grid(ep.n, MAP["resolution"], ep.origin, BOX[0], BOX[1], map_size=sdf_map_geometry(MAP)[2])
    fmap = FakeMap(ep.n, MAP["resolution"], ep.origin)
    mine = OracleBackedFinder(fmap, g, ep.tri, ep.inf_known, **FF)
    mine.setViewParams(min_visib_num=FF["min_visib_num"], min_view_finish_fraction=FF["min_view_finish_fraction"])
    total_removed = 0
    for k, c in enumerate(PATH):
        _, fmap.update_min_, fmap.update_max_ = ep.reveal(k, c)
        mine.searchFrontiers()
        for key, v in mirror_arrays("f%d_tmp_" % k, mine.tmp_frontiers_).items():
            P.check(key, v)
        P.check("f%d_removed" % k, np.asarray(mine.removed_ids_, np.int64), "removed_ids_")
        total_removed += len(mine.removed_ids_)
        P.check("f%d_flags" % k, mine.flag.reshape(-1), "frontier_flag_")
        mine.computeFrontiersToVisit()
        for key, v in mirror_arrays("f%d_visit_" % k, mine.frontiers_).items():
            P.check(key, v)
        for key, v in mirror_arrays("f%d_dormant_" % k, mine.dormant_frontiers_).items():
            P.check(key, v)
        P.check("f%d_ids" % k, [a.id_ for a in mine.frontiers_])
        for i, a in enumerate(mine.frontiers_):
            vp = a.viewpoints_
            P.check("f%d_vp%d" % (k, i), viewpoint_rows([v[2] for v in vp], [v[1] for v in vp], [v[0] for v in vp]))
            assert [v[2] for v in vp] == sorted((v[2] for v in vp), reverse=True)
    assert total_removed >= 3 and len(mine.frontiers_) >= 2   # the episode did exercise removal and survival


REF_PINS = {"episode": (ref_episode, [()])}
