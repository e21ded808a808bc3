"""Pins the oracle against the REFERENCE's own code: plan_env/src/{raycast,sdf_map}.cpp,
bspline_opt/src/bspline_optimizer.cpp and active_perception/src/{frontier_finder,perception_utils}.cpp compiled
UNMODIFIED into oracle/_ref/libfuel_ref.so (oracle/Makefile) against interface stand-ins for the headers the image
lacks (oracle/ref_standin: Eigen small vectors/matrices, ros::NodeHandle::param, pcl containers, the NLopt API, ...).
Every comparison below is bit-exact.  Not covered, by construction: pcl::VoxelGrid and Eigen::EigenSolver
(third-party algorithms; the stand-ins call the oracle's own reconstructions) and NLopt's iterates.

Each test has a reference side, ref_<name>(), listed in REF_PINS: tools/make_ref_pins.py runs it on the reference
library and stores what it returns in tests/golden/ref_pins.npz (tests/ref_pins.py).  The tests run the oracle on the
same seeded inputs and compare with those stored outputs, so they need no reference library.  Where the reference fed
one of its own results to the next step (an ESDF under a cost evaluation, a local bound under an inflation), the
oracle's result is pinned first and then used."""
import numpy as np
import pytest

import oracle as O
from fuel_b200 import workloads as W
from tests import ref_pins as RP
from tests.helpers import sdf_map_geometry as geometry
from tests.helpers import viewpoint_rows

O.build()  # also builds oracle/_ref/libfuel_ref.so where the reference sources are present (it is git-ignored)
MODULE = "test_oracle_refpin"


def pins(name, *args):
    return RP.load(MODULE, name, REF_PINS, args)


def _cat(*arrays):
    return np.concatenate([np.ravel(np.asarray(a, dtype=np.float64)) for a in arrays])


def _intbound_args():
    rng = np.random.default_rng(0)
    s = np.concatenate([rng.uniform(-300, 300, 4000), np.round(rng.uniform(-300, 300, 500)), [0.0, -0.0, 1e-17, -1e-17]])
    ds = np.concatenate([rng.integers(-40, 41, 4000).astype(float), rng.integers(-40, 41, 504).astype(float)])
    return s, ds


def ref_intbound():
    R = O.ref_raycast()
    return {"t": [R.ref_intbound(a, b) for a, b in zip(*_intbound_args())]}


def test_intbound_matches_reference():
    L = O.lib()
    L.orc_intbound.restype = O.C.c_double
    L.orc_intbound.argtypes = [O.C.c_double, O.C.c_double]
    pins("intbound").check("t", [L.orc_intbound(a, b) for a, b in zip(*_intbound_args())])


RAY_GRIDS = [((-10.0, -6.0, -1.0), 0.1), ((-25.6, -25.6, -1.0), 0.1), ((0.3, -2.7, 0.05), 0.15)]


def _rays(origin, res):
    """Thousands of rays: random, axis-aligned, starting on voxel faces / corners, zero length, long diagonals."""
    rng = np.random.default_rng(7)
    o = np.array(origin)
    span = np.array([200, 120, 40]) * res
    for k in range(3000):
        a = o + rng.uniform(-0.1, 1.1, 3) * span
        b = o + rng.uniform(-0.1, 1.1, 3) * span
        if k % 5 == 1:
            b[rng.integers(0, 3)] = a[rng.integers(0, 3)]          # shared coordinate values
        if k % 7 == 2:
            a = o + np.round((a - o) / res) * res                  # start on voxel faces / corners
        if k % 11 == 3:
            b = a.copy()                                           # zero-length ray
        if k % 13 == 4:
            b = a + np.array([rng.uniform(-4.5, 4.5), 0.0, 0.0])   # axis-aligned
        if k % 17 == 5:
            a, b = np.float32(a).astype(np.float64), np.float32(b).astype(np.float64)  # float32 points, like pcl
        yield a, b


def _ray_outputs(fn, origin, res):
    g = O.make_grid((200, 120, 40), res, origin)
    ids = [fn(g, a, b) for a, b in _rays(origin, res)]
    return {"n": [len(i) for i in ids], "ids": np.concatenate(ids)}


def ref_rays(origin, res):
    return _ray_outputs(O.ref_raycast_ids, origin, res)


@pytest.mark.parametrize("origin,res", RAY_GRIDS)
def test_ray_traversal_matches_reference(origin, res):
    got = _ray_outputs(O.raycast_ids, origin, res)
    assert len(got["n"]) == 3000
    P = pins("rays", origin, res)
    P.check("n", got["n"], "voxels per ray")
    P.check("ids", got["ids"])


# ---------------------------------------------------------------------------------------------------------
# SDFMap: the reference's own sdf_map.cpp (updateESDF3d / fillESDF, clearAndInflateLocalMap, inputPointCloud,
# getDistWithGrad) vs the oracle restatement, bit for bit (both are fp64, no FMA contraction).
# ---------------------------------------------------------------------------------------------------------
BASE = dict(resolution=0.1, map_size_x=8.0, map_size_y=6.0, map_size_z=3.0, ground_height=-0.5, obstacles_inflation=0.199,
            local_bound_inflate=0.5, local_map_margin=50, default_dist=0.0, optimistic=0, signed_dist=0, p_hit=0.65,
            p_miss=0.35, p_min=0.12, p_max=0.90, p_occ=0.80, max_ray_length=4.5, virtual_ceil_height=-10.0)


def logit(p):
    return np.log(p / (1 - p))


def grid(params, box_mind=None, box_maxd=None):
    n, origin, size = geometry(params)
    if box_maxd is None:
        box_maxd = origin + size  # map_max_boundary_ (sdf_map.cpp:39,80-81)
    return O.make_grid(n, params["resolution"], origin, box_mind, box_maxd, map_size=size)


def wgrid(params):
    n, origin, _ = geometry(params)
    return W.Grid(n, tuple(origin), params["resolution"])


def occupancy_of(tri):
    return np.where(tri == W.UNKNOWN, logit(0.12) - 0.01, np.where(tri == W.OCCUPIED, logit(0.90), logit(0.12)))


def random_state(n, seed, p_site=0.02):
    """random inflate bits + a blobby unknown region"""
    rng = np.random.default_rng(seed)
    inflate = (rng.random(n) < p_site).astype(np.int8)
    tri = np.full(n, W.FREE, np.uint8)
    X, Y, Z = np.meshgrid(*[np.arange(k) for k in n], indexing="ij")
    for _ in range(5):
        c = rng.uniform(0, 1, 3) * np.array(n)
        r = rng.uniform(0.15, 0.4) * min(n)
        tri[((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) < r * r] = W.UNKNOWN
    tri[(inflate == 1) & (tri == W.FREE)] = W.OCCUPIED
    return inflate, tri


def load_state(ref, inflate, tri):
    """write a state straight into the reference's buffers"""
    ref.inflate[:] = inflate.reshape(-1)
    ref.occupancy[:] = occupancy_of(tri).reshape(-1)


def box_slice(lo, hi):
    return tuple(slice(lo[i], hi[i] + 1) for i in range(3))


ESDF_MODES = [(1, 0), (0, 0), (1, 1), (0, 1)]
ESDF_BOXES = [((0, 0, 0), (79, 59, 29)), ((10, 5, 3), (60, 50, 25)), ((33, 20, 7), (33, 40, 7)), ((0, 0, 0), (79, 0, 29))]


def ref_esdf(optimistic, signed):
    ref = O.RefSDFMap(**BASE)
    out = {"n": ref.n, "origin": ref.origin.copy()}
    for seed, (lo, hi) in enumerate(ESDF_BOXES):
        load_state(ref, *random_state(ref.n, seed))
        ref.distance[:] = 0.0
        ref.set_modes(optimistic, signed)
        ref.set_local_bound(lo, hi)
        ref.update_esdf3d()
        out["d%d" % seed] = ref.distance.reshape(ref.n)[box_slice(lo, hi)].copy()
    ref.close()
    return out


@pytest.mark.parametrize("optimistic,signed", ESDF_MODES)
def test_update_esdf3d_matches_reference(optimistic, signed):
    P = pins("esdf", optimistic, signed)
    n, origin, _ = geometry(BASE)
    P.check("n", n)
    P.check("origin", origin)
    assert n == (80, 60, 30)
    g = grid(BASE)
    for seed, (lo, hi) in enumerate(ESDF_BOXES):
        inflate, tri = random_state(n, seed)
        got = O.update_esdf3d(g, inflate, tri, lo, hi, optimistic, signed)
        P.check("d%d" % seed, got[box_slice(lo, hi)], "seed %d" % seed)


SENTINEL_BOX = ((5, 5, 5), (20, 20, 20))


def ref_esdf_sentinel():
    ref = O.RefSDFMap(**BASE)
    ref.inflate[:] = 0
    ref.occupancy[:] = logit(0.12)  # all free, no obstacle: every voxel keeps the DBL_MAX envelope
    ref.set_modes(1, 0)
    ref.set_local_bound(*SENTINEL_BOX)
    ref.update_esdf3d()
    out = {"d": ref.distance.reshape(ref.n)[box_slice(*SENTINEL_BOX)].copy()}
    ref.close()
    return out


def test_esdf_sentinel_when_the_box_has_no_site():
    n, _, _ = geometry(BASE)
    got = O.update_esdf3d(grid(BASE), np.zeros(n, np.int8), np.full(n, W.FREE, np.uint8), *SENTINEL_BOX, 1, 0)
    got = got[box_slice(*SENTINEL_BOX)]
    pins("esdf_sentinel").check("d", got)
    assert got.min() > 1e150


INFLATE_CEILINGS = [(-10.0,), (1.5,)]
INFLATE_BOXES = [((0, 0, 0), (79, 59, 29)), ((12, 8, 2), (70, 50, 27)), ((0, 0, 0), (3, 59, 29))]


def _inflate_case(n, seed):
    inflate, tri = random_state(n, 10 + seed, p_site=0.01)
    stale = (np.random.default_rng(seed).random(n) < 0.05).astype(np.int8)   # leftovers the call must clear in the box
    return inflate, tri, stale


def ref_clear_and_inflate(ceil_h):
    ref = O.RefSDFMap(**dict(BASE, virtual_ceil_height=ceil_h))
    out = {}
    for seed, (lo, hi) in enumerate(INFLATE_BOXES):
        inflate, tri, stale = _inflate_case(ref.n, seed)
        load_state(ref, inflate, tri)
        ref.inflate[:] = stale.reshape(-1)
        ref.set_local_bound(lo, hi)
        ref.clear_and_inflate()
        out["inflate%d" % seed] = ref.inflate.copy()
        out["tri%d" % seed] = O.tristate_from_logodds(ref.occupancy, logit(0.12), logit(0.80))
    ref.close()
    return out


@pytest.mark.parametrize("ceil_h", [c[0] for c in INFLATE_CEILINGS])
def test_clear_and_inflate_matches_reference(ceil_h):
    P = pins("clear_and_inflate", ceil_h)
    params = dict(BASE, virtual_ceil_height=ceil_h)
    n, origin, _ = geometry(params)
    g = grid(params)
    for seed, (lo, hi) in enumerate(INFLATE_BOXES):
        inflate, tri, stale = _inflate_case(n, seed)
        inf_o, tri_o = stale.copy(), tri.copy()
        ceil_id = int(np.floor((ceil_h - origin[2]) * 10.0)) if ceil_h > -0.5 else -1
        O.clear_and_inflate(g, tri_o, inf_o, lo, hi, 2, ceil_id)
        P.check("inflate%d" % seed, inf_o.reshape(-1), "seed %d" % seed)
        P.check("tri%d" % seed, tri_o.reshape(-1), "seed %d" % seed)


def _clouds():
    rng = np.random.default_rng(3)
    for frame in range(6):
        cam = np.array([rng.uniform(-3, 3), rng.uniform(-2, 2), rng.uniform(0.3, 2.0)])
        pts = cam + rng.normal(size=(4000, 3)) * np.array([2.0, 2.0, 0.8])
        pts[:60] = np.round(pts[:60])          # coordinates on voxel faces
        pts[60:120] = pts[60]                  # many points in one voxel
        pts[120:160] *= 6.0                    # far outside the map
        yield frame, cam, pts.astype(np.float32)


def ref_input_point_cloud():
    ref = O.RefSDFMap(**dict(BASE, max_ray_length=2.5))
    out = {"init": ref.occupancy.copy()}
    for frame, cam, pts in _clouds():
        ref.input_point_cloud(pts, cam)
        out["logodds%d" % frame] = ref.occupancy.copy()
        out["bound%d" % frame] = _cat(*ref.get_local_bound())
        if frame == 2:
            out["box2"] = _cat(*ref.updated_box(reset=True))
    out["box"] = _cat(*ref.updated_box())
    ref.close()
    return out


def test_input_point_cloud_matches_reference():
    P = pins("input_point_cloud")
    f = O.Fusion(grid(BASE), O.fusion_params(max_ray_length=2.5))
    P.check("init", f.logodds, "initMap fill, sdf_map.cpp:64")
    for frame, cam, pts in _clouds():
        lo, hi = f.input_point_cloud(pts, cam)
        P.check("logodds%d" % frame, f.logodds, "frame %d" % frame)
        P.check("bound%d" % frame, _cat(lo, hi), "frame %d" % frame)
        if frame == 2:
            P.check("box2", _cat(*f.updated_box(reset=True)))
    P.check("box", _cat(*f.updated_box()))


def _furnished_room():
    """the truth volume and the four depth frames of the chain below"""
    n, _, _ = geometry(BASE)
    rng = np.random.default_rng(5)
    truth = np.zeros(n, np.int8)
    truth[:, :, :6] = 1                                   # floor slab
    for _ in range(25):
        c = (rng.uniform(0.1, 0.9, 3) * np.array(n)).astype(int)
        s = rng.integers(2, 8, 3)
        truth[c[0]:c[0] + s[0], c[1]:c[1] + s[1], 6:6 + 3 * s[2]] = 1
    for k, yaw in enumerate((0.0, 1.3, 2.9, 4.4)):
        cam = np.array([0.3 * k - 0.4, 0.2 * k - 0.3, 1.0])
        yield k, cam, W.depth_frame(wgrid(BASE), truth, cam, yaw)


def ref_depth_chain():
    ref = O.RefSDFMap(**BASE)
    out = {}
    for k, cam, pts in _furnished_room():
        ref.input_point_cloud(pts, cam)
        out["logodds%d" % k] = ref.occupancy.copy()
        lo, hi = ref.get_local_bound()
        out["bound%d" % k] = _cat(lo, hi)
        ref.clear_and_inflate()
        out["inflate%d" % k] = ref.inflate.copy()
        ref.update_esdf3d()
        out["esdf%d" % k] = ref.distance.reshape(ref.n)[box_slice(lo, hi)].copy()
    ref.close()
    return out


def test_depth_frames_then_inflate_then_esdf_chain_matches_reference():
    """The MapROS::depthPoseCallback + updateESDFCallback chain on synthetic depth frames of a furnished room."""
    P = pins("depth_chain")
    n, _, _ = geometry(BASE)
    g = grid(BASE)
    f = O.Fusion(g, O.fusion_params())
    inf_o = np.zeros(n, np.int8)
    for k, cam, pts in _furnished_room():
        lo, hi = f.input_point_cloud(pts, cam)
        P.check("logodds%d" % k, f.logodds, "frame %d" % k)
        P.check("bound%d" % k, _cat(lo, hi), "frame %d" % k)
        tri = f.tristate().reshape(n).copy()
        O.clear_and_inflate(g, tri, inf_o, lo, hi, 2, -1)
        P.check("inflate%d" % k, inf_o.reshape(-1), "frame %d" % k)
        got = O.update_esdf3d(g, inf_o, tri, lo, hi, 0, 0)
        P.check("esdf%d" % k, got[box_slice(lo, hi)], "frame %d" % k)


FULL_BOX = ((0, 0, 0), (79, 59, 29))


def _dist_probe_points():
    n, origin, _ = geometry(BASE)
    rng = np.random.default_rng(1)
    pos = origin + rng.uniform(-0.05, 1.05, (3000, 3)) * np.array(n) * BASE["resolution"]
    pos[:50] = origin + np.round(rng.uniform(0, 1, (50, 3)) * np.array(n)) * BASE["resolution"]   # on voxel faces
    return pos


def ref_dist_with_grad():
    ref = O.RefSDFMap(**BASE)
    load_state(ref, *random_state(ref.n, 42, p_site=0.03))
    ref.set_modes(1, 0)
    ref.set_local_bound(*FULL_BOX)
    ref.update_esdf3d()
    d, gr = ref.dist_with_grad(_dist_probe_points())
    out = {"esdf": ref.distance.copy(), "d": d, "grad": gr}
    ref.close()
    return out


def test_dist_with_grad_matches_reference():
    P = pins("dist_with_grad")
    n, _, _ = geometry(BASE)
    inflate, tri = random_state(n, 42, p_site=0.03)
    dist = O.update_esdf3d(grid(BASE), inflate, tri, *FULL_BOX, 1, 0)
    P.check("esdf", dist.reshape(-1))
    d, gr = O.dist_with_grad(grid(BASE), dist, _dist_probe_points())
    P.check("d", d)
    P.check("grad", gr)


# ---------------------------------------------------------------------------------------------------------
# BsplineOptimizer::combineCost: the reference's own bspline_optimizer.cpp (every calc*Cost, costFunction, the
# set-up half of optimize()) vs the oracle restatement.  The NLopt stand-in evaluates the reference's objective
# at its own start point and at probe points.
# ---------------------------------------------------------------------------------------------------------
OPT = dict(ld_smooth=20.0, ld_dist=10.0, ld_feasi=2.0, ld_start=100.0, ld_end=0.5, ld_guide=1.5, ld_waypt=0.3, ld_view=0.0,
           ld_time=1.0, dist0=0.7, max_vel=2.0, max_acc=2.0, dlmin=0.0, wnl=0.0, max_iteration_num1=2, max_iteration_num2=2000,
           max_iteration_num3=200, max_iteration_num4=200, max_iteration_time1=0.0001, max_iteration_time2=0.005,
           max_iteration_time3=0.003, max_iteration_time4=0.003, algorithm1=15, algorithm2=11, bspline_degree=3)


def _opt_inputs():
    n, _, _ = geometry(BASE)
    inflate, tri = random_state(n, 77, p_site=0.004)
    return inflate, tri, W.make_trajectories(wgrid(BASE), inflate, B=12, n_pts=20, seed=31)


def _ref_opt_scene(inflate, tri, optimistic=1, **weights):
    ref = O.RefSDFMap(**BASE)
    load_state(ref, inflate, tri)
    ref.set_modes(optimistic, 0)
    ref.set_local_bound(*FULL_BOX)
    ref.update_esdf3d()
    return ref, O.RefBsplineOptimizer(ref, **dict(OPT, **weights))


@pytest.fixture(scope="module")
def opt_scene():
    inflate, tri, tr = _opt_inputs()
    dist = O.update_esdf3d(grid(BASE), inflate, tri, *FULL_BOX, 1, 0)
    return dict(tr=tr, g=grid(BASE), dist=dist, p=O.opt_params(ld_waypt=0.3))


def _probes(tr, b, mask, n_probe, seed):
    N = 20
    rng = np.random.default_rng(seed + 100 * b)
    nvar = 3 * N + (1 if mask & O.MINTIME else 0)
    x_init = np.concatenate([tr["ctrl"][b].reshape(-1), [tr["dt"][b]]])[:nvar]
    probes = x_init + rng.normal(size=(n_probe, nvar)) * 0.25
    if mask & O.MINTIME:
        probes[:, -1] = np.abs(probes[:, -1]) + 0.05
        probes[0, -1] = 0.11      # fast: velocity / acceleration limits active
    return x_init, probes


def _ref_eval(opt, tr, b, mask, end, guide=None, waypts=None, widx=None, time_lb=-1.0, n_probe=6, seed=0):
    _, probes = _probes(tr, b, mask, n_probe, seed)
    r = opt.evaluate(tr["ctrl"][b], float(tr["dt"][b]), mask, tr["start"][b], end, guide, waypts, widx, time_lb, probes)
    return {k: r[k] for k in ("f", "grad", "x0", "lb", "ub")}


def _orc_eval(sc, b, mask, end, guide=None, waypts=None, widx=None, time_lb=-1.0, n_probe=6, seed=0):
    """the oracle on the points the reference evaluates, and the start point / bounds optimize() hands to NLopt: start
    point clamped to the box shrunk by 0.1 m, bounds +-10 m clipped to it (:175-217)"""
    tr, N = sc["tr"], 20
    ctrl, dt, start = tr["ctrl"][b], float(tr["dt"][b]), tr["start"][b]
    x_init, probes = _probes(tr, b, mask, n_probe, seed)
    n, origin, _ = geometry(BASE)
    bmin, bmax = origin + 0.1, origin + np.array(n) * BASE["resolution"] - 0.1
    x0 = x_init.copy()
    x0[:3 * N] = np.clip(ctrl, bmin, bmax).reshape(-1)
    lb = np.maximum(x0[:3 * N].reshape(N, 3) - 10.0, bmin).reshape(-1)
    ub = np.minimum(x0[:3 * N].reshape(N, 3) + 10.0, bmax).reshape(-1)
    if mask & O.MINTIME:
        lb, ub = np.append(lb, 0.0), np.append(ub, 5.0)
    tc = O.traj_consts(1)
    O.fill_traj_const(tc[0], O.pt_dist(ctrl), dt, start, end, time_lb, guide, waypts, widx)
    X = np.concatenate([x0[None, :], probes])
    f = np.zeros(len(X))
    g = np.zeros((len(X), len(x0)))
    for i in range(len(X)):
        fi, gi = O.combine_cost_batch(sc["g"], sc["dist"], sc["p"], tc, N, mask, X[i:i + 1])
        f[i], g[i] = fi[0], gi[0]
    return {"f": f, "grad": g, "x0": x0, "lb": lb, "ub": ub}


def _check_eval(P, key, got):
    for k in ("x0", "lb", "ub", "f", "grad"):
        P.check(key + "_" + k, got[k])


def _exploration_cases(tr):
    for b in range(12):
        yield "b%d" % b, b, O.NORMAL_PHASE | O.MINTIME, tr["end_pos"][b][None, :], {}


def ref_exploration_objective():
    inflate, tri, tr = _opt_inputs()
    ref, opt = _ref_opt_scene(inflate, tri)
    out = {"esdf": ref.distance.copy()}
    for key, b, mask, end, kw in _exploration_cases(tr):
        out.update({key + "_" + k: v for k, v in _ref_eval(opt, tr, b, mask, end, **kw).items()})
    opt.close()
    ref.close()
    return out


def test_combine_cost_exploration_objective_matches_reference(opt_scene):
    """NORMAL_PHASE | MINTIME, the objective of the exploration replan (and of bench.py), bit for bit."""
    P = pins("exploration_objective")
    P.check("esdf", opt_scene["dist"].reshape(-1))
    for key, b, mask, end, kw in _exploration_cases(opt_scene["tr"]):
        _check_eval(P, key, _orc_eval(opt_scene, b, mask, end, **kw))


def _other_term_cases(tr):
    rng = np.random.default_rng(9)
    for b in range(6):
        endp = tr["end_pos"][b]
        # fixed knot span (no MINTIME), end state with 1, 2, 3 rows
        for n_end in (1, 2, 3):
            end = np.concatenate([endp[None, :], rng.normal(size=(2, 3)) * 0.5])[:n_end]
            yield "b%d_end%d" % (b, n_end), b, O.NORMAL_PHASE, end, dict(seed=n_end)
        # GUIDE_PHASE with a guide path (N - 2*order points) and a duration lower bound
        guide = tr["ctrl"][b][3:17] + rng.normal(size=(14, 3)) * 0.2
        yield "b%d_guide" % b, b, O.GUIDE_PHASE | O.MINTIME, endp[None, :], dict(guide=guide, time_lb=9.0, seed=7)
        # way points
        widx = np.array([2, 7, 11], np.int32)
        wp = tr["ctrl"][b][widx + 1] + rng.normal(size=(3, 3)) * 0.1
        yield ("b%d_waypt" % b, b, O.SMOOTHNESS | O.WAYPOINTS | O.START | O.END | O.MINTIME, endp[None, :],
               dict(waypts=wp, widx=widx, seed=8))


def ref_other_terms():
    inflate, tri, tr = _opt_inputs()
    ref, opt = _ref_opt_scene(inflate, tri)
    out = {}
    for key, b, mask, end, kw in _other_term_cases(tr):
        out.update({key + "_" + k: v for k, v in _ref_eval(opt, tr, b, mask, end, **kw).items()})
    opt.close()
    ref.close()
    return out


def test_combine_cost_other_terms_match_reference(opt_scene):
    P = pins("other_terms")
    for key, b, mask, end, kw in _other_term_cases(opt_scene["tr"]):
        _check_eval(P, key, _orc_eval(opt_scene, b, mask, end, **kw))


# ---------------------------------------------------------------------------------------------------------
# FrontierFinder: the reference's own frontier_finder.cpp + perception_utils.cpp (searchFrontiers, expandFrontier,
# computeFrontierInfo, splitLargeFrontiers, computeFrontiersToVisit / sampleViewpoints / countVisibleCells,
# isFrontierCovered) vs the oracle.  pcl::VoxelGrid and Eigen::EigenSolver are the oracle's reconstructions on BOTH
# sides (ref_standin), so they are not what is being checked here.
# ---------------------------------------------------------------------------------------------------------
FF = dict(cluster_min=20, cluster_size_xy=1.0, cluster_size_z=10.0, min_candidate_dist=0.75, min_candidate_clearance=0.21,
          candidate_dphi=15 * 3.1415926 / 180.0, candidate_rmax=2.5, candidate_rmin=1.5, candidate_rnum=3, down_sample=3,
          min_visib_num=8, min_view_finish_fraction=0.2)
PU = dict(top_angle=0.56125, left_angle=0.69222, right_angle=0.68901, max_dist=4.5, vis_dist=1.0)


def frontier_params(box):
    params = dict(BASE)
    if box is not None:
        for ax, lo, hi in zip("xyz", box[0], box[1]):
            params["box_min_" + ax], params["box_max_" + ax] = lo, hi
    return params


def frontier_scene(seed):
    """known region: a few camera balls; the rest unknown"""
    n, _, _ = geometry(BASE)
    rng = np.random.default_rng(seed)
    inflate = (rng.random(n) < 0.003).astype(np.int8)
    X, Y, Z = np.meshgrid(*[np.arange(k) for k in n], indexing="ij")
    known = np.zeros(n, bool)
    for _ in range(5):
        c = rng.uniform(0.2, 0.8, 3) * np.array(n)
        r = rng.uniform(0.2, 0.45) * min(n[0], n[1])
        known |= ((X - c[0]) ** 2 + (Y - c[1]) ** 2 + 4.0 * (Z - c[2]) ** 2) < r * r
    tri = np.where(known, W.FREE, W.UNKNOWN).astype(np.uint8)
    tri[known & (inflate == 1)] = W.OCCUPIED
    inflate[~known] = 0
    return inflate, tri


def ref_frontier_scene(seed, box):
    ref = O.RefSDFMap(**frontier_params(box))
    inflate, tri = frontier_scene(seed)
    load_state(ref, inflate, tri)
    return ref, O.RefFrontierFinder(ref, PU, **FF), inflate, tri


def cluster_arrays(clusters, prefix=""):
    """a cluster list (dicts of the oracle or the reference) as flat arrays"""
    out = {"count": [len(clusters)],
           "offsets": np.cumsum([0] + [len(c["addr"]) for c in clusters]),
           "foffsets": np.cumsum([0] + [len(c["filtered"]) for c in clusters])}
    for k in ("addr", "filtered", "average", "box_min", "box_max"):
        out[k] = np.concatenate([np.ravel(c[k]) for c in clusters]) if clusters else np.zeros(0)
    return {prefix + k: v for k, v in out.items()}


def check_clusters(P, got, prefix, what=""):
    for k, v in cluster_arrays(got, prefix).items():
        P.check(k, v, what)


SEARCHES = [
    (1, None, ((-4.0, -3.0, -0.5), (4.0, 3.0, 2.5))),
    (2, ((-3.5, -2.5, -0.3), (3.5, 2.5, 2.2)), ((-4.0, -3.0, -0.5), (4.0, 3.0, 2.5))),
    (3, ((-3.5, -2.5, -0.3), (3.5, 2.5, 2.2)), ((-1.0, -2.0, 0.0), (2.5, 1.0, 1.5))),
    (4, None, ((0.5, -1.0, 0.2), (3.0, 2.5, 1.8))),
]
SECOND_UPDATE = ((-4.0, -3.0, -0.5), (0.0, 3.0, 2.5))


def ref_search_frontiers(seed, box, upd):
    ref, ff, _, _ = ref_frontier_scene(seed, box)
    out = cluster_arrays(ff.search(*upd), "first_")
    out["first_flags"] = ff.flags.copy()
    # a second search over a different updated box keeps the flags of the first (persistent frontier_flag_)
    out.update(cluster_arrays(ff.search(*SECOND_UPDATE), "second_"))
    out["second_flags"] = ff.flags.copy()
    ff.close()
    ref.close()
    return out


@pytest.mark.parametrize("seed,box,upd", SEARCHES)
def test_search_frontiers_matches_reference(seed, box, upd):
    P = pins("search_frontiers", seed, box, upd)
    n, _, _ = geometry(BASE)
    inflate, tri = frontier_scene(seed)
    g = grid(frontier_params(box), *(box if box is not None else (None, None)))
    flag = np.zeros(n, np.int8)
    p = O.frontier_params(cluster_min=FF["cluster_min"], cluster_size_xy=FF["cluster_size_xy"], down_sample=FF["down_sample"],
                          cell_order=0)
    got = O.frontier_search(g, tri, flag, upd[0], upd[1], p)
    assert len(got) >= 3
    check_clusters(P, got, "first_")
    P.check("first_flags", flag.reshape(-1))
    got2 = O.frontier_search(g, tri, flag, SECOND_UPDATE[0], SECOND_UPDATE[1], p)
    check_clusters(P, got2, "second_")
    P.check("second_flags", flag.reshape(-1))


VIEW_BOX = ((-3.6, -2.6, -0.3), (3.6, 2.6, 2.2))
VIEW_UPDATE = ((-4.0, -3.0, -0.5), (4.0, 3.0, 2.5))


def reveal_around(tri, occ, addr, n):
    """make the unknown 6-neighbours of the given cells known free"""
    idx = np.stack(np.unravel_index(addr, n), axis=1)
    for d in (-1, 1):
        for ax in range(3):
            j = idx.copy()
            j[:, ax] = np.clip(j[:, ax] + d, 0, n[ax] - 1)
            sel = tri[j[:, 0], j[:, 1], j[:, 2]] == W.UNKNOWN
            tri[j[sel, 0], j[sel, 1], j[sel, 2]] = W.FREE
            if occ is not None:
                occ[j[sel, 0], j[sel, 1], j[sel, 2]] = logit(0.12)


def ref_viewpoints_and_coverage():
    ref, ff, _, tri = ref_frontier_scene(6, VIEW_BOX)
    tmp = ff.search(*VIEW_UPDATE)
    visit, dormant = ff.compute_to_visit()
    assert len(visit) + len(dormant) == len(tmp) and len(visit) >= 2
    first = [int(t["addr"][0]) for t in tmp]
    out = cluster_arrays(tmp, "tmp_")
    out["visit_index"] = [first.index(int(v["addr"][0])) for v in visit]
    out["dormant_index"] = [first.index(int(v["addr"][0])) for v in dormant]
    out["visit_ids"] = [v["id"] for v in visit]
    for i, v in enumerate(visit):
        assert list(v["view_visib"]) == sorted(v["view_visib"], reverse=True)
        out["visit_addr%d" % i] = v["addr"]
        out["visit_vp%d" % i] = viewpoint_rows(v["view_visib"], v["view_yaw"], v["view_pos"])
    # isFrontierCovered: nothing changed -> False; reveal the surroundings of the first cluster -> True
    ref.R.ref_map_set_updated_box(ref.h, O._p(np.array(VIEW_UPDATE[0])), O._p(np.array(VIEW_UPDATE[1])))
    covered = [ff.is_covered()]
    reveal_around(tri.copy(), ref.occupancy.reshape(ref.n), visit[0]["addr"], ref.n)
    covered.append(ff.is_covered())
    out["covered"] = covered
    ff.close()
    ref.close()
    return out


def test_viewpoints_and_coverage_match_reference():
    """computeFrontiersToVisit (sampleViewpoints / countVisibleCells / isNearUnknown, PerceptionUtils) and
    isFrontierCovered.  Same libm on both sides here, so yaw and counts are compared exactly."""
    P = pins("viewpoints_and_coverage")
    n, _, _ = geometry(BASE)
    inflate, tri = frontier_scene(6)
    g = grid(frontier_params(VIEW_BOX), *VIEW_BOX)
    p = O.frontier_params(cluster_min=FF["cluster_min"], cluster_size_xy=FF["cluster_size_xy"], down_sample=FF["down_sample"],
                          cell_order=0)
    tmp = O.frontier_search(g, tri, np.zeros(n, np.int8), VIEW_UPDATE[0], VIEW_UPDATE[1], p)
    check_clusters(P, tmp, "tmp_")
    vp = O.view_params()
    visit, dormant = [], []
    for i, t in enumerate(tmp):
        r = O.sample_viewpoints(g, tri, inflate, vp, t["average"], t["filtered"])
        keep = np.nonzero(r["visib"] > FF["min_visib_num"])[0]
        if len(keep) == 0:
            dormant.append(i)
            continue
        P.check("visit_addr%d" % len(visit), t["addr"])
        P.check("visit_vp%d" % len(visit), viewpoint_rows(r["visib"][keep], r["yaw"][keep], r["pos"][keep]))
        visit.append(i)
    P.check("visit_index", visit)
    P.check("dormant_index", dormant)
    P.check("visit_ids", np.arange(len(visit)))
    # isFrontierCovered: nothing changed -> no cell of the first cluster changed; reveal its surroundings -> enough did
    first = tmp[visit[0]]["addr"]
    thresh = max(int(FF["min_view_finish_fraction"] * len(first)), 1)
    cnt0 = O.frontier_changed_count(g, tri, first)
    tri2 = tri.copy()
    reveal_around(tri2, None, first, n)
    cnt = O.frontier_changed_count(g, tri2, first)
    assert cnt0 == 0 and cnt >= thresh
    P.check("covered", [cnt0 >= thresh, cnt >= thresh])


ODD_MAP = dict(BASE, map_size_x=6.45, map_size_y=4.83, map_size_z=2.41, max_ray_length=2.0)


def _odd_map_frames():
    """four clouds close to the +x/+y/+z faces, then probe points around the upper faces (one generator)"""
    rng = np.random.default_rng(8)
    for frame in range(4):
        cam = np.array([rng.uniform(1.5, 3.0), rng.uniform(1.0, 2.2), rng.uniform(0.5, 1.6)])
        pts = (cam + rng.normal(size=(3000, 3)) * np.array([1.5, 1.5, 0.8])).astype(np.float32)
        yield frame, cam, pts
    _, origin, size = geometry(ODD_MAP)
    yield None, None, origin + size - rng.uniform(-0.02, 0.15, (2000, 3))


def ref_odd_map_size():
    ref = O.RefSDFMap(**ODD_MAP)
    out = {"n": ref.n, "origin": ref.origin.copy()}
    for frame, cam, pts in _odd_map_frames():
        if frame is None:
            ref.set_modes(0, 0)
            ref.set_local_bound((0, 0, 0), np.array(ref.n) - 1)
            ref.update_esdf3d()
            out["esdf"] = ref.distance.copy()
            out["d"], out["grad"] = ref.dist_with_grad(pts)
            break
        ref.input_point_cloud(pts, cam)
        out["logodds%d" % frame] = ref.occupancy.copy()
        out["bound%d" % frame] = _cat(*ref.get_local_bound())
    ref.close()
    return out


def test_map_size_that_is_not_a_multiple_of_the_resolution():
    """map_voxel_num_ = ceil(size / resolution) but map_max_boundary_ = origin + size (sdf_map.cpp:34-39): with a size of
    6.45 m the last voxel column lies partly outside the map.  isInMap / closetPointInMap / getDistWithGrad use the
    metric boundary; the oracle takes it through OrcGrid.map_size (the C ABI through FuelGridDesc.map_size)."""
    P = pins("odd_map_size")
    n, origin, _ = geometry(ODD_MAP)
    P.check("n", n)
    P.check("origin", origin)
    assert n == (65, 49, 25)
    g = grid(ODD_MAP)
    f = O.Fusion(g, O.fusion_params(max_ray_length=2.0))
    for frame, cam, pts in _odd_map_frames():
        if frame is None:
            # the reference's inflation buffer is still empty: no clearAndInflateLocalMap ran
            dist = O.update_esdf3d(g, np.zeros(n, np.int8), f.tristate().reshape(n), (0, 0, 0), np.array(n) - 1, 0, 0)
            P.check("esdf", dist.reshape(-1))
            d, gr = O.dist_with_grad(g, dist, pts)
            P.check("d", d)
            P.check("grad", gr)
            assert (d == 0).sum() > 100 and (d != 0).sum() > 100
            break
        lo, hi = f.input_point_cloud(pts, cam)
        P.check("logodds%d" % frame, f.logodds, "frame %d" % frame)
        P.check("bound%d" % frame, _cat(lo, hi), "frame %d" % frame)


WEIGHT_SEEDS = [(0,), (1,), (2,)]


def _random_weights_case(seed):
    """Random lambda weights / limits, 8..31 control points, random term masks, end-state rows and duration bounds."""
    rng = np.random.default_rng(seed)
    n, _, _ = geometry(BASE)
    inflate, tri = random_state(n, 300 + seed, p_site=float(rng.choice([0.002, 0.01])))
    optimistic = int(rng.integers(0, 2))
    keys = ("ld_smooth", "ld_dist", "ld_feasi", "ld_start", "ld_end", "ld_guide", "ld_waypt", "ld_time", "dist0", "max_vel", "max_acc")
    lo_hi = dict(ld_smooth=(1, 30), ld_dist=(1, 20), ld_feasi=(0.5, 5), ld_start=(1, 100), ld_end=(0.1, 5), ld_guide=(0.5, 3),
                 ld_waypt=(0.1, 2), ld_time=(0.5, 3), dist0=(0.3, 1.2), max_vel=(0.5, 3), max_acc=(0.5, 3))
    w = {k: float(rng.uniform(*lo_hi[k])) for k in keys}
    N = int(rng.choice([8, 12, 20, 31]))
    tr = W.make_trajectories(wgrid(BASE), inflate, B=5, n_pts=N, seed=seed)
    cases = []
    for b in range(5):
        mask = int(rng.choice([O.NORMAL_PHASE | O.MINTIME, O.NORMAL_PHASE, O.GUIDE_PHASE | O.MINTIME,
                               O.SMOOTHNESS | O.WAYPOINTS | O.START | O.END, O.DISTANCE | O.FEASIBILITY | O.MINTIME]))
        ctrl, dt = tr["ctrl"][b], float(tr["dt"][b])
        guide = ctrl[3:N - 3] + rng.normal(size=(N - 6, 3)) * 0.2 if mask & O.GUIDE else None
        widx = np.array([1, N // 2 - 1, N - 4], np.int32) if mask & O.WAYPOINTS else None
        wp = ctrl[widx + 1] + rng.normal(size=(3, 3)) * 0.1 if widx is not None else None
        end = np.concatenate([tr["end_pos"][b][None, :], rng.normal(size=(2, 3)) * 0.5])[:int(rng.integers(1, 4))]
        tlb = float(rng.choice([-1.0, 6.0, 20.0]))
        nvar = 3 * N + (1 if mask & O.MINTIME else 0)
        probes = np.concatenate([ctrl.reshape(-1), [dt]])[:nvar] + rng.normal(size=(4, nvar)) * 0.3
        if mask & O.MINTIME:
            probes[:, -1] = np.abs(probes[:, -1]) + 0.03
        cases.append((b, mask, guide, widx, wp, end, tlb, probes))
    return inflate, tri, optimistic, w, N, tr, cases


def clamped_start(tr, b, nvar):
    """the start point optimize() hands to NLopt: control points clamped to the box shrunk by 0.1 m (:175-217)"""
    n, origin, _ = geometry(BASE)
    x0 = np.concatenate([tr["ctrl"][b].reshape(-1), [tr["dt"][b]]])[:nvar]
    x0[:3 * tr["ctrl"].shape[1]] = np.clip(tr["ctrl"][b], origin + 0.1, origin + np.array(n) * BASE["resolution"] - 0.1).reshape(-1)
    return x0


def ref_random_weights(seed):
    inflate, tri, optimistic, w, N, tr, cases = _random_weights_case(seed)
    ref, opt = _ref_opt_scene(inflate, tri, optimistic, **w)
    out = {"esdf": ref.distance.copy()}
    for b, mask, guide, widx, wp, end, tlb, probes in cases:
        r = opt.evaluate(tr["ctrl"][b], float(tr["dt"][b]), mask, tr["start"][b], end, guide, wp, widx, tlb, probes)
        out.update({"b%d_x0" % b: r["x0"], "b%d_f" % b: r["f"], "b%d_grad" % b: r["grad"]})
    opt.close()
    ref.close()
    return out


@pytest.mark.parametrize("seed", [s[0] for s in WEIGHT_SEEDS])
def test_combine_cost_random_weights_sizes_and_masks(seed):
    P = pins("random_weights", seed)
    inflate, tri, optimistic, w, N, tr, cases = _random_weights_case(seed)
    g = grid(BASE)
    dist = O.update_esdf3d(g, inflate, tri, *FULL_BOX, optimistic, 0)
    P.check("esdf", dist.reshape(-1))
    p = O.opt_params(**w)
    for b, mask, guide, widx, wp, end, tlb, probes in cases:
        x0 = clamped_start(tr, b, probes.shape[1])
        P.check("b%d_x0" % b, x0)
        tc = O.traj_consts(1)
        O.fill_traj_const(tc[0], O.pt_dist(tr["ctrl"][b]), float(tr["dt"][b]), tr["start"][b], end, tlb, guide, wp, widx)
        X = np.concatenate([x0[None, :], probes])
        out = [O.combine_cost_batch(g, dist, p, tc, N, mask, X[i:i + 1]) for i in range(len(X))]
        f, gr = np.concatenate([o[0] for o in out]), np.concatenate([o[1] for o in out])
        P.check("b%d_f" % b, f, "mask %d" % mask)
        P.check("b%d_grad" % b, gr, "mask %d" % mask)


def test_host_mirror_pt_dist_is_the_reference_value(opt_scene):
    """pt_dist_ (bspline_optimizer.cpp:136-140) as the Python mirror and workloads.make_trajectories compute it ==
    the oracle's, which the tests above pin to the reference through the smoothness term."""
    import fuel_b200
    tr = opt_scene["tr"]
    for b in range(tr["ctrl"].shape[0]):
        assert fuel_b200.BsplineOptimizer.pt_dist(tr["ctrl"][b]) == O.pt_dist(tr["ctrl"][b]) == tr["pt_dist"][b]


VIEW_SEEDS = [(0,), (1,)]


def _view_cost_case(seed):
    rng = np.random.default_rng(40 + seed)
    n, _, _ = geometry(BASE)
    inflate, tri = random_state(n, 500 + seed)
    w = dict(ld_view=float(rng.uniform(0.5, 5)), wnl=float(rng.uniform(0.2, 3)))
    N = 20
    tr = W.make_trajectories(wgrid(BASE), inflate, B=6, n_pts=N, seed=seed)
    cases = []
    for b in range(6):
        ctrl, dt = tr["ctrl"][b], float(tr["dt"][b])
        idx = int(rng.integers(3, N - 3))
        pt = ctrl[idx] + rng.normal(size=3) * 0.4
        # direction roughly along / against (pt -> control point), short or long safe distance
        d = (ctrl[idx] - pt) * float(rng.choice([-1.0, 1.0])) + rng.normal(size=3) * 0.1
        d = d / np.linalg.norm(d) * float(rng.choice([0.2, 1.5]))
        for mask in (O.VIEWCONS, O.NORMAL_PHASE | O.VIEWCONS | O.MINTIME):
            nvar = 3 * N + (1 if mask & O.MINTIME else 0)
            probes = np.concatenate([ctrl.reshape(-1), [dt]])[:nvar] + rng.normal(size=(3, nvar)) * 0.2
            if mask & O.MINTIME:
                probes[:, -1] = np.abs(probes[:, -1]) + 0.03
            cases.append((b, mask, (pt, d, idx), probes))
    return inflate, tri, w, N, tr, cases


def ref_view_cost(seed):
    inflate, tri, w, N, tr, cases = _view_cost_case(seed)
    ref, opt = _ref_opt_scene(inflate, tri, 1, **w)
    out = {"esdf": ref.distance.copy()}
    for b, mask, view, probes in cases:
        r = opt.evaluate(tr["ctrl"][b], float(tr["dt"][b]), mask, tr["start"][b], tr["end_pos"][b][None, :], probes=probes,
                         view=view)
        out.update({"b%d_%d_x0" % (b, mask): r["x0"], "b%d_%d_f" % (b, mask): r["f"], "b%d_%d_grad" % (b, mask): r["grad"]})
    opt.close()
    ref.close()
    return out


@pytest.mark.parametrize("seed", [s[0] for s in VIEW_SEEDS])
def test_view_cost_matches_reference(seed):
    """calcViewCost (bspline_optimizer.cpp:477-502, VIEWCONS): the perpendicular part, the parallel part on both sides of
    its |dl| < |dir| switch, random ld_view / wnl, alone and inside a full objective -- bit for bit."""
    P = pins("view_cost", seed)
    inflate, tri, w, N, tr, cases = _view_cost_case(seed)
    g = grid(BASE)
    dist = O.update_esdf3d(g, inflate, tri, *FULL_BOX, 1, 0)
    P.check("esdf", dist.reshape(-1))
    p = O.opt_params(**w)
    n_par = 0
    for b, mask, view, probes in cases:
        key = "b%d_%d_" % (b, mask)
        x0 = clamped_start(tr, b, probes.shape[1])
        P.check(key + "x0", x0)
        tc = O.traj_consts(1)
        O.fill_traj_const(tc[0], O.pt_dist(tr["ctrl"][b]), float(tr["dt"][b]), tr["start"][b], tr["end_pos"][b][None, :], view=view)
        X = np.concatenate([x0[None, :], probes])
        out = [O.combine_cost_batch(g, dist, p, tc, N, mask, X[i:i + 1]) for i in range(len(X))]
        f, gr = np.concatenate([o[0] for o in out]), np.concatenate([o[1] for o in out])
        P.check(key + "f", f)
        P.check(key + "grad", gr)
        if mask == O.VIEWCONS:
            pt, d, idx = view
            q = X[0][:3 * N].reshape(N, 3)[idx] - pt
            n_par += int(abs(np.dot(q, d / np.linalg.norm(d))) < np.linalg.norm(d))
            assert np.count_nonzero(gr[0]) <= 3  # one control point only
    assert n_par >= 1  # the wnl branch was taken at least once


# the reference side of every test above: name -> (function, argument tuples)
REF_PINS = {
    "intbound": (ref_intbound, [()]),
    "rays": (ref_rays, [tuple(a) for a in RAY_GRIDS]),
    "esdf": (ref_esdf, ESDF_MODES),
    "esdf_sentinel": (ref_esdf_sentinel, [()]),
    "clear_and_inflate": (ref_clear_and_inflate, INFLATE_CEILINGS),
    "input_point_cloud": (ref_input_point_cloud, [()]),
    "depth_chain": (ref_depth_chain, [()]),
    "dist_with_grad": (ref_dist_with_grad, [()]),
    "exploration_objective": (ref_exploration_objective, [()]),
    "other_terms": (ref_other_terms, [()]),
    "search_frontiers": (ref_search_frontiers, SEARCHES),
    "viewpoints_and_coverage": (ref_viewpoints_and_coverage, [()]),
    "odd_map_size": (ref_odd_map_size, [()]),
    "random_weights": (ref_random_weights, WEIGHT_SEEDS),
    "view_cost": (ref_view_cost, VIEW_SEEDS),
}
