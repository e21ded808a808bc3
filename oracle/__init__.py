"""ctypes binding of the CPU oracle (oracle/fuel_oracle.c).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  fuel_b200/ must never import this package.
PARITY UNPINNED by reference tests (the reference ships none for this path); see
fuel_oracle.h.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libfuel_oracle.so")

ORC_MAX_PTS = 64

UNKNOWN, FREE, OCCUPIED = 0, 1, 2
SMOOTHNESS, DISTANCE, FEASIBILITY, START, END, GUIDE, WAYPOINTS, VIEWCONS, MINTIME = (
    1 << 0, 1 << 1, 1 << 2, 1 << 3, 1 << 4, 1 << 5, 1 << 6, 1 << 7, 1 << 8)
NORMAL_PHASE = SMOOTHNESS | DISTANCE | FEASIBILITY | START | END
GUIDE_PHASE = SMOOTHNESS | GUIDE | START | END


def build(force=False):
    """Compile the oracle with the committed Makefile (gcc -O3, the reference's flags)."""
    src = [os.path.join(_HERE, f) for f in ("fuel_oracle.c", "fuel_oracle_fusion.c", "fuel_oracle_viewpoints.c",
                                            "fuel_oracle.h", "Makefile", "ref_raycast_wrap.cpp", "ref_sdfmap_wrap.cpp", "ref_bspline_wrap.cpp",
                                            "ref_frontier_wrap.cpp")]
    ref_src = "/root/reference/fuel_planner/plan_env/src/raycast.cpp"
    ref_ok = not os.path.exists(ref_src) or os.path.exists(os.path.join(_HERE, "_ref", "libfuel_ref.so"))
    if (not force and os.path.exists(_SO) and ref_ok
            and all(os.path.getmtime(_SO) >= os.path.getmtime(s) for s in src)):
        return _SO
    subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


class OrcGrid(C.Structure):
    _fields_ = [("n", C.c_int32 * 3), ("res", C.c_double), ("origin", C.c_double * 3),
                ("box_mind", C.c_double * 3), ("box_maxd", C.c_double * 3), ("map_size", C.c_double * 3)]


class OrcFrontierParams(C.Structure):
    _fields_ = [("cluster_min", C.c_int32), ("cluster_size_xy", C.c_double),
                ("down_sample", C.c_int32), ("min_z", C.c_double), ("cell_order", C.c_int32)]


class OrcFusionParams(C.Structure):
    _fields_ = [(k, C.c_double) for k in
                ("p_hit", "p_miss", "p_min", "p_max", "p_occ", "max_ray_length", "local_bound_inflate")]


class OrcFusionState(C.Structure):
    _fields_ = [("count_hit", C.c_void_p), ("count_miss", C.c_void_p), ("flag_rayend", C.c_void_p),
                ("raycast_num", C.c_int8), ("reset_updated_box", C.c_int32),
                ("update_min", C.c_double * 3), ("update_max", C.c_double * 3)]


class OrcCameraParams(C.Structure):
    _fields_ = [(k, C.c_double) for k in ("fx", "fy", "cx", "cy", "k_depth_scaling_factor", "depth_filter_maxdist",
                                          "depth_filter_mindist")] + [("depth_filter_margin", C.c_int32),
                                                                      ("skip_pixel", C.c_int32)]


class OrcViewParams(C.Structure):
    _fields_ = [("candidate_rmin", C.c_double), ("candidate_rmax", C.c_double), ("candidate_rnum", C.c_int32),
                ("candidate_dphi", C.c_double), ("min_candidate_clearance", C.c_double), ("top_angle", C.c_double),
                ("left_angle", C.c_double), ("right_angle", C.c_double), ("max_dist", C.c_double)]


class OrcOptParams(C.Structure):
    _fields_ = [(k, C.c_double) for k in
                ("ld_smooth", "ld_dist", "ld_feasi", "ld_start", "ld_end", "ld_guide",
                 "ld_waypt", "ld_view", "ld_time", "dist0", "max_vel", "max_acc")] + [
                     ("order", C.c_int32), ("wnl", C.c_double)]


class OrcTrajConst(C.Structure):
    _fields_ = [("pt_dist", C.c_double), ("knot_span", C.c_double),
                ("start", (C.c_double * 3) * 3), ("end", (C.c_double * 3) * 3),
                ("n_end", C.c_int32), ("time_lb", C.c_double), ("n_guide", C.c_int32),
                ("guide", (C.c_double * 3) * ORC_MAX_PTS), ("n_waypt", C.c_int32),
                ("waypt", (C.c_double * 3) * ORC_MAX_PTS), ("waypt_idx", C.c_int32 * ORC_MAX_PTS),
                ("view_pt", C.c_double * 3), ("view_dir", C.c_double * 3), ("view_idx", C.c_int32)]


class OrcSolveParams(C.Structure):
    _fields_ = [("max_eval", C.c_int32), ("lbfgs_m", C.c_int32), ("xtol_rel", C.c_double), ("flags", C.c_int32),
                ("reserved", C.c_int32)]


class OrcSolveTrace(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("n_kept", "n_curv_reject", "n_full_reject", "n_restart", "n_ls_fail",
                                          "first_full_reject", "first_ls_fail")]


SOLVE_EXACT_EVALS = 1


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.orc_dist_with_grad.restype = C.c_double
        _lib.orc_pt_dist.restype = C.c_double
        _lib.orc_frontier_search.restype = C.c_void_p
        for name in ("orc_frontier_count", "orc_frontier_num_cells", "orc_frontier_num_filtered",
                     "orc_frontier_is_changed", "orc_is_frontier_cell", "orc_is_in_map_pos"):
            getattr(_lib, name).restype = C.c_int32
    return _lib


def _p(a, ty=None):
    if a is None:
        return None
    return a.ctypes.data_as(C.c_void_p)


def make_grid(n, res, origin, box_mind=None, box_maxd=None, map_size=None):
    """map_size = map_size_ of the reference (map_max_boundary_ = origin + map_size_); None -> n * res"""
    g = OrcGrid()
    for i in range(3):
        g.n[i] = int(n[i])
        g.origin[i] = float(origin[i])
    g.res = float(res)
    if box_mind is None:
        box_mind = [origin[i] for i in range(3)]
    if box_maxd is None:
        box_maxd = [origin[i] + n[i] * res for i in range(3)]
    for i in range(3):
        g.box_mind[i] = float(box_mind[i])
        g.box_maxd[i] = float(box_maxd[i])
        g.map_size[i] = 0.0 if map_size is None else float(map_size[i])
    return g


def pos_to_index(g, pos):
    pos = np.ascontiguousarray(pos, dtype=np.float64)
    out = np.zeros(3, dtype=np.int32)
    lib().orc_pos_to_index(C.byref(g), _p(pos), _p(out))
    return out


def tristate_from_logodds(logodds, clamp_min_log, min_occupancy_log):
    logodds = np.ascontiguousarray(logodds, dtype=np.float64)
    tri = np.empty(logodds.shape, dtype=np.uint8)
    lib().orc_tristate_from_logodds(_p(logodds), C.c_int64(logodds.size), C.c_double(clamp_min_log),
                                    C.c_double(min_occupancy_log), _p(tri))
    return tri


def update_esdf3d(g, inflate, tri, bmin, bmax, optimistic, signed_dist, dist=None, threads=1):
    """updateESDF3d.  inflate int8 [nx,ny,nz]; tri uint8 or None.  Returns distance_buffer_
    (float64 [nx,ny,nz]); voxels outside the box keep their previous value (`dist` in, or 0 =
    sdf_map/default_dist of algorithm.xml:41)."""
    shape = tuple(g.n)
    inflate = np.ascontiguousarray(inflate, dtype=np.int8).reshape(shape)
    if tri is not None:
        tri = np.ascontiguousarray(tri, dtype=np.uint8).reshape(shape)
    if dist is None:
        dist = np.zeros(shape, dtype=np.float64)
    else:
        dist = np.ascontiguousarray(dist, dtype=np.float64).reshape(shape)
    neg = np.zeros(shape, dtype=np.float64) if signed_dist else None
    t1 = np.zeros(shape, dtype=np.float64)
    t2 = np.zeros(shape, dtype=np.float64)
    bmin = np.ascontiguousarray(bmin, dtype=np.int32)
    bmax = np.ascontiguousarray(bmax, dtype=np.int32)
    lib().orc_update_esdf3d(C.byref(g), _p(inflate), _p(tri), _p(bmin), _p(bmax),
                            C.c_int(int(optimistic)), C.c_int(int(signed_dist)), _p(dist), _p(neg),
                            _p(t1), _p(t2), C.c_int(threads))
    return dist


def clear_and_inflate(g, tri, inflate, bmin, bmax, inf_step, ceil_id=-1):
    """clearAndInflateLocalMap (sdf_map.cpp:364-472); tri (uint8) and inflate (int8) are updated in place."""
    assert tri.dtype == np.uint8 and inflate.dtype == np.int8 and tri.flags["C_CONTIGUOUS"] and inflate.flags["C_CONTIGUOUS"]
    bmin = np.ascontiguousarray(bmin, dtype=np.int32)
    bmax = np.ascontiguousarray(bmax, dtype=np.int32)
    lib().orc_clear_and_inflate(C.byref(g), _p(tri), _p(inflate), _p(bmin), _p(bmax), C.c_int(inf_step), C.c_int(ceil_id))


def fusion_params(p_hit=0.65, p_miss=0.35, p_min=0.12, p_max=0.90, p_occ=0.80, max_ray_length=4.5,
                  local_bound_inflate=0.5):
    """defaults = exploration_manager/launch/algorithm.xml:39-50"""
    p = OrcFusionParams()
    p.p_hit, p.p_miss, p.p_min, p.p_max, p.p_occ = p_hit, p_miss, p_min, p_max, p_occ
    p.max_ray_length, p.local_bound_inflate = max_ray_length, local_bound_inflate
    return p


def camera_params(fx=387.229248046875, fy=387.229248046875, cx=321.04638671875, cy=243.44969177246094,
                  k_depth_scaling_factor=1000.0, depth_filter_maxdist=5.0, depth_filter_mindist=0.2,
                  depth_filter_margin=2, skip_pixel=2):
    """defaults = exploration.launch:38-41, algorithm.xml:61-69"""
    c = OrcCameraParams()
    c.fx, c.fy, c.cx, c.cy = fx, fy, cx, cy
    c.k_depth_scaling_factor, c.depth_filter_maxdist, c.depth_filter_mindist = (
        k_depth_scaling_factor, depth_filter_maxdist, depth_filter_mindist)
    c.depth_filter_margin, c.skip_pixel = depth_filter_margin, skip_pixel
    return c


def process_depth_image(cp, depth, R, camera_pos):
    """proessDepthImage (map_ros.cpp:176-215) -> float32 [proj_points_cnt, 3]"""
    depth = np.ascontiguousarray(depth, dtype=np.uint16)
    rows, cols = depth.shape
    R = np.ascontiguousarray(R, dtype=np.float64).reshape(9)
    cam = np.ascontiguousarray(camera_pos, dtype=np.float64)
    out = np.empty((rows * cols, 3), dtype=np.float32)
    lib().orc_process_depth_image.restype = C.c_int32
    n = lib().orc_process_depth_image(C.byref(cp), _p(depth), C.c_int32(rows), C.c_int32(cols), _p(R), _p(cam), _p(out))
    return out[:n].copy()


class Fusion:
    """occupancy_buffer_ + the cache arrays of MapData driven by inputPointCloud (sdf_map.cpp:259-345)."""

    def __init__(self, g, params):
        self.g, self.p = g, params
        self.nvox = int(g.n[0]) * int(g.n[1]) * int(g.n[2])
        clamp_min = np.log(params.p_min / (1 - params.p_min))
        self.logodds = np.full(self.nvox, clamp_min - 0.01, dtype=np.float64)  # sdf_map.cpp:56,64
        self.st = OrcFusionState()
        lib().orc_fusion_state_init(C.byref(self.st), C.c_int64(self.nvox))

    def __del__(self):
        try:
            lib().orc_fusion_state_free(C.byref(self.st))
        except Exception:
            pass

    def input_point_cloud(self, points, camera_pos):
        pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
        cam = np.ascontiguousarray(camera_pos, dtype=np.float64)
        lo = np.zeros(3, np.int32)
        hi = np.zeros(3, np.int32)
        lib().orc_input_point_cloud(C.byref(self.g), C.byref(self.p), C.byref(self.st), _p(self.logodds), _p(pts),
                                    C.c_int32(pts.shape[0]), _p(cam), _p(lo), _p(hi))
        return lo, hi

    def updated_box(self, reset=False):
        lo, hi = np.array(self.st.update_min), np.array(self.st.update_max)
        if reset:
            self.st.reset_updated_box = 1
        return lo, hi

    def tristate(self):
        p = self.p
        return tristate_from_logodds(self.logodds, np.log(p.p_min / (1 - p.p_min)), np.log(p.p_occ / (1 - p.p_occ)))


def view_params(candidate_rmin=1.5, candidate_rmax=2.5, candidate_rnum=3, candidate_dphi=15 * 3.1415926 / 180.0,
                min_candidate_clearance=0.21, top_angle=0.56125, left_angle=0.69222, right_angle=0.68901, max_dist=4.5):
    """defaults = exploration_manager/launch/algorithm.xml:106-121"""
    v = OrcViewParams()
    v.candidate_rmin, v.candidate_rmax, v.candidate_rnum, v.candidate_dphi = (
        candidate_rmin, candidate_rmax, candidate_rnum, candidate_dphi)
    v.min_candidate_clearance = min_candidate_clearance
    v.top_angle, v.left_angle, v.right_angle, v.max_dist = top_angle, left_angle, right_angle, max_dist
    return v


def sample_viewpoints(g, tri, inflate, vp, average, cells):
    """sampleViewpoints (frontier_finder.cpp:662-695) for one cluster, all candidates reported.
    -> dict(pos [c,3], yaw [c], visib [c] (-1 = rejected candidate), border [c])"""
    L = lib()
    L.orc_viewpoint_candidates.restype = C.c_int32
    L.orc_sample_viewpoints.restype = C.c_int32
    nc = L.orc_viewpoint_candidates(C.byref(vp), None, C.c_int32(0))
    tri = np.ascontiguousarray(tri, dtype=np.uint8)
    inflate = np.ascontiguousarray(inflate, dtype=np.int8)
    cells = np.ascontiguousarray(cells, dtype=np.float64).reshape(-1, 3)
    avg = np.ascontiguousarray(average, dtype=np.float64)
    pos = np.zeros((nc, 3))
    yaw = np.zeros(nc)
    vis = np.zeros(nc, np.int32)
    brd = np.zeros(nc, np.uint8)
    L.orc_sample_viewpoints(C.byref(g), _p(tri), _p(inflate), C.byref(vp), _p(avg), _p(cells), C.c_int32(cells.shape[0]),
                            _p(pos), _p(yaw), _p(vis), _p(brd))
    return dict(pos=pos, yaw=yaw, visib=vis, border=brd)


def frontier_changed_count(g, tri, addr):
    addr = np.ascontiguousarray(addr, dtype=np.int32)
    lib().orc_frontier_changed_count.restype = C.c_int32
    return lib().orc_frontier_changed_count(C.byref(g), _p(np.ascontiguousarray(tri, dtype=np.uint8)), _p(addr),
                                            C.c_int32(addr.shape[0]))


def raycast_ids(g, start, end, max_ids=8192):
    """the oracle's RayCaster: voxel indices nextId() reports for input(start, end)"""
    out = np.zeros((max_ids, 3), np.int32)
    lib().orc_raycast_ids.restype = C.c_int32
    n = lib().orc_raycast_ids(C.byref(g), _p(np.ascontiguousarray(start, dtype=np.float64)),
                              _p(np.ascontiguousarray(end, dtype=np.float64)), _p(out), C.c_int32(max_ids))
    return out[:n]


_REF_RAYCAST = os.path.join(_HERE, "_ref", "libfuel_ref.so")
_ref_rc = None


def ref_raycast():
    """The REFERENCE's own code (plan_env/src/raycast.cpp + sdf_map.cpp compiled unmodified into
    oracle/_ref/libfuel_ref.so by the Makefile, only where /root/reference exists) or None."""
    global _ref_rc
    if _ref_rc is None and os.path.exists(_REF_RAYCAST):
        _ref_rc = C.CDLL(_REF_RAYCAST)
        _ref_rc.ref_raycast_ids.restype = C.c_int32
        _ref_rc.ref_intbound.restype = C.c_double
        _ref_rc.ref_intbound.argtypes = [C.c_double, C.c_double]
    return _ref_rc


def ref_raycast_ids(g, start, end, max_ids=8192):
    out = np.zeros((max_ids, 3), np.int32)
    origin = np.array([g.origin[0], g.origin[1], g.origin[2]], dtype=np.float64)
    n = ref_raycast().ref_raycast_ids(C.c_double(g.res), _p(origin), _p(np.ascontiguousarray(start, dtype=np.float64)),
                                      _p(np.ascontiguousarray(end, dtype=np.float64)), _p(out), C.c_int32(max_ids))
    return out[:n]


class RefSDFMap:
    """The reference's SDFMap object (sdf_map.cpp compiled from /root/reference), driven through
    oracle/ref_sdfmap_wrap.cpp.  params = the sdf_map/* ROS parameters without the prefix.  The map is centred in
    x,y: origin = (-size_x/2, -size_y/2, ground_height) (sdf_map.cpp:33)."""

    def __init__(self, **params):
        R = ref_raycast()
        keys = [("sdf_map/" + k).encode() for k in params]
        karr = (C.c_char_p * len(keys))(*keys)
        vals = np.array([float(v) for v in params.values()], dtype=np.float64)
        R.ref_map_create.restype = C.c_void_p
        for fn in ("ref_map_occupancy", "ref_map_inflate", "ref_map_distance"):
            getattr(R, fn).restype = C.c_void_p
        R.ref_map_dist_with_grad.restype = C.c_double
        self.R = R
        self.h = C.c_void_p(R.ref_map_create(C.c_int32(len(keys)), karr, _p(vals)))
        n = np.zeros(3, np.int32)
        o = np.zeros(3)
        res = C.c_double()
        R.ref_map_geometry(self.h, _p(n), _p(o), C.byref(res))
        self.n, self.origin, self.res = tuple(int(v) for v in n), o, res.value
        self.map_size = np.array([float(params["map_size_" + a]) for a in "xyz"])
        nv = int(np.prod(n))
        self.occupancy = np.ctypeslib.as_array(C.cast(R.ref_map_occupancy(self.h), C.POINTER(C.c_double)), (nv,))
        self.inflate = np.ctypeslib.as_array(C.cast(R.ref_map_inflate(self.h), C.POINTER(C.c_int8)), (nv,))
        self.distance = np.ctypeslib.as_array(C.cast(R.ref_map_distance(self.h), C.POINTER(C.c_double)), (nv,))

    def close(self):
        if self.h:
            self.occupancy = self.inflate = self.distance = None
            self.R.ref_map_destroy(self.h)
            self.h = None

    def grid(self, box_mind=None, box_maxd=None):
        if box_maxd is None:
            box_maxd = self.origin + self.map_size  # map_max_boundary_ (sdf_map.cpp:39,80-81)
        return make_grid(self.n, self.res, self.origin, box_mind, box_maxd, map_size=self.map_size)

    def set_local_bound(self, lo, hi):
        self.R.ref_map_set_local_bound(self.h, _p(np.ascontiguousarray(lo, dtype=np.int32)),
                                       _p(np.ascontiguousarray(hi, dtype=np.int32)))

    def get_local_bound(self):
        lo, hi = np.zeros(3, np.int32), np.zeros(3, np.int32)
        self.R.ref_map_get_local_bound(self.h, _p(lo), _p(hi))
        return lo, hi

    def set_modes(self, optimistic, signed_dist):
        self.R.ref_map_set_modes(self.h, C.c_int(int(optimistic)), C.c_int(int(signed_dist)))

    def update_esdf3d(self):
        self.R.ref_map_update_esdf3d(self.h)

    def clear_and_inflate(self):
        self.R.ref_map_clear_and_inflate(self.h)

    def input_point_cloud(self, pts, cam):
        pts = np.ascontiguousarray(pts, dtype=np.float32).reshape(-1, 3)
        self.R.ref_map_input_point_cloud(self.h, _p(pts), C.c_int32(pts.shape[0]),
                                         _p(np.ascontiguousarray(cam, dtype=np.float64)))

    def updated_box(self, reset=False):
        a, b = np.zeros(3), np.zeros(3)
        self.R.ref_map_get_updated_box(self.h, _p(a), _p(b), C.c_int(int(reset)))
        return a, b

    def dist_with_grad(self, pos):
        pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 3)
        d = np.zeros(pos.shape[0])
        g = np.zeros((pos.shape[0], 3))
        for i in range(pos.shape[0]):
            d[i] = self.R.ref_map_dist_with_grad(self.h, _p(pos[i]), _p(g[i]))
        return d, g


class RefBsplineOptimizer:
    """The reference's BsplineOptimizer (bspline_optimizer.cpp compiled from /root/reference) on a RefSDFMap.
    params = optimization/* ROS parameters without the prefix (+ bspline_degree)."""

    def __init__(self, ref_map, **params):
        self.R = ref_map.R
        self.map = ref_map
        keys = [(("manager/" if k == "bspline_degree" else "optimization/") + k).encode() for k in params]
        karr = (C.c_char_p * len(keys))(*keys)
        vals = np.array([float(v) for v in params.values()], dtype=np.float64)
        self.R.ref_opt_create.restype = C.c_void_p
        self.R.ref_opt_evaluate.restype = C.c_int32
        self.h = C.c_void_p(self.R.ref_opt_create(ref_map.h, C.c_int32(len(keys)), karr, _p(vals)))

    def close(self):
        if self.h:
            self.R.ref_opt_destroy(self.h)
            self.h = None

    def evaluate(self, ctrl, dt, cost_function, start, end, guide=None, waypts=None, waypt_idx=None, time_lb=-1.0,
                 probes=None, view=None):
        """optimize(points, dt, cost_function, 1, 1) with the NLopt stand-in -> dict(f [1+P], grad [1+P,nvar], x0, lb, ub):
        the reference's objective at its own start point x0 and at the P probe points."""
        ctrl = np.ascontiguousarray(ctrl, dtype=np.float64).reshape(-1, 3)
        n = ctrl.shape[0]
        nvar = 3 * n + (1 if cost_function & MINTIME else 0)
        start = np.ascontiguousarray(start, dtype=np.float64).reshape(-1, 3)
        end = np.ascontiguousarray(end, dtype=np.float64).reshape(-1, 3)
        guide = np.zeros((0, 3)) if guide is None else np.ascontiguousarray(guide, dtype=np.float64).reshape(-1, 3)
        waypts = np.zeros((0, 3)) if waypts is None else np.ascontiguousarray(waypts, dtype=np.float64).reshape(-1, 3)
        widx = np.zeros(0, np.int32) if waypt_idx is None else np.ascontiguousarray(waypt_idx, dtype=np.int32)
        probes = np.zeros((0, nvar)) if probes is None else np.ascontiguousarray(probes, dtype=np.float64).reshape(-1, nvar)
        P = probes.shape[0]
        f = np.zeros(1 + P)
        grad = np.zeros((1 + P, nvar))
        x0, lb, ub = np.zeros(nvar), np.zeros(nvar), np.zeros(nvar)
        if view is not None:  # setViewConstraint (:91-93)
            self.R.ref_opt_set_view(self.h, _p(np.ascontiguousarray(view[0], dtype=np.float64)),
                                    _p(np.ascontiguousarray(view[1], dtype=np.float64)), C.c_int32(int(view[2])))
        rc = self.R.ref_opt_evaluate(self.h, C.c_int32(n), _p(ctrl), C.c_double(dt), C.c_int32(cost_function), _p(start),
                                     C.c_int32(start.shape[0]), _p(end), C.c_int32(end.shape[0]), _p(guide),
                                     C.c_int32(guide.shape[0]), _p(waypts), _p(widx), C.c_int32(waypts.shape[0]),
                                     C.c_double(time_lb), _p(probes), C.c_int32(P), _p(f), _p(grad), _p(x0), _p(lb), _p(ub))
        assert rc == nvar, rc
        return dict(f=f, grad=grad, x0=x0, lb=lb, ub=ub)


def ref_combine_cost_batch(ref_map, opt_params_dict, ctrl, dt, cost_function, start, end_pos, probes, threads=1):
    """K = 1 + probes.shape[1] evaluations of the REFERENCE's combineCost per trajectory (its own start point, then the
    probe points), B trajectories over `threads` host threads with one BsplineOptimizer each
    (oracle/ref_bspline_wrap.cpp: ref_opt_evaluate_batch).  -> f [B, K]"""
    R = ref_map.R
    keys = [(("manager/" if k == "bspline_degree" else "optimization/") + k).encode() for k in opt_params_dict]
    karr = (C.c_char_p * len(keys))(*keys)
    vals = np.array([float(v) for v in opt_params_dict.values()], dtype=np.float64)
    ctrl = np.ascontiguousarray(ctrl, dtype=np.float64)
    B, n = ctrl.shape[0], ctrl.shape[1]
    probes = np.ascontiguousarray(probes, dtype=np.float64)
    K = probes.shape[1] + 1
    f = np.zeros((B, K))
    R.ref_opt_evaluate_batch.restype = C.c_int32
    bad = R.ref_opt_evaluate_batch(ref_map.h, C.c_int32(len(keys)), karr, _p(vals), C.c_int32(B), C.c_int32(n), _p(ctrl),
                                   _p(np.ascontiguousarray(dt, dtype=np.float64)), C.c_int32(cost_function),
                                   _p(np.ascontiguousarray(start, dtype=np.float64)),
                                   _p(np.ascontiguousarray(end_pos, dtype=np.float64)), _p(probes), C.c_int32(K),
                                   C.c_int32(threads), _p(f))
    assert bad == 0
    return f


class RefFrontierFinder:
    """The reference's FrontierFinder (frontier_finder.cpp + perception_utils.cpp compiled from /root/reference) on a
    RefSDFMap.  params: frontier/* keys without prefix; pu_params: perception_utils/* keys without prefix."""

    def __init__(self, ref_map, pu_params=None, **params):
        self.R = ref_map.R
        self.map = ref_map
        kv = {("frontier/" + k): v for k, v in params.items()}
        kv.update({("perception_utils/" + k): v for k, v in (pu_params or {}).items()})
        keys = [k.encode() for k in kv]
        karr = (C.c_char_p * len(keys))(*keys)
        vals = np.array([float(v) for v in kv.values()], dtype=np.float64)
        self.R.ref_ff_create.restype = C.c_void_p
        self.R.ref_ff_flags.restype = C.c_void_p
        self.R.ref_ff_count.restype = C.c_int32
        self.R.ref_ff_is_covered.restype = C.c_int32
        self.h = C.c_void_p(self.R.ref_ff_create(ref_map.h, C.c_int32(len(keys)), karr, _p(vals)))
        nv = int(np.prod(ref_map.n))
        self.flags = np.ctypeslib.as_array(C.cast(self.R.ref_ff_flags(self.h), C.POINTER(C.c_int8)), (nv,))

    def close(self):
        if self.h:
            self.flags = None
            self.R.ref_ff_destroy(self.h)
            self.h = None

    def search(self, upd_min, upd_max):
        """md_->update_min_/max_ := the given box, then searchFrontiers()"""
        self.R.ref_map_set_updated_box(self.map.h, _p(np.ascontiguousarray(upd_min, dtype=np.float64)),
                                       _p(np.ascontiguousarray(upd_max, dtype=np.float64)))
        self.R.ref_ff_search(self.h)
        return self.get_list(0)

    def compute_to_visit(self):
        self.R.ref_ff_compute_to_visit(self.h)
        return self.get_list(1), self.get_list(2)

    def is_covered(self):
        return bool(self.R.ref_ff_is_covered(self.h))

    def search_frontiers(self):
        """searchFrontiers() on whatever updated box the map holds (getUpdatedBox(reset=true) inside)"""
        self.R.ref_ff_search(self.h)
        return self.get_list(0)

    def removed_ids(self):
        out = np.zeros(4096, np.int32)
        self.R.ref_ff_removed_ids.restype = C.c_int32
        n = self.R.ref_ff_removed_ids(self.h, _p(out), C.c_int32(4096))
        return out[:n].tolist()

    def get_list(self, list_id):
        """0 tmp_frontiers_, 1 frontiers_, 2 dormant_frontiers_ -> list of dicts"""
        out = []
        for i in range(self.R.ref_ff_count(self.h, C.c_int32(list_id))):
            nc, nf, nvw, fid = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
            self.R.ref_ff_sizes(self.h, C.c_int32(list_id), C.c_int32(i), C.byref(nc), C.byref(nf), C.byref(nvw), C.byref(fid))
            addr = np.zeros(nc.value, np.int32)
            filt = np.zeros((nf.value, 3))
            avg, bmin, bmax = np.zeros(3), np.zeros(3), np.zeros(3)
            vpos = np.zeros((nvw.value, 3))
            vyaw = np.zeros(nvw.value)
            vvis = np.zeros(nvw.value, np.int32)
            self.R.ref_ff_get(self.h, C.c_int32(list_id), C.c_int32(i), _p(addr), _p(filt), _p(avg), _p(bmin), _p(bmax),
                              _p(vpos), _p(vyaw), _p(vvis))
            out.append(dict(addr=addr, filtered=filt, average=avg, box_min=bmin, box_max=bmax, id=fid.value,
                            view_pos=vpos, view_yaw=vyaw, view_visib=vvis))
        return out


def dist_with_grad(g, dist_buf, pos):
    pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 3)
    dist_buf = np.ascontiguousarray(dist_buf, dtype=np.float64)
    d = np.empty(pos.shape[0], dtype=np.float64)
    gr = np.empty((pos.shape[0], 3), dtype=np.float64)
    lib().orc_dist_with_grad_batch(C.byref(g), _p(dist_buf), C.c_int64(pos.shape[0]), _p(pos), _p(d),
                                   _p(gr))
    return d, gr


def frontier_params(cluster_min=100, cluster_size_xy=2.0, down_sample=3, min_z=0.4, cell_order=0):
    p = OrcFrontierParams()
    p.cluster_min, p.cluster_size_xy, p.down_sample, p.min_z, p.cell_order = (
        cluster_min, cluster_size_xy, down_sample, min_z, cell_order)
    return p


def frontier_search(g, tri, flag, upd_min, upd_max, params):
    """searchFrontiers core.  flag (int8, full volume) is updated in place.  Returns a list of
    dicts {addr, filtered, average, box_min, box_max} in tmp_frontiers_ order."""
    L = lib()
    tri = np.ascontiguousarray(tri, dtype=np.uint8)
    assert flag.dtype == np.int8 and flag.flags["C_CONTIGUOUS"]
    umin = np.ascontiguousarray(upd_min, dtype=np.float64)
    umax = np.ascontiguousarray(upd_max, dtype=np.float64)
    h = C.c_void_p(L.orc_frontier_search(C.byref(g), _p(tri), _p(flag), _p(umin), _p(umax),
                                         C.byref(params)))
    out = []
    try:
        for i in range(L.orc_frontier_count(h)):
            n = L.orc_frontier_num_cells(h, i)
            m = L.orc_frontier_num_filtered(h, i)
            addr = np.empty(n, dtype=np.int32)
            filt = np.empty((m, 3), dtype=np.float64)
            avg = np.empty(3)
            bmin = np.empty(3)
            bmax = np.empty(3)
            L.orc_frontier_get(h, i, _p(addr), _p(filt), _p(avg), _p(bmin), _p(bmax))
            out.append(dict(addr=addr, filtered=filt, average=avg, box_min=bmin, box_max=bmax))
    finally:
        L.orc_frontier_free(h)
    return out


def principal_axis_2x2(a, b, d):
    pc = np.empty(2)
    lib().orc_principal_axis_2x2(C.c_double(a), C.c_double(b), C.c_double(d), _p(pc))
    return pc


def opt_params(ld_smooth=20.0, ld_dist=10.0, ld_feasi=2.0, ld_start=100.0, ld_end=0.5, ld_guide=1.5,
               ld_waypt=0.3, ld_view=0.0, ld_time=1.0, dist0=0.7, max_vel=2.0, max_acc=2.0, order=3, wnl=0.0):
    """Defaults = exploration_manager/launch/algorithm.xml:170-181 and exploration.launch max_vel/acc."""
    p = OrcOptParams()
    p.wnl = wnl
    (p.ld_smooth, p.ld_dist, p.ld_feasi, p.ld_start, p.ld_end, p.ld_guide, p.ld_waypt, p.ld_view,
     p.ld_time, p.dist0, p.max_vel, p.max_acc, p.order) = (ld_smooth, ld_dist, ld_feasi, ld_start,
                                                           ld_end, ld_guide, ld_waypt, ld_view,
                                                           ld_time, dist0, max_vel, max_acc, order)
    return p


def traj_consts(B):
    return (OrcTrajConst * B)()


def fill_traj_const(tc, pt_dist, knot_span, start, end, time_lb=-1.0, guide=None, waypt=None,
                    waypt_idx=None, view=None):
    """view = (pt_ [3], dir_ [3], idx_) of setViewConstraint (bspline_optimizer.cpp:91-93), or None"""
    tc.view_idx = -1
    if view is not None:
        for k in range(3):
            tc.view_pt[k] = float(view[0][k])
            tc.view_dir[k] = float(view[1][k])
        tc.view_idx = int(view[2])
    tc.pt_dist = float(pt_dist)
    tc.knot_span = float(knot_span)
    start = np.asarray(start, dtype=np.float64).reshape(3, 3)
    end = np.asarray(end, dtype=np.float64).reshape(-1, 3)
    for i in range(3):
        for k in range(3):
            tc.start[i][k] = start[i, k]
    tc.n_end = end.shape[0]
    for i in range(end.shape[0]):
        for k in range(3):
            tc.end[i][k] = end[i, k]
    tc.time_lb = float(time_lb)
    tc.n_guide = 0
    tc.n_waypt = 0
    if guide is not None:
        guide = np.asarray(guide, dtype=np.float64).reshape(-1, 3)
        tc.n_guide = guide.shape[0]
        for i in range(guide.shape[0]):
            for k in range(3):
                tc.guide[i][k] = guide[i, k]
    if waypt is not None:
        waypt = np.asarray(waypt, dtype=np.float64).reshape(-1, 3)
        tc.n_waypt = waypt.shape[0]
        for i in range(waypt.shape[0]):
            for k in range(3):
                tc.waypt[i][k] = waypt[i, k]
            tc.waypt_idx[i] = int(waypt_idx[i])


def pt_dist(ctrl):
    ctrl = np.ascontiguousarray(ctrl, dtype=np.float64).reshape(-1, 3)
    return lib().orc_pt_dist(_p(ctrl), C.c_int32(ctrl.shape[0]))


def combine_cost_batch(g, dist_buf, p, tcs, n_pts, mask, x, threads=1):
    x = np.ascontiguousarray(x, dtype=np.float64)
    B = x.shape[0]
    nvar = 3 * n_pts + (1 if mask & MINTIME else 0)
    assert x.shape[1] == nvar
    dist_buf = np.ascontiguousarray(dist_buf, dtype=np.float64)
    f = np.empty(B, dtype=np.float64)
    grad = np.empty((B, nvar), dtype=np.float64)
    lib().orc_combine_cost_batch(C.byref(g), _p(dist_buf), C.byref(p), tcs, C.c_int32(n_pts),
                                 C.c_int32(mask), C.c_int32(B), _p(x), _p(f), _p(grad),
                                 C.c_int(threads))
    return f, grad


def optimize_batch(g, dist_buf, p, tcs, n_pts, mask, x, max_eval=64, lbfgs_m=6, xtol_rel=1e-5, threads=1,
                   exact_evals=False, trace=False):
    """CPU twin of fuelgpu_bspline_optimize_batch (NOT NLopt).  Returns (x_best, f_best, n_eval).
    exact_evals: the FUELGPU_SOLVE_EXACT_EVALS mode (max_eval evaluations, restarts instead of stops).
    trace=True appends a dict of per-trajectory arrays: the OrcSolveTrace fields ([B] each) and "margin"
    [B][max_eval], the smallest relative margin of the branch decisions taken up to each evaluation count."""
    x = np.array(x, dtype=np.float64, order="C", copy=True)
    B = x.shape[0]
    dist_buf = np.ascontiguousarray(dist_buf, dtype=np.float64)
    sp = OrcSolveParams()
    sp.max_eval, sp.lbfgs_m, sp.xtol_rel = max_eval, lbfgs_m, xtol_rel
    sp.flags = SOLVE_EXACT_EVALS if exact_evals else 0
    fb = np.empty(B, dtype=np.float64)
    ne = np.empty(B, dtype=np.int32)
    args = (C.byref(g), _p(dist_buf), C.byref(p), tcs, C.c_int32(n_pts), C.c_int32(mask), C.c_int32(B), C.byref(sp),
            _p(x), _p(fb), _p(ne))
    if not trace:
        lib().orc_optimize_batch(*args, C.c_int(threads))
        return x, fb, ne
    tr = (OrcSolveTrace * B)()
    margin = np.empty((B, max_eval), dtype=np.float64)
    lib().orc_optimize_batch_traced(*args, tr, _p(margin), C.c_int(threads))
    t = np.frombuffer(tr, dtype=np.int32).reshape(B, len(OrcSolveTrace._fields_))
    out = {name: t[:, i].copy() for i, (name, _) in enumerate(OrcSolveTrace._fields_)}
    out["margin"] = margin
    return x, fb, ne, out
