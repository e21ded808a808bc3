"""Shared builders for the parity tests (inputs only)."""
import numpy as np

from fuel_b200 import workloads as W


def random_scene(n, seed, p_site=0.02, p_unknown=0.3, blobs=6):
    """Small random occupancy: sparse inflate bits + blobby known region."""
    rng = np.random.default_rng(seed)
    inflate = (rng.random(n) < p_site).astype(np.int8)
    tri = np.full(n, W.FREE, dtype=np.uint8)
    # unknown blobs
    ax = [np.arange(k) for k in n]
    X, Y, Z = np.meshgrid(*ax, indexing="ij")
    unk = np.zeros(n, dtype=bool)
    for _ in range(blobs):
        c = rng.uniform(0, 1, 3) * np.array(n)
        r = rng.uniform(0.15, 0.45) * min(n)
        unk |= ((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) < r * r
    if p_unknown > 0:
        tri[unk] = W.UNKNOWN
    tri[(inflate == 1) & (tri == W.FREE)] = W.OCCUPIED
    return inflate, tri


def make_sdf_map(fuel, g, inflate, tri, optimistic=False, signed=False):
    m = fuel.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=optimistic, signed_dist=signed)
    m.occupancy_buffer_inflate_[...] = inflate
    m.setOccupancyBuffer(tristate=tri)
    m.upload()
    return m


def sdf_map_geometry(params):
    """map_voxel_num_, map_origin_ and map_size_ as the reference's SDFMap::initMap derives them from its
    sdf_map/* parameters (sdf_map.cpp:33-37): the map is centred in x, y and starts at ground_height in z"""
    size = np.array([params["map_size_" + a] for a in "xyz"])
    n = tuple(int(np.ceil(s / params["resolution"])) for s in size)
    return n, np.array([-size[0] / 2.0, -size[1] / 2.0, params["ground_height"]]), size


def viewpoint_rows(visib, yaw, pos):
    """the viewpoints of one cluster as sorted rows (-visib, yaw, x, y, z): the reference sorts them by visib_num_
    with std::sort, whose order among ties is unspecified, so they are compared as multisets"""
    rows = np.column_stack([-np.asarray(visib, np.float64), yaw, np.reshape(pos, (-1, 3))])
    return rows[np.lexsort(rows.T[::-1])]


def orc_grid(orc, g):
    return orc.make_grid(g.n, g.res, g.origin, g.box_min, g.box_max)


ESDF_SENTINEL = 1e150  # the reference holds resolution*sqrt(DBL_MAX) ~ 1.34e153 where the box has no site
EXACT_N_MAX = 1 << 20
# largest |(got/res)^2 - N_ref| assert_esdf_exact has seen in this process (N_ref <= EXACT_N_MAX)
ESDF_EXACT_STATS = {"max_dev": 0.0, "voxels": 0}


def _esdf_box(got, ref, box):
    if box is None:
        return got, ref
    sl = tuple(slice(int(box[0][i]), int(box[1][i]) + 1) for i in range(3))
    return got[sl], ref[sl]


def _esdf_sentinel(got, ref):
    """+inf on the device exactly where the reference holds its sentinel, with the same sign (a signed field whose box
    is all inflated ends at -inf); returns the mask of finite reference values"""
    nosite = np.abs(ref) > ESDF_SENTINEL
    assert np.array_equal(np.isinf(got), nosite), "sentinel mismatch at %d voxels" % int(
        np.count_nonzero(np.isinf(got) != nosite))
    assert np.array_equal(np.signbit(got[nosite]), np.signbit(ref[nosite])), "sentinel sign mismatch"
    return ~nosite


def assert_esdf_rel(got_f32, ref_f64, box=None, rtol=1e-4):
    """The relative bar: |got - ref| <= rtol*|ref| where the reference is finite, plus the sentinel check."""
    got, ref = _esdf_box(got_f32, ref_f64, box)
    fin = _esdf_sentinel(got, ref)
    g, r = got[fin].astype(np.float64), ref[fin]
    err = np.abs(g - r)
    assert np.all(err <= rtol * np.abs(r)), "max rel err %g" % np.max(err / np.maximum(np.abs(r), 1e-12))


def assert_esdf_exact(got_f32, ref_f64, res, box=None, signed=False):
    """The device field against the fp64 reference to the exact squared voxel distance N.

    Every finite intermediate of the transform is an integer N, and the device stores fl32(res32 * sqrt.approx(N))
    (res32 = float32(res)): a relative error of a few units of 2^-24, so (got/res32)^2 is within 0.4 of N up to
    N = 2^20, while N +- 1 moves the distance by only ~1/(2N) relative (5e-5 at N = 10^4, below a 1e-4 relative bar).
    So N_dev = rint((got/res32)^2) must equal N_ref = rint((ref/res)^2) wherever N_ref <= 2^20, and the largest
    |(got/res32)^2 - N_ref| must stay below 0.45; above 2^20 (diagonals over 1024 voxels) the 1e-4 relative bar
    applies.  Signed fields (esdf.cu signed_merge_kernel: dist += res - neg where neg > 0) are recovered from d where
    the reference is positive and from res - d where it is <= 0.  Returns the largest deviation."""
    got, ref = _esdf_box(got_f32, ref_f64, box)
    fin = _esdf_sentinel(got, ref)
    g, r = got[fin].astype(np.float64), ref[fin]
    res32 = float(np.float32(res))
    if signed:
        neg = r <= 0.0
        g = np.where(neg, res32 - g, g)
        r = np.where(neg, res - r, r)
    q_ref = (r / res) ** 2
    n_ref = np.rint(q_ref)
    assert np.all(np.abs(q_ref - n_ref) < 1e-6), "the reference is not res*sqrt(integer)"
    q_dev = (g / res32) ** 2
    small = n_ref <= EXACT_N_MAX
    dev = np.abs(q_dev[small] - n_ref[small])
    worst = float(dev.max()) if dev.size else 0.0
    bad = np.count_nonzero(np.rint(q_dev[small]) != n_ref[small])
    if bad:
        i = int(np.argmax(dev))
        raise AssertionError("squared voxel distance differs at %d of %d voxels (e.g. N_dev %.3f vs N_ref %d)" %
                             (bad, dev.size, q_dev[small][i], n_ref[small][i]))
    assert worst < 0.45, "largest |(got/res)^2 - N| %.3f: the device rounding is worse than its derivation" % worst
    big = ~small
    if np.any(big):
        gb, rb = got[fin][big].astype(np.float64), ref[fin][big]
        assert np.all(np.abs(gb - rb) <= 1e-4 * np.abs(rb)), "relative error above 1e-4 beyond N = 2^20"
    ESDF_EXACT_STATS["max_dev"] = max(ESDF_EXACT_STATS["max_dev"], worst)
    ESDF_EXACT_STATS["voxels"] += int(dev.size)
    return worst


def rel_err(a, b, floor=0.0):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), floor if floor > 0 else np.finfo(np.float64).tiny)


# ---- a convex quadratic solver objective with a linear-algebra answer -----------------------------------------------
# SMOOTHNESS | START | END | GUIDE | WAYPOINTS with a 3-entry end state and no MINTIME: every term is a square of an
# affine map of the control points, and START / GUIDE / END together pin every point, so the Hessian is positive
# definite.  The weights keep its condition number near 50 (the default weights with dt ~ 0.25 s give ~1e6, where
# 2000 L-BFGS evaluations do not converge and the test would say nothing about the solver's arithmetic).
QUAD_WEIGHTS = dict(ld_smooth=0.05, ld_start=0.2, ld_end=1.0, ld_guide=2.0, ld_waypt=1.0)


def quad_mask(mod):
    return mod.SMOOTHNESS | mod.START | mod.END | mod.GUIDE | mod.WAYPOINTS


def quadratic_problems(g, B, n, seed, bound=False):
    """B seeded instances on the box of grid g.  bound=True puts the guide points 0.5 m above the box, which pushes
    the minimiser onto its ceiling (every instance from n = 8 on; about half at n = 7, where one guide point competes
    with the START and END terms).  The waypoints include the last legal index (idx + 2 == n - 1)."""
    rng = np.random.default_rng(seed)
    bmin, bmax = np.asarray(g.box_min, np.float64), np.asarray(g.box_max, np.float64)
    lo, hi = bmin + 1.0, bmax - 1.0
    out = []
    for _ in range(B):
        while True:
            s = rng.uniform(lo, hi)
            d = rng.normal(size=3)
            d[2] *= 0.15
            d /= np.linalg.norm(d)
            e = s + d * 0.35 * (n - 1)
            if np.all(e > lo) and np.all(e < hi):
                break
        t = np.linspace(0.0, 1.0, n)[:, None]
        line = s * (1 - t) + e * t
        dt = rng.uniform(0.8, 1.2)
        st, en = W.cubic_boundary_states(line, dt)
        start = st + rng.normal(scale=0.2, size=(3, 3))
        end = np.stack([en, (line[-1] - line[-3]) / (2 * dt), np.zeros(3)]) + rng.normal(scale=0.2, size=(3, 3))
        guide = line[3:n - 3] + rng.normal(scale=0.3, size=(n - 6, 3))
        if bound:
            guide[:, 2] = bmax[2] + 0.5
        widx = sorted({0, n // 2 - 1, n - 3})
        waypt = line[[i + 1 for i in widx]] + rng.normal(scale=0.3, size=(len(widx), 3))
        x0 = np.clip(line + rng.normal(scale=0.5, size=line.shape), bmin + 0.1, bmax - 0.1)
        acc = 0.0
        for v in np.sqrt(np.sum((x0[1:] - x0[:-1]) ** 2, axis=1)):  # pt_dist_ (:136-140)
            acc += v
        out.append(dict(x0=x0.reshape(-1), dt=dt, start=start, end=end, guide=guide, waypt=waypt, widx=widx,
                        pt_dist=acc / n))
    return out


def quad_consts(fill, arr, problems):
    """Fill a ctypes array of trajectory constants (oracle or library layout) with `fill` (fill_traj_const)."""
    for b, q in enumerate(problems):
        fill(arr[b], q["pt_dist"], q["dt"], q["start"], q["end"], -1.0, q["guide"], q["waypt"], q["widx"])
    return arr


def quad_minimisers(orc, og, params, tcs, n, problems, g):
    """The exact minimiser of every instance: the Hessian from the oracle's (affine) gradient, one column per unit
    vector; numpy.linalg.solve when the minimiser is inside the solver's bounds, otherwise the bound-constrained
    least-squares form 1/2 |L^T x + L^-1 c|^2 (H = L L^T) with scipy's BVLS.  Returns (x* [B, 3n], bound [B])."""
    import scipy.linalg as sl
    from scipy.optimize import lsq_linear
    nv = 3 * n
    mask = quad_mask(orc)
    bmin = np.tile(np.asarray(g.box_min, np.float64) + 0.1, n)
    bmax = np.tile(np.asarray(g.box_max, np.float64) - 0.1, n)
    xs, bound = [], []
    for b, q in enumerate(problems):
        X = np.repeat(q["x0"][None, :], nv + 1, axis=0)
        X[1:] += np.eye(nv)
        tb = orc.traj_consts(nv + 1)
        for i in range(nv + 1):
            tb[i] = tcs[b]
        _, gr = orc.combine_cost_batch(og, np.zeros(1), params, tb, n, mask, X)
        H = (gr[1:] - gr[0]).T
        H = 0.5 * (H + H.T)
        c = gr[0] - H @ q["x0"]
        xu = np.linalg.solve(H, -c)
        c0 = np.clip(q["x0"], bmin, bmax)  # the solver's bounds (optimize() :196-217)
        lb, ub = np.maximum(c0 - 10.0, bmin), np.minimum(c0 + 10.0, bmax)
        if np.all(xu >= lb) and np.all(xu <= ub):
            xs.append(xu)
            bound.append(False)
        else:
            L = np.linalg.cholesky(H)
            r = lsq_linear(L.T, -sl.solve_triangular(L, c, lower=True), bounds=(lb, ub), method="bvls", tol=1e-15)
            xs.append(r.x)
            bound.append(True)
    return np.stack(xs), np.array(bound)
