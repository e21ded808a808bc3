"""The device solver (fuelgpu_bspline_optimize_batch) step by step against its fp64 CPU twin (oracle.optimize_batch),
for both kernels: optimize_gram_kernel (lbfgs_m == 6, the benchmark's) and optimize_warp_kernel (every other history
length, or FUELGPU_SOLVER=vec).

(a) a convex quadratic whose minimiser linear algebra gives exactly;
(b) non-convex objectives, where the device must take the twin's path wherever the twin's branch decisions are
    clear of the device's rounding -- same evaluation count, same best point;
(c) the two kernels against each other at lbfgs_m = 6;
(d) the device-pointer entry points the benchmark calls;
(e) argument edges.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests.helpers import (QUAD_WEIGHTS, make_sdf_map, orc_grid, quad_consts, quad_mask, quad_minimisers,
                           quadratic_problems)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def scene(fuel, orc):
    g, inflate = W.office_map()
    tri = W.office_known(g, inflate)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    d32 = m.download().copy()
    env = fuel.EDTEnvironment()
    env.setMap(m)
    yield dict(g=g, inflate=inflate, m=m, env=env, og=orc_grid(orc, g), d32=d32,
               # the twin samples the device's own fp32 field widened to fp64: the field is then not a difference
               dw=d32.astype(np.float64))
    m.close()


def optimizer(fuel, scene, **params):
    opt = fuel.BsplineOptimizer()
    opt.setEnvironment(scene["env"])
    opt.setParam(**params)
    return opt


# ---------------------------------------------------------------------------------------------------------------------
# (a) convergence on the quadratic
# ---------------------------------------------------------------------------------------------------------------------
_QUAD = {}


def quad_case(fuel, orc, scene, n, bound):
    key = (n, bound)
    if key not in _QUAD:
        g = scene["g"]
        P = quadratic_problems(g, 1027, n, 100 + n, bound=bound)
        par = orc.opt_params(**QUAD_WEIGHTS)
        to = quad_consts(orc.fill_traj_const, orc.traj_consts(len(P)), P)
        tg = quad_consts(fuel.BsplineOptimizer.fill_traj_const, (fuel._lib.FuelTrajConst * len(P))(), P)
        xs, is_bound = quad_minimisers(orc, scene["og"], par, to, n, P, g)
        _QUAD[key] = (par, to, tg, xs, is_bound, np.stack([q["x0"] for q in P]))
    return _QUAD[key]


@pytest.mark.parametrize("bound", [False, True], ids=["interior", "box_bound"])
@pytest.mark.parametrize("n", [7, 8, 20, 31, 32])
def test_quadratic_reaches_minimiser(fuel, orc, scene, n, bound):
    """Every history length 1..8 (both kernels), B = 1, 5 and 1027 (a partial last block of WPB = 4 warps), interior
    and box-bound minimisers, max_eval = 2000 with the default xtol_rel.  The bar is the twin's (tests/
    test_oracle_solver.py): within 1e-3 m of x*, cost within 1e-6 of the minimum; f_best is the cost at x_best.
    Measured on a B200: at most 7.5e-4 m from x* over all cases (the xtol stop, as for the twin)."""
    par, to, tg, xs, is_bound, X0 = quad_case(fuel, orc, scene, n, bound)
    # (a few of the unpushed instances have their minimiser outside the box too: the bar is the same)
    if bound and n >= 8:
        assert is_bound.all()
    if not bound:
        assert is_bound.mean() < 0.05
    opt = optimizer(fuel, scene, **QUAD_WEIGHTS)
    mask = quad_mask(fuel.BsplineOptimizer)
    fs, _ = orc.combine_cost_batch(scene["og"], np.zeros(1), par, to, n, mask, xs, threads=8)
    worst = 0.0
    for m in range(1, 9):
        for B in (1, 5, 1027):
            x, f, ne = opt.optimizeBatch(X0[:B], tg, n, mask, 2000, lbfgs_m=m)
            err = np.max(np.abs(x - xs[:B]))
            worst = max(worst, err)
            assert err < 1e-3, (m, B, err)
            assert np.all(np.abs(f - fs[:B]) <= 1e-6 * np.abs(fs[:B])), (m, B)
            assert np.all(ne <= 2000) and np.all(ne >= 2)
            fo, _ = orc.combine_cost_batch(scene["og"], np.zeros(1), par, to, n, mask, x, threads=8)
            assert np.all(np.abs(fo - f) <= 1e-12 * np.abs(fo)), (m, B, np.max(np.abs(fo - f) / np.abs(fo)))
    print("n=%d %s: max |x_best - x*| %.3g m" % (n, "bound" if bound else "interior", worst))


# ---------------------------------------------------------------------------------------------------------------------
# (b) step-level parity on non-convex objectives
# ---------------------------------------------------------------------------------------------------------------------
N_PTS = 20
B_PAR = 4096
KS = (2, 3, 5, 8, 13, 21, 34, 64)
OBJECTIVES = {  # name -> (setParam overrides, MINTIME?)
    "bench": ({}, True),
    "normal_fixed_dt": ({}, False),
    "ld100_d1.5": (dict(ld_dist=100.0, dist0=1.5), True),
    "ld300_d2.0": (dict(ld_dist=300.0, dist0=2.0), True),
}
# tau = TAU_FACTOR * eps.  eps is the fast evaluator's relative cost disagreement with the twin at the same x; the
# device's own solver arithmetic (fp32 warp reductions, fp32 Gram data and direction) moves its iterates off the
# twin's by ~1e-7 relative per step on top of that, and a decision is only reproducible when its margin clears both
# by a wide factor.
TAU_FACTOR = 100.0
TAU_FLOOR = 1e-6
_PAR = {}


def parity_inputs(fuel, orc, scene):
    if "tr" not in _PAR:
        tr = W.make_trajectories(scene["g"], scene["inflate"], B=B_PAR, n_pts=N_PTS, seed=4242)
        to = orc.traj_consts(B_PAR)
        for b in range(B_PAR):
            orc.fill_traj_const(to[b], tr["pt_dist"][b], tr["dt"][b], tr["start"][b], tr["end_pos"][b][None, :])
        tg = fuel.BsplineOptimizer.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"])
        _PAR.update(tr=tr, to=to, tg=tg)
    return _PAR["tr"], _PAR["to"], _PAR["tg"]


def twin_runs(orc, scene, to, name, x0, mask, m, exact):
    key = (name, m, exact)
    if key not in _PAR:
        par = orc.opt_params(**OBJECTIVES[name][0])
        out = {}
        for K in KS:
            xc, fc, nc, tr = orc.optimize_batch(scene["og"], scene["dw"], par, to, N_PTS, mask, x0, max_eval=K,
                                                lbfgs_m=m, exact_evals=exact, trace=True, threads=8)
            out[K] = (xc, fc, nc, tr)
        _PAR[key] = out
    return _PAR[key]


def evaluator_eps(opt, orc, scene, par, to, tg, mask, xs):
    """eps: max relative disagreement of the fast evaluator (what the solver loop runs) with the twin's evaluator,
    over the given points."""
    eps = 0.0
    for x in xs:
        f, _ = opt.combineCostBatch(x, tg, N_PTS, mask, fast_eval=True)
        fr, _ = orc.combine_cost_batch(scene["og"], scene["dw"], par, to, N_PTS, mask, x, threads=8)
        eps = max(eps, float(np.max(np.abs(f - fr) / np.abs(fr))))
    return eps


def compare_runs(opt_run, twin, K, tau):
    """-> dict of counts and agreement over the trajectories that qualify at K."""
    xg, fg, ng = opt_run
    xc, fc, nc, tr = twin
    q = tr["margin"][:, K - 1] >= tau
    full = q & (tr["first_full_reject"] >= 0) & (tr["first_full_reject"] < K)
    rst = q & (tr["first_ls_fail"] >= 0) & (tr["first_ls_fail"] < K)
    dx = np.max(np.abs(xg - xc), axis=1)
    df = np.abs(fg - fc) / np.abs(fc)
    close = (dx <= DX_TOL) & (df <= DF_TOL)
    return dict(K=K, n=int(q.sum()), frac=float(q.mean()), full=int(full.sum()), restart=int(rst.sum()),
                restart_all=int(((tr["first_ls_fail"] >= 0) & (tr["first_ls_fail"] < K)).sum()),
                neval_mismatch=int(np.sum(q & (ng != nc))),
                close=float(np.mean(close[q])) if q.any() else 1.0,
                close_full=float(np.mean(close[full])) if full.any() else 1.0,
                dx_q=np.quantile(dx[q], [0.5, 0.9, 0.99, 1.0]) if q.any() else np.zeros(4),
                dx_full=np.quantile(dx[full], [0.5, 0.9, 1.0]) if full.any() else np.zeros(3))


# Qualifying trajectories take the twin's branches; what is left between the two is the rounding of the path (fast
# evaluator, fp32 solver scalars), which the iterations amplify: measured on a B200 over 4096 trajectories, the share
# of qualifying trajectories within DX_TOL and DF_TOL of the twin is 1.0 up to K = 8, >= 0.98 at 13, >= 0.90 at 21,
# >= 0.52 at 34 and 0.01 .. 0.26 at 64 (cm-level drift after 64 non-convex steps).  So the bars are on that share,
# with K = 64 checked for branch parity only.
DX_TOL = 1e-3   # metres (and seconds, for dt)
DF_TOL = 1e-4   # relative
CLOSE_FLOOR = {2: 0.99, 3: 0.99, 5: 0.99, 8: 0.99, 13: 0.97, 21: 0.85, 34: 0.4, 64: 0.0}
# least qualifying fraction per K (margins shrink as the trajectories converge: late line searches compare costs that
# agree to many digits; measured minima 1.0 / 0.98 / 0.90 / 0.66 / 0.16 at K <= 8 / 13 / 21 / 34 / 64)
FRAC_FLOOR = {2: 0.9, 3: 0.9, 5: 0.9, 8: 0.9, 13: 0.85, 21: 0.7, 34: 0.5, 64: 0.1}
# Trajectories whose curvature test refused a pair while the ring was full, K = 13 and 21 together: measured share
# within the bars 0.86 .. 1.0 for every kernel; 0.03 .. 0.14 for a coefficient-space kernel that leaves the oldest
# pair's s.pg, y.pg stale after such a refusal.
FULL_RING_KS = (13, 21)
FULL_RING_FLOOR = 0.7


def run_parity(fuel, orc, scene, m, device_runs=None):
    tr, to, tg = parity_inputs(fuel, orc, scene)
    rows = []
    for name, (over, mintime) in OBJECTIVES.items():
        O = fuel.BsplineOptimizer
        mask = O.NORMAL_PHASE | (O.MINTIME if mintime else 0)
        x0 = W.pack_x(tr["ctrl"], tr["dt"], mintime=mintime)
        opt = optimizer(fuel, scene, **over)
        par = orc.opt_params(**over)
        for exact in (False, True):
            twin = twin_runs(orc, scene, to, name, x0, mask, m, exact)
            eps = evaluator_eps(opt, orc, scene, par, to, tg, mask, [x0, twin[64][0]])
            tau = max(TAU_FACTOR * eps, TAU_FLOOR)
            for K in KS:
                if device_runs is None:
                    run = opt.optimizeBatch(x0, tg, N_PTS, mask, K, lbfgs_m=m, exact_evals=exact,
                                            xtol_rel=0.0 if exact else 1e-5)
                else:
                    run = device_runs[(name, exact, K)]
                r = compare_runs(run, twin[K], K, tau)
                r.update(obj=name, exact=exact, eps=eps, tau=tau)
                rows.append(r)
    return rows


def report(rows, label):
    for r in rows:
        print("%s %-16s %-6s K=%2d eps=%.2e tau=%.2e qualify %4d (%.3f) full-ring %3d restart %3d/%3d  "
              "n_eval mismatches %d  close %.4f (full-ring %.4f)  |dx| q50/90/99/max %s  full-ring q50/90/max %s"
              % (label, r["obj"], "exact" if r["exact"] else "normal", r["K"], r["eps"], r["tau"], r["n"], r["frac"],
                 r["full"], r["restart"], r["restart_all"], r["neval_mismatch"], r["close"], r["close_full"],
                 " ".join("%.1e" % v for v in r["dx_q"]), " ".join("%.1e" % v for v in r["dx_full"])))


def assert_parity(rows):
    for r in rows:
        key = (r["obj"], r["exact"], r["K"])
        # normal mode can stop early on xtol once the paths have drifted (K = 64: at most 6 of 630 measured)
        assert r["neval_mismatch"] <= 0.02 * r["n"], (key, r["neval_mismatch"], r["n"])
        assert r["close"] >= CLOSE_FLOOR[r["K"]], (key, r["close"])
        assert r["frac"] >= FRAC_FLOOR[r["K"]], (key, r["frac"])
    # the rare branch was exercised by enough qualifying trajectories, and they followed the twin
    full = [r for r in rows if r["K"] in FULL_RING_KS]
    n_full = sum(r["full"] for r in full)
    assert n_full >= 10, n_full
    share = sum(r["full"] * r["close_full"] for r in full) / n_full
    print("full-ring refusals before K in %s: %d qualifying, %.3f within the bars; exact-mode restarts: %d trajectories, "
          "%d qualifying" % (FULL_RING_KS, n_full, share, sum(r["restart_all"] for r in rows),
                             sum(r["restart"] for r in rows)))
    assert share >= FULL_RING_FLOOR, share


@pytest.mark.parametrize("m", [6, 3, 8], ids=["gram_m6", "vec_m3", "vec_m8"])
def test_step_parity_with_twin(fuel, orc, scene, m):
    """Objectives: the bench objective, NORMAL_PHASE with a fixed knot span, and two strong-distance settings that
    make the curvature test refuse pairs while the history ring is full.  Both modes, K = 2 .. 64.
    A failed line search (exact mode restarts after one) never qualifies: it is some 40 halvings whose Armijo tests
    compare costs below the fast evaluator's rounding.  Such trajectories are counted, not compared."""
    rows = run_parity(fuel, orc, scene, m)
    report(rows, "m=%d" % m)
    assert_parity(rows)


# ---------------------------------------------------------------------------------------------------------------------
# (c) gram kernel vs vector kernel at lbfgs_m = 6
# ---------------------------------------------------------------------------------------------------------------------
_CHILD = r"""
import sys, ctypes as C, numpy as np
sys.path.insert(0, sys.argv[1])
import fuel_b200
from fuel_b200 import workloads as W
from fuel_b200._lib import FuelTrajConst
inp = np.load(sys.argv[2], allow_pickle=True)
g, inflate = W.office_map()
tri = W.office_known(g, inflate)
m = fuel_b200.SDFMap(g.n, g.res, g.origin, g.box_min, g.box_max, optimistic=True)
m.occupancy_buffer_inflate_[...] = inflate
m.setOccupancyBuffer(tristate=tri)
m.upload()
m.updateESDF3d()
assert np.array_equal(m.download(), inp["d32"])
env = fuel_b200.EDTEnvironment()
env.setMap(m)
tcb = inp["tcs"]
tg = (FuelTrajConst * (tcb.size // C.sizeof(FuelTrajConst))).from_buffer_copy(tcb.tobytes())
out = {}
for job in inp["jobs"]:
    name, over, mintime, exact, K = job
    opt = fuel_b200.BsplineOptimizer()
    opt.setEnvironment(env)
    opt.setParam(**over)
    mask = opt.NORMAL_PHASE | (opt.MINTIME if mintime else 0)
    x0 = inp["x0_%d" % int(mintime)]
    x, f, n = opt.optimizeBatch(x0, tg, 20, mask, int(K), lbfgs_m=6, exact_evals=bool(exact),
                                xtol_rel=0.0 if exact else 1e-5)
    key = "%s|%d|%d" % (name, int(exact), int(K))
    out["x|" + key], out["f|" + key], out["n|" + key] = x, f, n
m.close()
np.savez(sys.argv[3], **out)
"""


def test_vector_kernel_matches_gram_kernel(fuel, orc, scene, tmp_path):
    """FUELGPU_SOLVER=vec (read once per process, so in a child process) runs optimize_warp_kernel at lbfgs_m = 6.
    Both kernels must follow the twin under the bars of test_step_parity_with_twin, and agree with each other on the
    trajectories that qualify up to K = 21 (beyond, both have drifted from the twin by the amplified rounding)."""
    tr, to, tg = parity_inputs(fuel, orc, scene)
    jobs = [(name, over, mintime, exact, K) for name, (over, mintime) in OBJECTIVES.items()
            for exact in (False, True) for K in KS]
    inp = tmp_path / "in.npz"
    np.savez(inp, d32=scene["d32"], tcs=np.frombuffer(tg, dtype=np.uint8),
             x0_0=W.pack_x(tr["ctrl"], tr["dt"], mintime=False), x0_1=W.pack_x(tr["ctrl"], tr["dt"]),
             jobs=np.array(jobs, dtype=object))
    out = tmp_path / "vec.npz"
    env = dict(os.environ, FUELGPU_SOLVER="vec")
    subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(inp), str(out)], env=env, check=True, timeout=900)
    res = np.load(out)
    runs = {}
    for name, over, mintime, exact, K in jobs:
        key = "%s|%d|%d" % (name, int(exact), K)
        runs[(name, exact, K)] = (res["x|" + key], res["f|" + key], res["n|" + key])
    vec_rows = run_parity(fuel, orc, scene, 6, device_runs=runs)
    report(vec_rows, "vec m=6")
    assert_parity(vec_rows)
    gram_rows = run_parity(fuel, orc, scene, 6)
    # and directly: where both kernels qualify, they agree with each other to twice the bar
    for rv, rg in zip(vec_rows, gram_rows):
        assert rv["n"] == rg["n"]
    for name, over, mintime, exact, K in jobs:
        O = fuel.BsplineOptimizer
        mask = O.NORMAL_PHASE | (O.MINTIME if mintime else 0)
        x0 = W.pack_x(tr["ctrl"], tr["dt"], mintime=mintime)
        opt = optimizer(fuel, scene, **over)
        xg, fg, ng = opt.optimizeBatch(x0, tg, N_PTS, mask, K, lbfgs_m=6, exact_evals=exact,
                                       xtol_rel=0.0 if exact else 1e-5)
        xv, fv, nv = runs[(name, exact, K)]
        assert not np.array_equal(xg, xv) or K <= 2, "FUELGPU_SOLVER=vec did not switch kernels"
        if K > 21:
            continue
        twin = _PAR[(name, 6, exact)][K]
        tau = [r["tau"] for r in gram_rows if r["obj"] == name and r["exact"] == exact and r["K"] == K][0]
        q = twin[3]["margin"][:, K - 1] >= tau
        assert np.array_equal(ng[q], nv[q])
        close = np.max(np.abs(xg[q] - xv[q]), axis=1) <= 2 * DX_TOL
        assert np.mean(close) >= CLOSE_FLOOR[K] if q.any() else True


# ---------------------------------------------------------------------------------------------------------------------
# (d) the device-pointer entry points (what bench.py calls)
# ---------------------------------------------------------------------------------------------------------------------
def test_device_entry_points_equal_host_ones(fuel, orc, scene):
    """fuelgpu_bspline_optimize_batch_dev and fuelgpu_bspline_cost_batch_dev on torch device tensors, built as the
    benchmark's planner builds them, give the bits of the host-buffer entry points."""
    import torch
    L = fuel.lib()
    O = fuel.BsplineOptimizer
    h = scene["m"].handle
    opt = optimizer(fuel, scene)
    dev = "cuda:%d" % torch.cuda.current_device()
    for n, B in ((20, 1027), (7, 5), (32, 64), (47, 33)):
        tr = W.make_trajectories(scene["g"], scene["inflate"], B=B, n_pts=n, seed=n, spacing=0.35 if n <= 32 else 0.2)
        tg = O.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"])
        d_tc = torch.from_numpy(np.frombuffer(tg, dtype=np.uint8).copy()).to(dev)
        for mask in (O.NORMAL_PHASE | O.MINTIME, O.NORMAL_PHASE):
            x0 = W.pack_x(tr["ctrl"], tr["dt"], mintime=bool(mask & O.MINTIME))
            nvar = x0.shape[1]
            d_x = torch.from_numpy(x0).to(dev)
            d_f = torch.empty(B, dtype=torch.float64, device=dev)
            d_g = torch.empty((B, nvar), dtype=torch.float64, device=dev)
            for fast in ((False, True) if n <= 32 else (False,)):
                mk = mask | (fuel.bspline_optimizer.COST_FAST_EVAL if fast else 0)
                rc = L.fuelgpu_bspline_cost_batch_dev(h, B, n, mk, C.byref(opt.params_), C.c_void_p(d_tc.data_ptr()),
                                                      C.c_void_p(d_x.data_ptr()), C.c_void_p(d_f.data_ptr()),
                                                      C.c_void_p(d_g.data_ptr()))
                assert rc == 0, L.fuelgpu_last_error(h)
                torch.cuda.synchronize()
                f, g = opt.combineCostBatch(x0, tg, n, mask, fast_eval=fast)
                assert np.array_equal(d_f.cpu().numpy(), f) and np.array_equal(d_g.cpu().numpy(), g)
            if n + int(bool(mask & O.MINTIME)) > 32:
                continue
            for exact in (False, True):
                sp = fuel._lib.FuelSolveParams()
                sp.max_eval, sp.lbfgs_m, sp.xtol_rel, sp.flags = 64, 6, 0.0 if exact else 1e-5, int(exact)
                d_xw = d_x.clone()
                d_n = torch.empty(B, dtype=torch.int32, device=dev)
                rc = L.fuelgpu_bspline_optimize_batch_dev(h, B, n, mask, C.byref(opt.params_),
                                                          C.c_void_p(d_tc.data_ptr()), C.byref(sp),
                                                          C.c_void_p(d_xw.data_ptr()), C.c_void_p(d_f.data_ptr()),
                                                          C.c_void_p(d_n.data_ptr()))
                assert rc == 0, L.fuelgpu_last_error(h)
                torch.cuda.synchronize()
                xh, fh, nh = opt.optimizeBatch(x0, tg, n, mask, 64, exact_evals=exact, xtol_rel=sp.xtol_rel)
                assert np.array_equal(d_xw.cpu().numpy(), xh)
                assert np.array_equal(d_f.cpu().numpy(), fh) and np.array_equal(d_n.cpu().numpy(), nh)


# ---------------------------------------------------------------------------------------------------------------------
# (e) argument edges
# ---------------------------------------------------------------------------------------------------------------------
def test_solver_argument_edges(fuel, orc, scene):
    """n_pts + dt must fit the 32 lanes of a warp; history length 1..8; max_eval >= 1; an empty batch is a no-op."""
    O = fuel.BsplineOptimizer
    opt = optimizer(fuel, scene)
    for n, mask, ok in ((31, O.NORMAL_PHASE | O.MINTIME, True), (32, O.NORMAL_PHASE | O.MINTIME, False),
                        (32, O.NORMAL_PHASE, True)):
        tr = W.make_trajectories(scene["g"], scene["inflate"], B=6, n_pts=n, seed=n)
        tg = O.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"])
        x0 = W.pack_x(tr["ctrl"], tr["dt"], mintime=bool(mask & O.MINTIME))
        if ok:
            x, f, ne = opt.optimizeBatch(x0, tg, n, mask, 16)
            f0, _ = opt.combineCostBatch(x0, tg, n, mask)
            assert np.all(ne >= 2) and np.all(f <= f0 * (1 + 1e-9))
        else:
            with pytest.raises(fuel.FuelGpuError) as e:
                opt.optimizeBatch(x0, tg, n, mask, 16)
            assert e.value.code == fuel._lib.EUNSUPPORTED
    tr = W.make_trajectories(scene["g"], scene["inflate"], B=4, n_pts=20, seed=1)
    tg = O.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"])
    x0 = W.pack_x(tr["ctrl"], tr["dt"])
    mask = O.NORMAL_PHASE | O.MINTIME
    for kw in (dict(lbfgs_m=0), dict(lbfgs_m=9), dict(max_eval=0)):
        args = dict(lbfgs_m=6, max_eval=16)
        args.update(kw)
        with pytest.raises(fuel.FuelGpuError) as e:
            opt.optimizeBatch(x0, tg, 20, mask, args["max_eval"], lbfgs_m=args["lbfgs_m"])
        assert e.value.code == fuel._lib.EINVAL
    # B = 0: nothing runs and nothing is written
    out = (np.full((0, 61), 7.0), np.full(0, 7.0), np.full(0, 7, dtype=np.int32))
    x, f, ne = opt.optimizeBatch(x0[:0], tg, 20, mask, 16, out=out)
    assert x.shape == (0, 61) and f.shape == (0,) and ne.shape == (0,)
    sentinel = np.full(3, 7.0)
    rc = fuel.lib().fuelgpu_bspline_optimize_batch(scene["m"].handle, 0, 20, mask, C.byref(opt.params_), tg,
                                                    C.byref(fuel._lib.FuelSolveParams(16, 6, 1e-5, 0, 0)),
                                                    sentinel.ctypes.data_as(C.c_void_p), None, None)
    assert rc == 0 and np.all(sentinel == 7.0)
