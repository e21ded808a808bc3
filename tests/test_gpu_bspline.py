"""B-spline cost/gradient parity: fuelgpu_bspline_cost_batch vs the CPU oracle of
BsplineOptimizer::combineCost (bspline_opt/src/bspline_optimizer.cpp:518-647).
Tolerance (north_star): 1e-4 relative on cost and gradient."""
import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests.helpers import make_sdf_map, orc_grid

pytestmark = pytest.mark.gpu
RTOL = 1e-4


@pytest.fixture(scope="module")
def scene(fuel, orc):
    g, inflate = W.office_map()
    tri = W.office_known(g, inflate)
    m = make_sdf_map(fuel, g, inflate, tri, optimistic=True)
    m.updateESDF3d()
    d32 = m.download().copy()
    env = fuel.EDTEnvironment()
    env.setMap(m)
    opt = fuel.BsplineOptimizer()
    opt.setEnvironment(env)
    # the oracle reads the reference's own fp64 field (resolution*sqrt(int) in double)
    d64 = orc.update_esdf3d(orc_grid(orc, g), inflate, tri, [0, 0, 0], np.array(g.n) - 1, True, False, threads=8)
    yield dict(g=g, inflate=inflate, m=m, opt=opt, d32=d32, d64=d64)
    m.close()


def orc_consts(orc, tr, B, guide=None, waypt=None, waypt_idx=None, n_end=1, time_lb=None):
    tcs = orc.traj_consts(B)
    for b in range(B):
        end = np.zeros((n_end, 3))
        end[0] = tr["end_pos"][b]
        orc.fill_traj_const(tcs[b], tr["pt_dist"][b], tr["dt"][b], tr["start"][b], end,
                            -1.0 if time_lb is None else time_lb[b],
                            None if guide is None else guide[b], None if waypt is None else waypt[b], waypt_idx)
    return tcs


def gpu_consts(fuel, tr, B, guide=None, waypt=None, waypt_idx=None, n_end=1, time_lb=None):
    from fuel_b200._lib import FuelTrajConst
    tcs = (FuelTrajConst * B)()
    for b in range(B):
        end = np.zeros((n_end, 3))
        end[0] = tr["end_pos"][b]
        fuel.BsplineOptimizer.fill_traj_const(tcs[b], tr["pt_dist"][b], tr["dt"][b], tr["start"][b], end,
                                              -1.0 if time_lb is None else time_lb[b],
                                              None if guide is None else guide[b],
                                              None if waypt is None else waypt[b], waypt_idx)
    return tcs


def check(f, g, fr, gr):
    assert np.all(np.abs(f - fr) <= RTOL * np.abs(fr) + 1e-12), np.max(np.abs(f - fr) / np.abs(fr))
    scale = np.max(np.abs(gr), axis=1, keepdims=True)
    err = np.abs(g - gr)
    # every component within 1e-4 of its own magnitude, with the trajectory's gradient
    # scale as the floor for components that cancel to ~0
    assert np.all(err <= RTOL * np.maximum(np.abs(gr), 1e-3 * scale) + 1e-12), np.max(err / scale)


def test_benchmark_objective(fuel, orc, scene):
    """NORMAL_PHASE | MINTIME (the exploration objective, planner_manager.cpp:304-305) on the
    config-2 batch."""
    B, N = 1024, 20
    tr = W.make_trajectories(scene["g"], scene["inflate"], B=B, n_pts=N)
    mask = fuel.BsplineOptimizer.NORMAL_PHASE | fuel.BsplineOptimizer.MINTIME
    x = W.pack_x(tr["ctrl"], tr["dt"])
    f, g = scene["opt"].combineCostBatch(x, gpu_consts(fuel, tr, B), N, mask)
    fr, gr = orc.combine_cost_batch(orc_grid(orc, scene["g"]), scene["d64"], orc.opt_params(),
                                    orc_consts(orc, tr, B), N, mask, x, threads=8)
    check(f, g, fr, gr)
    # the distance term must be active for a realistic share of control points (SURVEY 8d)
    d, _ = scene["m"].getDistWithGrad(tr["ctrl"].reshape(-1, 3))
    frac = np.mean(d < 0.7)
    assert 0.15 < frac < 0.8, frac
    # vectorised constant builder gives the same bytes as the field-by-field one
    arr = fuel.BsplineOptimizer.traj_consts_from_arrays(tr["pt_dist"], tr["dt"], tr["start"], tr["end_pos"])
    f2, g2 = scene["opt"].combineCostBatch(x, arr, N, mask)
    assert np.array_equal(f, f2) and np.array_equal(g, g2)


# control-point counts: 7, 8, 31, 32 run the warp kernels (one lane per point; 7 has a single interior segment,
# 32 fills the warp), 33 .. 64 the thread kernel, which only the faithful evaluator has
N_WARP = [7, 8, 20, 31, 32]
N_THREAD = [33, 47, 64]


def trajectories(scene, B, n, seed):
    # lines longer than the 0.35 m spacing allows inside the 18 m x 10 m box would never be drawn
    return W.make_trajectories(scene["g"], scene["inflate"], B=B, n_pts=n, seed=seed, spacing=0.35 if n <= 32 else 0.2)


def check_both(fuel, opt, x, tg, n, mask, fr, gr):
    """the faithful evaluator (both kernels) and, where it exists (n <= 32), the solver's fast one"""
    f, g = opt.combineCostBatch(x, tg, n, mask)
    check(f, g, fr, gr)
    if n <= 32:
        f, g = opt.combineCostBatch(x, tg, n, mask, fast_eval=True)
        check(f, g, fr, gr)
    else:
        with pytest.raises(fuel.FuelGpuError) as e:
            opt.combineCostBatch(x, tg, n, mask, fast_eval=True)
        assert e.value.code == fuel._lib.EUNSUPPORTED


@pytest.mark.parametrize("n_pts", N_WARP + N_THREAD)
@pytest.mark.parametrize("mask_name", ["SMOOTHNESS", "DISTANCE", "FEASIBILITY", "START", "END", "MINTIME",
                                       "NORMAL_PHASE"])
def test_single_terms(fuel, orc, scene, mask_name, n_pts):
    B, N = 64, n_pts
    tr = trajectories(scene, B, N, seed=5)
    O = fuel.BsplineOptimizer
    mask = getattr(O, mask_name)
    if mask_name == "MINTIME":
        mask |= O.SMOOTHNESS
    x = W.pack_x(tr["ctrl"], tr["dt"], mintime=bool(mask & O.MINTIME))
    # make feasibility bite: shrink dt for half of the batch
    if mask & O.MINTIME:
        x[::2, -1] *= 0.5
    else:
        tr["dt"][::2] *= 0.5
    fr, gr = orc.combine_cost_batch(orc_grid(orc, scene["g"]), scene["d64"], orc.opt_params(),
                                    orc_consts(orc, tr, B), N, mask, x)
    check_both(fuel, scene["opt"], x, gpu_consts(fuel, tr, B), N, mask, fr, gr)


def test_guide_waypoints_end3_timelb(fuel, orc, scene):
    """GUIDE_PHASE, WAYPOINTS (one at the last legal index, idx + 2 == N - 1), a 3-entry end_state_ and an active
    time lower bound, at 24 control points."""
    guide_waypoints_end3_timelb(fuel, orc, scene, 24)


@pytest.mark.parametrize("n_pts", [7, 8, 31, 32] + N_THREAD)
def test_guide_waypoints_end3_timelb_n_pts(fuel, orc, scene, n_pts):
    """The same at the warp kernels' edges and on the thread kernel."""
    guide_waypoints_end3_timelb(fuel, orc, scene, n_pts)


def guide_waypoints_end3_timelb(fuel, orc, scene, n_pts):
    B, N = 32, n_pts
    tr = trajectories(scene, B, N, seed=9)
    O = fuel.BsplineOptimizer
    rng = np.random.default_rng(3)
    guide = tr["ctrl"][:, 3:N - 3] + rng.normal(scale=0.2, size=(B, N - 6, 3))
    widx = sorted({i for i in (0, 4, 9) if i < N - 3} | {N - 3})
    waypt = rng.uniform(-1, 1, size=(B, len(widx), 3)) + tr["ctrl"][:, [i + 1 for i in widx]]
    time_lb = (N - 3) * tr["dt"] * 1.3
    for mask, n_end in ((O.GUIDE_PHASE, 1), (O.SMOOTHNESS | O.WAYPOINTS, 1), (O.NORMAL_PHASE | O.MINTIME, 3),
                        (O.SMOOTHNESS | O.WAYPOINTS | O.START | O.END, 2)):
        if N + int(bool(mask & O.MINTIME)) > 64:
            continue
        x = W.pack_x(tr["ctrl"], tr["dt"], mintime=bool(mask & O.MINTIME))
        kw = dict(guide=guide, waypt=waypt, waypt_idx=widx, n_end=n_end, time_lb=time_lb)
        tg = gpu_consts(fuel, tr, B, **kw)
        to = orc_consts(orc, tr, B, **kw)
        if n_end > 1:
            for b in range(B):
                for i in range(1, n_end):
                    for k in range(3):
                        v = float(rng.normal())
                        tg[b].end[i][k] = v
                        to[b].end[i][k] = v
        fr, gr = orc.combine_cost_batch(orc_grid(orc, scene["g"]), scene["d64"], orc.opt_params(), to, N, mask, x)
        check_both(fuel, scene["opt"], x, tg, N, mask, fr, gr)


def test_adversarial_positions(fuel, orc, scene):
    """Control points on the map boundary, outside the map, and in flat ESDF regions."""
    B, N = 48, 20
    g = scene["g"]
    tr = W.make_trajectories(g, scene["inflate"], B=B, n_pts=N, seed=13)
    ctrl = tr["ctrl"].copy()
    ctrl[0:8, 5] = g.origin + [0.02, 0.5, 0.5]        # stencil pokes outside the map
    ctrl[8:16, 7] = g.map_max + 0.3                   # outside the map -> (0, 0-grad)
    ctrl[16:24, 9] = g.map_max - [1e-4, 0.5, 0.5]     # the isInMap margin
    tr["ctrl"] = ctrl
    O = fuel.BsplineOptimizer
    mask = O.NORMAL_PHASE | O.MINTIME
    x = W.pack_x(ctrl, tr["dt"])
    f, gg = scene["opt"].combineCostBatch(x, gpu_consts(fuel, tr, B), N, mask)
    fr, gr = orc.combine_cost_batch(orc_grid(orc, g), scene["d64"], orc.opt_params(), orc_consts(orc, tr, B), N,
                                    mask, x)
    check(f, gg, fr, gr)


def test_b1_trampoline_and_rejects(fuel, orc, scene):
    """B == 1 (the costFunction trampoline, :693-706) and argument errors."""
    O = fuel.BsplineOptimizer
    tr = W.make_trajectories(scene["g"], scene["inflate"], B=1, n_pts=20, seed=2)
    opt = scene["opt"]
    opt.setBoundaryStates(list(tr["start"][0]), [tr["end_pos"][0]])
    opt.begin(tr["ctrl"][0], tr["dt"][0], O.NORMAL_PHASE | O.MINTIME)
    x = opt.initial_variables()
    f, g = opt.costFunction(x)
    tcs = orc.traj_consts(1)
    orc.fill_traj_const(tcs[0], opt.pt_dist_, tr["dt"][0], tr["start"][0], tr["end_pos"][0][None, :])
    assert abs(opt.pt_dist_ - orc.pt_dist(tr["ctrl"][0])) < 1e-15
    fr, gr = orc.combine_cost_batch(orc_grid(orc, scene["g"]), scene["d64"], orc.opt_params(), tcs, 20,
                                    O.NORMAL_PHASE | O.MINTIME, x[None, :])
    check(np.array([f]), g[None, :], fr, gr)
    with pytest.raises(fuel.FuelGpuError):
        opt.combineCostBatch(x[None, :], opt._tc, 20, O.NORMAL_PHASE | O.MINTIME | O.VIEWCONS)


def test_optimize_batch_matches_cpu_twin(fuel, orc, scene):
    """Device-side projected L-BFGS (replaces the NLopt loop of optimize(), :165-253) vs its CPU
    twin oracle.orc_optimize_batch.  Iterates diverge in the last bits (warp-reduction order), so
    the check is on the result: the returned x re-evaluates to the returned cost on the oracle,
    the cost never exceeds the start, the eval budget is respected, and the batch statistics
    agree with the twin."""
    B, N, K = 256, 20, 64
    O = fuel.BsplineOptimizer
    tr = W.make_trajectories(scene["g"], scene["inflate"], B=B, n_pts=N, seed=77)
    mask = O.NORMAL_PHASE | O.MINTIME
    x0 = W.pack_x(tr["ctrl"], tr["dt"])
    og = orc_grid(orc, scene["g"])
    to = orc_consts(orc, tr, B)
    f0, _ = orc.combine_cost_batch(og, scene["d64"], orc.opt_params(), to, N, mask, x0)
    xg, fg, ng = scene["opt"].optimizeBatch(x0, gpu_consts(fuel, tr, B), N, mask, K)
    xc, fc, nc = orc.optimize_batch(og, scene["d64"], orc.opt_params(), to, N, mask, x0, max_eval=K, threads=8)
    assert np.all(ng <= K) and np.all(ng >= 1)
    assert np.all(fg <= f0 * (1 + 1e-9))
    # returned variables are inside the bounds of :196-217
    pts = xg[:, :3 * N].reshape(B, N, 3)
    assert np.all(pts >= scene["g"].box_min + 0.1 - 1e-12) and np.all(pts <= scene["g"].box_max - 0.1 + 1e-12)
    assert np.all(xg[:, -1] >= 0.0) and np.all(xg[:, -1] <= 5.0)
    # best_variable_ re-evaluates to min_cost_ (fp32 ESDF samples vs the oracle's fp64 field: 1e-4)
    fchk, _ = orc.combine_cost_batch(og, scene["d64"], orc.opt_params(), to, N, mask, xg)
    assert np.all(np.abs(fchk - fg) <= 1e-4 * np.abs(fg) + 1e-9)
    # same algorithm, same budget.  The device loop samples the fp32 ESDF with fp32 lerps and contracts
    # FMAs, so after 64 non-convex iterations individual trajectories sit at slightly different points
    # than the fp64 twin; the gate is on solution quality: per-trajectory costs within a few percent
    # for the bulk, batch mean within 2 %, and never worse than the twin by more than 25 %.
    rel = np.abs(fg - fc) / np.abs(fc)
    print("median rel diff %.3g, p90 %.3g, mean gpu %.4f cpu %.4f" % (np.median(rel), np.quantile(rel, 0.9),
                                                                      np.mean(fg), np.mean(fc)))
    assert np.median(rel) < 0.03, np.median(rel)
    assert np.quantile(fg / fc, 0.99) < 1.25
    assert abs(np.mean(fg) - np.mean(fc)) < 0.02 * np.mean(fc)
    assert np.mean(fg) < 0.01 * np.mean(f0)


def test_optimize_single_and_small_budget(fuel, orc, scene):
    """optimize() through the mirror for one trajectory; max_eval=1 returns the clamped start."""
    O = fuel.BsplineOptimizer
    tr = W.make_trajectories(scene["g"], scene["inflate"], B=2, n_pts=20, seed=4)
    opt = scene["opt"]
    opt.setBoundaryStates(list(tr["start"][0]), [tr["end_pos"][0]])
    pts, dt = opt.optimize(tr["ctrl"][0], tr["dt"][0], O.NORMAL_PHASE | O.MINTIME, 1)
    assert pts.shape == (20, 3) and 0 < dt <= 5.0 and opt.iter_num_ <= 2000 and opt.start_state_ == []
    x0 = W.pack_x(tr["ctrl"], tr["dt"])
    xg, fg, ng = opt.optimizeBatch(x0, gpu_consts(fuel, tr, 2), 20, O.NORMAL_PHASE | O.MINTIME, 1)
    assert np.all(ng == 1)
    assert np.allclose(xg, x0)  # the workload's control points are already inside the shrunk box


def test_optimize_begin_end_equals_one_shot(fuel, orc, scene):
    """fuelgpu_bspline_optimize_batch_begin/_end is the one-shot call cut in two: same bits out, the input x untouched,
    a second begin before the end is refused."""
    B, N, K = 64, 20, 32
    O = fuel.BsplineOptimizer
    tr = W.make_trajectories(scene["g"], scene["inflate"], B=B, n_pts=N, seed=5)
    mask = O.NORMAL_PHASE | O.MINTIME
    x0 = W.pack_x(tr["ctrl"], tr["dt"])
    keep = x0.copy()
    tc = gpu_consts(fuel, tr, B)
    opt = scene["opt"]
    x1, f1, n1 = opt.optimizeBatch(x0, tc, N, mask, K)
    opt.optimizeBatchBegin(x0, tc, N, mask, K)
    with pytest.raises(fuel.FuelGpuError):
        opt.optimizeBatchBegin(x0, tc, N, mask, K)
    x2, f2, n2 = opt.optimizeBatchEnd()
    assert np.array_equal(x0, keep)
    assert np.array_equal(x1, x2) and np.array_equal(f1, f2) and np.array_equal(n1, n2)


def test_fast_evaluator_is_what_the_parity_bar_covers(fuel, orc, scene):
    """The solver loop (optimizeBatch, the kernel the benchmark times) evaluates with eval_warp<true>: fp32 trilinear
    lerps on the fp32 ESDF samples, reciprocals, one merged reduction, FMA contraction.  FUELGPU_COST_FAST_EVAL runs
    exactly that evaluator once: cost AND gradient against the oracle, same 1e-4 bar, on the config-2 batch, the
    adversarial positions and a 4096-trajectory batch."""
    O = fuel.BsplineOptimizer
    g = scene["g"]
    og = orc_grid(orc, g)
    mask = O.NORMAL_PHASE | O.MINTIME
    for B, seed in ((1024, 20260922), (4096, 101)):
        tr = W.make_trajectories(g, scene["inflate"], B=B, n_pts=20, seed=seed)
        x = W.pack_x(tr["ctrl"], tr["dt"])
        x[::3, -1] *= 0.5  # make feasibility and its dt-gradient bite
        f, gg = scene["opt"].combineCostBatch(x, gpu_consts(fuel, tr, B), 20, mask, fast_eval=True)
        fr, gr = orc.combine_cost_batch(og, scene["d64"], orc.opt_params(), orc_consts(orc, tr, B), 20, mask, x, threads=8)
        check(f, gg, fr, gr)
        f2, g2 = scene["opt"].combineCostBatch(x, gpu_consts(fuel, tr, B), 20, mask)
        assert not (np.array_equal(f, f2) and np.array_equal(gg, g2)), "the flag did not switch evaluators"
    fast_evaluator_adversarial_and_single_terms(fuel, orc, scene, 20)


@pytest.mark.parametrize("n_pts", [7, 8, 31, 32])
def test_fast_evaluator_n_pts(fuel, orc, scene, n_pts):
    """The fast evaluator's adversarial positions and single terms at the edges of its warp layout (one lane per
    control point: a single interior segment at 7, a full warp at 32)."""
    fast_evaluator_adversarial_and_single_terms(fuel, orc, scene, n_pts)


def fast_evaluator_adversarial_and_single_terms(fuel, orc, scene, n_pts):
    O = fuel.BsplineOptimizer
    g = scene["g"]
    og = orc_grid(orc, g)
    mask = O.NORMAL_PHASE | O.MINTIME
    # adversarial positions: map boundary, outside the map, the isInMap margin
    B = 48
    tr = W.make_trajectories(g, scene["inflate"], B=B, n_pts=n_pts, seed=13)
    ctrl = tr["ctrl"].copy()
    ctrl[0:8, 5 * n_pts // 20] = g.origin + [0.02, 0.5, 0.5]
    ctrl[8:16, 7 * n_pts // 20] = g.map_max + 0.3
    ctrl[16:24, 9 * n_pts // 20] = g.map_max - [1e-4, 0.5, 0.5]
    tr["ctrl"] = ctrl
    x = W.pack_x(ctrl, tr["dt"])
    f, gg = scene["opt"].combineCostBatch(x, gpu_consts(fuel, tr, B), n_pts, mask, fast_eval=True)
    fr, gr = orc.combine_cost_batch(og, scene["d64"], orc.opt_params(), orc_consts(orc, tr, B), n_pts, mask, x)
    check(f, gg, fr, gr)
    # every single term through the fast evaluator
    tr = W.make_trajectories(g, scene["inflate"], B=64, n_pts=n_pts, seed=5)
    for name in ("SMOOTHNESS", "DISTANCE", "FEASIBILITY", "START", "END"):
        m1 = getattr(O, name)
        x = W.pack_x(tr["ctrl"], tr["dt"] * 0.6, mintime=False)
        tr2 = dict(tr)
        tr2["dt"] = tr["dt"] * 0.6
        f, gg = scene["opt"].combineCostBatch(x, gpu_consts(fuel, tr2, 64), n_pts, m1, fast_eval=True)
        fr, gr = orc.combine_cost_batch(og, scene["d64"], orc.opt_params(), orc_consts(orc, tr2, 64), n_pts, m1, x)
        check(f, gg, fr, gr)


def test_exact_eval_mode_performs_every_evaluation(fuel, orc, scene):
    """FUELGPU_SOLVE_EXACT_EVALS (what bench.py times): every trajectory reports exactly max_eval evaluations and
    the result is never worse than the normal mode's start."""
    B, N, K = 1024, 20, 64
    O = fuel.BsplineOptimizer
    tr = W.make_trajectories(scene["g"], scene["inflate"], B=B, n_pts=N)
    mask = O.NORMAL_PHASE | O.MINTIME
    x0 = W.pack_x(tr["ctrl"], tr["dt"])
    tc = gpu_consts(fuel, tr, B)
    xe, fe, ne = scene["opt"].optimizeBatch(x0, tc, N, mask, K, xtol_rel=0.0, exact_evals=True)
    assert np.all(ne == K), (ne.min(), ne.max())
    xn, fn, nn = scene["opt"].optimizeBatch(x0, tc, N, mask, K, xtol_rel=0.0)
    assert np.all(nn <= K)
    print("normal mode evals: min %d mean %.2f" % (nn.min(), nn.mean()))
    f0, _ = orc.combine_cost_batch(orc_grid(orc, scene["g"]), scene["d64"], orc.opt_params(), orc_consts(orc, tr, B), N,
                                   mask, x0, threads=8)
    assert np.all(fe <= f0 * (1 + 1e-9))
    same = nn == K
    assert np.array_equal(xe[same], xn[same])  # trajectories that never stop early take the identical path


def test_view_cost(fuel, orc, scene):
    """calcViewCost (bspline_optimizer.cpp:477-502, the VIEWCONS bit): both sides of the |dl| < |dir| switch, alone and
    inside the full objective, through the faithful AND the solver's evaluator; missing constraint -> EINVAL."""
    O = fuel.BsplineOptimizer
    g = scene["g"]
    og = orc_grid(orc, g)
    B, N = 64, 20
    tr = W.make_trajectories(g, scene["inflate"], B=B, n_pts=N, seed=23)
    rng = np.random.default_rng(23)
    opt = fuel.BsplineOptimizer()
    opt.setEnvironment(scene["opt"].edt_environment_)
    opt.setParam(ld_view=2.5, wnl=1.3)
    po = orc.opt_params(ld_view=2.5, wnl=1.3)
    tg = gpu_consts(fuel, tr, B)
    to = orc_consts(orc, tr, B)
    n_par = 0
    for b in range(B):
        idx = int(rng.integers(0, N))
        pt = tr["ctrl"][b, idx] + rng.normal(size=3) * 0.4
        d = (tr["ctrl"][b, idx] - pt) * float(rng.choice([-1.0, 1.0])) + rng.normal(size=3) * 0.1
        d = d / np.linalg.norm(d) * float(rng.choice([0.2, 1.5]))
        for t in (tg[b], to[b]):
            for k in range(3):
                t.view_pt[k], t.view_dir[k] = pt[k], d[k]
            t.view_idx = idx
        n_par += int(abs(np.dot(tr["ctrl"][b, idx] - pt, d / np.linalg.norm(d))) < np.linalg.norm(d))
    assert 5 < n_par < B - 5
    for mask in (O.VIEWCONS, O.NORMAL_PHASE | O.VIEWCONS | O.MINTIME):
        x = W.pack_x(tr["ctrl"], tr["dt"], mintime=bool(mask & O.MINTIME))
        fr, gr = orc.combine_cost_batch(og, scene["d64"], po, to, N, mask, x)
        for fast in (False, True):
            f, gg = opt.combineCostBatch(x, tg, N, mask, fast_eval=fast)
            check(f, gg, fr, gr)
        if mask == O.VIEWCONS:
            assert np.all(np.count_nonzero(gg, axis=1) <= 3)
    # the solver accepts the bit as well and does not make things worse
    x0 = W.pack_x(tr["ctrl"], tr["dt"])
    mask = O.NORMAL_PHASE | O.VIEWCONS | O.MINTIME
    f0, _ = orc.combine_cost_batch(og, scene["d64"], po, to, N, mask, x0)
    xs, fs, ns = opt.optimizeBatch(x0, tg, N, mask, 32)
    assert np.all(fs <= f0 * (1 + 1e-9))
    fchk, _ = orc.combine_cost_batch(og, scene["d64"], po, to, N, mask, xs)
    assert np.all(np.abs(fchk - fs) <= 1e-4 * np.abs(fs) + 1e-9)
    # no constraint set (view_idx = -1): refused
    with pytest.raises(fuel.FuelGpuError):
        opt.combineCostBatch(x0, gpu_consts(fuel, tr, B), N, mask)
