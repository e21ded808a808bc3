"""The CPU twin of the device solver (oracle.optimize_batch) against linear algebra, and its two options: the
FUELGPU_SOLVE_EXACT_EVALS mode and the decision trace.

The objective is the convex quadratic of tests.helpers (SMOOTHNESS | START | END | GUIDE | WAYPOINTS, 3-entry end
state), whose minimiser numpy / scipy give exactly.  Tolerances measured on these seeds (48 instances per case):
- default xtol_rel = 1e-5: the solver stops once every step is below 1e-5 of |x| (~1e-4 m on this box), which leaves
  up to 3.3e-4 m between x_best and x* and 4.3e-8 relative on the cost; the bars are 1e-3 m and 1e-6.
- xtol_rel = 0: the solver runs until the projected gradient vanishes, the line search fails or 2000 evaluations,
  and lands within 1.1e-7 m of x* (the cost is then flat to its last bits); the bar is 1e-6 m.
"""
import numpy as np
import pytest

from fuel_b200 import workloads as W
from tests.helpers import QUAD_WEIGHTS, orc_grid, quad_consts, quad_mask, quad_minimisers, quadratic_problems

B = 48


@pytest.fixture(scope="module")
def box(orc):
    g, _ = W.office_map()
    return g, orc_grid(orc, g)


def quad_case(orc, box, n, bound, seed):
    g, og = box
    par = orc.opt_params(**QUAD_WEIGHTS)
    P = quadratic_problems(g, B, n, seed, bound=bound)
    tcs = quad_consts(orc.fill_traj_const, orc.traj_consts(B), P)
    xs, is_bound = quad_minimisers(orc, og, par, tcs, n, P, g)
    return par, P, tcs, xs, is_bound, np.stack([q["x0"] for q in P])


@pytest.mark.parametrize("bound", [False, True], ids=["interior", "box_bound"])
@pytest.mark.parametrize("n", [7, 20, 32])
def test_twin_reaches_quadratic_minimiser(orc, box, n, bound):
    """x_best reaches the exact (or box-constrained) minimiser for every history length 1..8."""
    g, og = box
    par, P, tcs, xs, is_bound, X0 = quad_case(orc, box, n, bound, seed=n)
    if bound and n >= 8:
        assert is_bound.all()
    if not bound:
        assert not is_bound.any()
    mask = quad_mask(orc)
    fs, _ = orc.combine_cost_batch(og, np.zeros(1), par, tcs, n, mask, xs)
    for m in range(1, 9):
        x, f, ne = orc.optimize_batch(og, np.zeros(1), par, tcs, n, mask, X0, max_eval=2000, lbfgs_m=m, threads=4)
        err = np.max(np.abs(x - xs))
        assert err < 1e-3, (m, err)
        assert np.all(np.abs(f - fs) <= 1e-6 * np.abs(fs)), (m, np.max(np.abs(f - fs) / np.abs(fs)))
        assert np.all(f >= fs * (1 - 1e-12))  # nothing beats the minimiser
        x, f, ne = orc.optimize_batch(og, np.zeros(1), par, tcs, n, mask, X0, max_eval=2000, lbfgs_m=m,
                                      xtol_rel=0.0, threads=4)
        err = np.max(np.abs(x - xs))
        assert err < 1e-6, (m, err)


def test_exact_mode_does_every_evaluation(orc, box):
    """FUELGPU_SOLVE_EXACT_EVALS: exactly K evaluations whatever happens -- quadratics run far past convergence (the
    line search fails at the bottom), starts at the minimiser, a start with an exactly zero gradient -- and the result
    is never worse than normal mode's at the same budget."""
    g, og = box
    n = 20
    par, P, tcs, xs, _, X0 = quad_case(orc, box, n, False, seed=3)
    mask = quad_mask(orc)
    for K in (1, 2, 37, 400):
        for start in (X0, xs):
            xe, fe, ne = orc.optimize_batch(og, np.zeros(1), par, tcs, n, mask, start, max_eval=K, exact_evals=True)
            assert np.all(ne == K), (K, ne.min(), ne.max())
            xn, fn, nn = orc.optimize_batch(og, np.zeros(1), par, tcs, n, mask, start, max_eval=K)
            assert np.all(fe <= fn * (1 + 1e-12))
    # a start whose gradient is exactly zero (GUIDE alone, guide points = the control points): exact mode evaluates
    # in place K times, normal mode stops after the first evaluation; both return the start
    pz = quadratic_problems(g, 4, n, 11)
    for q in pz:
        q["guide"] = q["x0"].reshape(n, 3)[3:n - 3].copy()
    tz = quad_consts(orc.fill_traj_const, orc.traj_consts(4), pz)
    xz = np.stack([q["x0"] for q in pz])
    fz, gz = orc.combine_cost_batch(og, np.zeros(1), par, tz, n, orc.GUIDE, xz)
    assert np.all(fz == 0.0) and np.all(gz == 0.0)
    for exact, want in ((True, 64), (False, 1)):
        xo, fo, no = orc.optimize_batch(og, np.zeros(1), par, tz, n, orc.GUIDE, xz, max_eval=64, exact_evals=exact)
        assert np.all(no == want) and np.array_equal(xo, xz) and np.all(fo == 0.0)


def bench_problem(orc, n=20, B=256, seed=5):
    g, inflate = W.office_map()
    tri = W.office_known(g, inflate)
    og = orc_grid(orc, g)
    d = orc.update_esdf3d(og, inflate, tri, [0, 0, 0], np.array(g.n) - 1, True, False, threads=8)
    tr = W.make_trajectories(g, inflate, B=B, n_pts=n, seed=seed)
    tcs = orc.traj_consts(B)
    for b in range(B):
        orc.fill_traj_const(tcs[b], tr["pt_dist"][b], tr["dt"][b], tr["start"][b], tr["end_pos"][b][None, :])
    return og, d, tcs, W.pack_x(tr["ctrl"], tr["dt"])


@pytest.mark.parametrize("exact", [False, True], ids=["normal", "exact"])
def test_trace_changes_no_result_bit(orc, exact):
    """The traced run returns the same bytes as the plain one, on the bench objective and on a curvature-heavy
    setting; the trace is self-consistent (margins non-increasing in k, counts add up, first events in range)."""
    og, d, tcs, x0 = bench_problem(orc)
    n = 20
    mask = orc.NORMAL_PHASE | orc.MINTIME
    for par, K, m in ((orc.opt_params(), 64, 6), (orc.opt_params(ld_dist=100.0, dist0=1.5), 128, 3)):
        a = orc.optimize_batch(og, d, par, tcs, n, mask, x0, max_eval=K, lbfgs_m=m, exact_evals=exact, threads=8)
        b = orc.optimize_batch(og, d, par, tcs, n, mask, x0, max_eval=K, lbfgs_m=m, exact_evals=exact, threads=8,
                               trace=True)
        for u, v in zip(a, b[:3]):
            assert u.dtype == v.dtype and np.array_equal(u, v)
        tr = b[3]
        mg = tr["margin"]
        assert mg.shape == (len(x0), K) and np.all(np.diff(mg, axis=1) <= 0) and np.all(mg >= 0)
        assert np.all(tr["n_full_reject"] <= tr["n_curv_reject"])
        assert np.all(tr["n_kept"] + tr["n_curv_reject"] <= b[2])
        for ev, cnt in (("first_full_reject", "n_full_reject"), ("first_ls_fail", "n_ls_fail")):
            assert np.all((tr[ev] < 0) == (tr[cnt] == 0))
            assert np.all(tr[ev][tr[cnt] > 0] >= 2) and np.all(tr[ev] < K)
        if not exact:
            assert np.all(tr["n_ls_fail"] <= 1)  # normal mode stops at the first failure
