// bspline_solve.cu -- persistent per-trajectory solver (the NLopt loop of BsplineOptimizer::optimize()).
// Compiled with FMA contraction enabled: the iterate sequence is our own (NLopt parity is unpinned),
// only the faithful cost kernel in bspline.cu keeps the reference's rounding order.
#include "bspline_eval.cuh"

#include <stdlib.h>
#include <string.h>

namespace {

// =========================================================================================
// Persistent per-trajectory solver: replaces the NLopt driver loop of
// BsplineOptimizer::optimize() (:165-253) -- clamp to the box shrunk by 0.1 m (:175-204),
// bounds q0 +- 10 m clipped to that box and dt in [0,5] (:206-217), maxeval stop (:170),
// xtol_rel stop (:173), best-x tracking of costFunction (:693-706) -- around a projected
// L-BFGS with Armijo backtracking.  One warp per trajectory for the whole solve; the
// iterate, gradient and search direction live in registers (lane i = control point i,
// lane n = dt), the (s,y) history in shared memory.
// =========================================================================================
constexpr int MAXM = 8;

struct V3 {
  double v[3];
};
// Solver-internal inner products (L-BFGS coefficients, Armijo slope, curvature test): the per-lane partial is
// formed in fp64 and the 32-lane sum runs as an fp32 xor butterfly (one SHFL per stage instead of two, the sum
// lands in every lane).  A relative 1e-7 on these scalars only perturbs the quasi-Newton direction; the cost F
// that decides acceptance and best-x stays fp64.
__device__ __forceinline__ double wsum_x(double v) {
  float f = (float)v;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) f += __shfl_xor_sync(0xffffffffu, f, o);
  return (double)f;
}
__device__ __forceinline__ double dot3(const V3& a, const V3& b) {
  return wsum_x(a.v[0] * b.v[0] + a.v[1] * b.v[1] + a.v[2] * b.v[2]);
}
// history element (slot, component k) of this lane: [slot][k][lane], conflict-free
#define HIDX(slot, k) ((slot) * 96 + (k) * 32 + lane)

__global__ void __launch_bounds__(WPB * 32) optimize_warp_kernel(
    Geom g, const float* __restrict__ dist, FuelOptParams p, const FuelTrajConst* __restrict__ tc, int n,
    int mask, int B, FuelSolveParams sp, double* __restrict__ x, double* __restrict__ fbest,
    int* __restrict__ neval_out) {
  extern __shared__ double hist[];  // [WPB][2][m][32][3]
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int b = blockIdx.x * WPB + w;
  if (b >= B) return;
  const bool opt_time = (mask & FUELGPU_MINTIME) != 0;
  const int nvar = opt_time ? 3 * n + 1 : 3 * n;
  const int m = sp.lbfgs_m;
  double* S = hist + (size_t)w * 2 * m * 96;
  double* Y = S + (size_t)m * 96;
  double* xb = x + (int64_t)b * nvar;
  TrajRegs t;
  load_traj(tc + b, t);

  // variables of this lane: control point (lane < n), dt in component 0 of lane n
  const bool is_pt = lane < n;
  const bool is_dt = opt_time && lane == n;
  V3 X, lb, ub;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    X.v[k] = 0.0;
    lb.v[k] = 0.0;
    ub.v[k] = 0.0;
    if (is_pt) {
      const double bmin = g.box_mind[k] + 0.1, bmax = g.box_maxd[k] - 0.1;
      double c = xb[3 * lane + k];
      c = fmax(fmin(c, bmax), bmin);  // :199-203
      X.v[k] = c;
      lb.v[k] = fmax(c - 10.0, bmin);  // :208-214
      ub.v[k] = fmin(c + 10.0, bmax);
    }
  }
  if (is_dt) {
    X.v[0] = xb[nvar - 1];
    lb.v[0] = 0.0;  // :215-218
    ub.v[0] = 5.0;
  }

  auto evaluate = [&](const V3& xx, double& fo, V3& go) {
    const double dtv = opt_time ? __shfl_sync(0xffffffffu, xx.v[0], n) : t.knot_span;
    double gr[3], gdt;
    eval_warp<true>(g, dist, p, t, tc + b, n, mask, xx.v, dtv, lane, fo, gr, gdt);
    go.v[0] = is_pt ? gr[0] : (is_dt ? gdt : 0.0);
    go.v[1] = is_pt ? gr[1] : 0.0;
    go.v[2] = is_pt ? gr[2] : 0.0;
  };
  auto store_best = [&](const V3& xx, double fv) {
    if (is_pt) {
      xb[3 * lane] = xx.v[0];
      xb[3 * lane + 1] = xx.v[1];
      xb[3 * lane + 2] = xx.v[2];
    }
    if (is_dt) xb[nvar - 1] = xx.v[0];
    if (lane == 0) fbest[b] = fv;
  };

  double F;
  V3 G;
  evaluate(X, F, G);
  int neval = 1;
  double best = F;
  store_best(X, F);
  // a NaN/inf start cannot be improved on by comparison; treat as +inf
  if (!(best == best)) best = 1.7976931348623157e308;

  const bool exact = (sp.flags & FUELGPU_SOLVE_EXACT_EVALS) != 0;
  int cnt = 0, head = 0;  // history ring: newest at (head-1) mod m
  double gamma_new = 1.0;
  double rho[MAXM];  // rho[j] belongs to the j-th newest pair (static indices: stays in registers)
#pragma unroll
  for (int j = 0; j < MAXM; ++j) rho[j] = 0.0;

  while (neval < sp.max_eval) {
    // projected gradient
    V3 PG, D;
    bool actv[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      actv[k] = (X.v[k] <= lb.v[k] && G.v[k] > 0.0) || (X.v[k] >= ub.v[k] && G.v[k] < 0.0);
      PG.v[k] = actv[k] ? 0.0 : G.v[k];
    }
    const double pgn2 = dot3(PG, PG);
    if (!(pgn2 > 1e-24)) {
      if (!exact) break;
      // benchmark mode: the objective is still evaluated max_eval times (in place: nothing left to descend)
      while (neval < sp.max_eval) {
        evaluate(X, F, G);
        ++neval;
      }
      break;
    }
    // two-loop recursion
    V3 Q = PG;
    double alpha[MAXM];
#pragma unroll
    for (int j = 0; j < MAXM; ++j) {
      alpha[j] = 0.0;
      if (j < cnt) {
        int slot = head - 1 - j;  // j < cnt <= m: one wrap at most
        if (slot < 0) slot += m;
        V3 s, y;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          s.v[k] = S[HIDX(slot, k)];
          y.v[k] = Y[HIDX(slot, k)];
        }
        alpha[j] = rho[j] * dot3(s, Q);
#pragma unroll
        for (int k = 0; k < 3; ++k) Q.v[k] -= alpha[j] * y.v[k];
      }
    }
    if (cnt > 0) {  // gamma = s.y / y.y of the newest pair, kept from the moment it was stored
#pragma unroll
      for (int k = 0; k < 3; ++k) Q.v[k] *= gamma_new;
    }
#pragma unroll
    for (int j = MAXM - 1; j >= 0; --j) {
      if (j < cnt) {
        int slot = head - 1 - j;
        if (slot < 0) slot += m;
        V3 s, y;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          s.v[k] = S[HIDX(slot, k)];
          y.v[k] = Y[HIDX(slot, k)];
        }
        const double beta = rho[j] * dot3(y, Q);
#pragma unroll
        for (int k = 0; k < 3; ++k) Q.v[k] += s.v[k] * (alpha[j] - beta);
      }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) D.v[k] = actv[k] ? 0.0 : -Q.v[k];
    double gd = dot3(G, D);
    if (!(gd < 0.0)) {  // not a descent direction: restart from steepest descent
#pragma unroll
      for (int k = 0; k < 3; ++k) D.v[k] = -PG.v[k];
      gd = -pgn2;
      cnt = 0;
    }
    double step = cnt == 0 ? fmin(1.0, 1.0 / sqrt(pgn2)) : 1.0;

    // Armijo backtracking on the projected path
    bool accepted = false;
    V3 XN, GN;
    double FN = 0.0;
    while (neval < sp.max_eval) {
      bool clipped = false;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double xt = X.v[k] + step * D.v[k];
        clipped = clipped || xt > ub.v[k] || xt < lb.v[k];
        XN.v[k] = fmax(fmin(xt, ub.v[k]), lb.v[k]);
      }
      evaluate(XN, FN, GN);
      ++neval;
      if (FN < best) {  // costFunction :698-704
        best = FN;
        store_best(XN, FN);
      }
      double dec = step * gd;  // = G.(XN - X) as long as no component hit a bound
      if (__any_sync(0xffffffffu, clipped)) {
        V3 dx;
#pragma unroll
        for (int k = 0; k < 3; ++k) dx.v[k] = XN.v[k] - X.v[k];
        dec = dot3(G, dx);
      }
      if (FN <= F + 1e-4 * dec) {
        accepted = true;
        break;
      }
      step *= 0.5;
      if (step < 1e-12) break;
    }
    if (!accepted) {
      if (!exact) break;
      cnt = 0;  // benchmark mode: drop the history and go on from steepest descent
      continue;
    }
    V3 s, y;
    bool small = true;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      s.v[k] = XN.v[k] - X.v[k];
      y.v[k] = GN.v[k] - G.v[k];
      small = small && (fabs(s.v[k]) <= sp.xtol_rel * fabs(XN.v[k]));
    }
    const double sy = dot3(s, y);
    const double ss = dot3(s, s), yy = dot3(y, y);
    if (sy > 1e-10 * sqrt(ss * yy)) {
      const int slot = head;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        S[HIDX(slot, k)] = s.v[k];
        Y[HIDX(slot, k)] = y.v[k];
      }
      __syncwarp();
#pragma unroll
      for (int j = MAXM - 1; j > 0; --j) rho[j] = rho[j - 1];
      rho[0] = 1.0 / sy;
      gamma_new = sy / yy;
      head = head + 1 == m ? 0 : head + 1;
      if (cnt < m) ++cnt;
    }
    X = XN;
    F = FN;
    G = GN;
    if (!exact && __all_sync(0xffffffffu, small)) break;  // xtol_rel, :173
  }
  // min_cost_ is reported from the full-precision evaluator (fp64 trilinear, per-term reductions) at
  // the returned best_variable_, so it equals what combineCost gives for that x.
  {
    __syncwarp();
    V3 XB;
#pragma unroll
    for (int k = 0; k < 3; ++k) XB.v[k] = is_pt ? xb[3 * lane + k] : 0.0;
    if (is_dt) XB.v[0] = xb[nvar - 1];
    const double dtv = opt_time ? __shfl_sync(0xffffffffu, XB.v[0], n) : t.knot_span;
    double fo, gr[3], gdt;
    eval_warp<false>(g, dist, p, t, tc + b, n, mask, XB.v, dtv, lane, fo, gr, gdt);
    if (lane == 0) fbest[b] = fo;
  }
  if (lane == 0) neval_out[b] = neval;
}


// =========================================================================================
// The same solver with the L-BFGS recursion in COEFFICIENT space.  The vector form above runs 2m + 5 dependent
// warp reductions per iteration (each ~190 cycles of shuffle latency: a third of the iteration).  Here the warp
// keeps the Gram data of the stored pairs -- SY[a][b] = s_a.y_b, YY[a][b] = y_a.y_b, and u_a = s_a.pg, w_a = y_a.pg
// for the current projected gradient -- so the two-loop recursion is scalar arithmetic every lane repeats, the
// direction is one linear combination of the stored vectors, and ALL inner products an iteration needs (the new
// pair against the stored ones, the new projected gradient against all pairs, s.y, y.y, s.s, pg.pg) are independent:
// they go through ONE batched butterfly (up to 5m+1 values interleaved) right after the accepted evaluation.
// Same mathematics as the vector form (direction = -H pg with the same pairs, rho and gamma); rounding differs.
// =========================================================================================

// 32 values per lane -> lane l ends with the warp-wide sum of value l: every stage sends half of the values still held
// to the partner lane and adds the other half (31 shuffles instead of 5 x 32), "transpose and reduce".
__device__ __forceinline__ float transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const bool hi = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      if (i < o) {
        const float keep = hi ? v[i + o] : v[i];
        const float send = hi ? v[i] : v[i + o];
        v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
      }
    }
  }
  return v[0];
}

// floats of shared memory per warp (a multiple of 4: the history is float4)
#define GRAM_FLOATS(M) ((2 * (M) * 32 * 4 + 2 * (M) * (M) + 3 * (M) + 32 + 3) / 4 * 4)

template <int M>  // history length, compile time: every recursion loop has static bounds (5*M + 1 <= 32 values per batch)
__global__ void __launch_bounds__(WPB * 32) optimize_gram_kernel(
    Geom g, const float* __restrict__ dist, FuelOptParams p, const FuelTrajConst* __restrict__ tc, int n,
    int mask, int B, FuelSolveParams sp, double* __restrict__ x, double* __restrict__ fbest,
    int* __restrict__ neval_out) {
  static_assert(5 * M + 1 <= 32, "the batched reduction holds 32 values");
  constexpr int MAXM = M;  // (shadows the file-level bound: Gram arrays are M wide here)
  extern __shared__ double hist[];  // per warp, as floats: S M*32 float4 | Y M*32 float4 | SY M*M | YY M*M | rho,u,w M | red 32
  const int lane = threadIdx.x & 31;
  const int w = threadIdx.x >> 5;
  const int b = blockIdx.x * WPB + w;
  if (b >= B) return;
  const bool opt_time = (mask & FUELGPU_MINTIME) != 0;
  const int nvar = opt_time ? 3 * n + 1 : 3 * n;
  constexpr int m = M;
  float4* S4 = reinterpret_cast<float4*>(hist) + (size_t)w * (GRAM_FLOATS(M) / 4);
  float4* Y4 = S4 + M * 32;
  float* SYg = reinterpret_cast<float*>(Y4 + M * 32);
  float* YYg = SYg + MAXM * MAXM;
  float* RHO = YYg + MAXM * MAXM;
  float* Ug = RHO + MAXM;
  float* Wg = Ug + MAXM;
  float* RED = Wg + MAXM;  // the 32 sums of the last batched reduction
  double* xb = x + (int64_t)b * nvar;
  TrajRegs t;
  load_traj(tc + b, t);

  const bool is_pt = lane < n;
  const bool is_dt = opt_time && lane == n;
  V3 X, lb, ub;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    X.v[k] = 0.0;
    lb.v[k] = 0.0;
    ub.v[k] = 0.0;
    if (is_pt) {
      const double bmin = g.box_mind[k] + 0.1, bmax = g.box_maxd[k] - 0.1;
      double c = xb[3 * lane + k];
      c = fmax(fmin(c, bmax), bmin);  // :199-203
      X.v[k] = c;
      lb.v[k] = fmax(c - 10.0, bmin);  // :208-214
      ub.v[k] = fmin(c + 10.0, bmax);
    }
  }
  if (is_dt) {
    X.v[0] = xb[nvar - 1];
    lb.v[0] = 0.0;  // :215-218
    ub.v[0] = 5.0;
  }
  auto evaluate = [&](const V3& xx, double& fo, V3& go) {
    const double dtv = opt_time ? __shfl_sync(0xffffffffu, xx.v[0], n) : t.knot_span;
    double gr[3], gdt;
    eval_warp<true>(g, dist, p, t, tc + b, n, mask, xx.v, dtv, lane, fo, gr, gdt);
    go.v[0] = is_pt ? gr[0] : (is_dt ? gdt : 0.0);
    go.v[1] = is_pt ? gr[1] : 0.0;
    go.v[2] = is_pt ? gr[2] : 0.0;
  };
  auto store_best = [&](const V3& xx, double fv) {
    if (is_pt) {
      xb[3 * lane] = xx.v[0];
      xb[3 * lane + 1] = xx.v[1];
      xb[3 * lane + 2] = xx.v[2];
    }
    if (is_dt) xb[nvar - 1] = xx.v[0];
    if (lane == 0) fbest[b] = fv;
  };
  auto project = [&](const V3& xx, const V3& gg, V3& pg, bool actv[3]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      actv[k] = (xx.v[k] <= lb.v[k] && gg.v[k] > 0.0) || (xx.v[k] >= ub.v[k] && gg.v[k] < 0.0);
      pg.v[k] = actv[k] ? 0.0 : gg.v[k];
    }
  };
  auto d3 = [](const V3& a, const V3& c) { return a.v[0] * c.v[0] + a.v[1] * c.v[1] + a.v[2] * c.v[2]; };

  double F;
  V3 G;
  evaluate(X, F, G);
  int neval = 1;
  double best = F;
  store_best(X, F);
  if (!(best == best)) best = 1.7976931348623157e308;

  const bool exact = (sp.flags & FUELGPU_SOLVE_EXACT_EVALS) != 0;
  int cnt = 0, head = 0;  // history ring: newest pair in slot (head-1) mod m
  float gamma = 1.f;
  V3 PG;
  bool actv[3];
  project(X, G, PG, actv);
  float pgf[3] = {(float)PG.v[0], (float)PG.v[1], (float)PG.v[2]};
  float pgn2 = (float)wsum_x(d3(PG, PG));

  while (neval < sp.max_eval) {
    if (!(pgn2 > 1e-24f)) {
      if (!exact) break;
      while (neval < sp.max_eval) {  // benchmark mode: the objective is still evaluated max_eval times
        evaluate(X, F, G);
        ++neval;
      }
      break;
    }
    // with no stored pair the direction is steepest descent, -pg (the scale of the last pair does not carry over a
    // restart: a failed line search or a non-descent direction empties the history)
    if (cnt == 0) gamma = 1.f;
    // ---- two-loop recursion on fp32 scalars (every lane the same values; Gram data by broadcast reads).  The Gram
    // entries come out of an fp32 reduction, so fp32 arithmetic on them loses nothing; the result is only the search
    // direction -- acceptance (F, Armijo) and the iterate stay fp64.
    float a[M], cs[M], cy[M];
    int slot[M];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      int sl = head - 1 - j;
      if (sl < 0) sl += m;
      slot[j] = j < cnt ? sl : 0;
      a[j] = 0.f;
      cs[j] = 0.f;
      cy[j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < M; ++j) {  // newest -> oldest
      if (j < cnt) {
        float acc = Ug[slot[j]];
#pragma unroll
        for (int i = 0; i < M; ++i)
          if (i < j) acc -= a[i] * SYg[slot[j] * M + slot[i]];
        a[j] = RHO[slot[j]] * acc;
      }
    }
    float gd = gamma * pgn2;  // accumulates pg.r
#pragma unroll
    for (int j = M - 1; j >= 0; --j) {  // oldest -> newest
      if (j < cnt) {
        float yq = Wg[slot[j]];
#pragma unroll
        for (int i = 0; i < M; ++i)
          if (i < cnt) yq -= a[i] * YYg[slot[j] * M + slot[i]];
        float acc = gamma * yq;
#pragma unroll
        for (int i = 0; i < M; ++i)
          if (i > j && i < cnt) acc += cs[i] * SYg[slot[i] * M + slot[j]];
        cs[j] = a[j] - RHO[slot[j]] * acc;
        cy[j] = -gamma * a[j];
      }
    }
    // direction: r = gamma pg + sum_j cs_j s_j + cy_j y_j ;  d = -r off the active bounds ;  g.d = -pg.r
    float R[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) R[k] = gamma * pgf[k];
#pragma unroll
    for (int j = 0; j < M; ++j) {
      if (j < cnt) {
        gd += cs[j] * Ug[slot[j]] + cy[j] * Wg[slot[j]];
        const float4 st = S4[slot[j] * 32 + lane], yt = Y4[slot[j] * 32 + lane];
        R[0] += cs[j] * st.x + cy[j] * yt.x;
        R[1] += cs[j] * st.y + cy[j] * yt.y;
        R[2] += cs[j] * st.z + cy[j] * yt.z;
      }
    }
    gd = -gd;
    V3 D;
#pragma unroll
    for (int k = 0; k < 3; ++k) D.v[k] = actv[k] ? 0.0 : -(double)R[k];
    if (!(gd < 0.f)) {  // not a descent direction: restart from steepest descent
#pragma unroll
      for (int k = 0; k < 3; ++k) D.v[k] = -PG.v[k];
      gd = -pgn2;
      cnt = 0;
    }
    double step = cnt == 0 ? (double)fminf(1.f, rsqrtf(pgn2)) : 1.0;

    // ---- Armijo backtracking on the projected path ----
    bool accepted = false;
    V3 XN, GN;
    double FN = 0.0;
    while (neval < sp.max_eval) {
      bool clipped = false;
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const double xt = X.v[k] + step * D.v[k];
        clipped = clipped || xt > ub.v[k] || xt < lb.v[k];
        XN.v[k] = fmax(fmin(xt, ub.v[k]), lb.v[k]);
      }
      evaluate(XN, FN, GN);
      ++neval;
      if (FN < best) {  // costFunction :698-704
        best = FN;
        store_best(XN, FN);
      }
      double dec = step * (double)gd;
      if (__any_sync(0xffffffffu, clipped)) {
        V3 dx;
#pragma unroll
        for (int k = 0; k < 3; ++k) dx.v[k] = XN.v[k] - X.v[k];
        dec = wsum_x(d3(G, dx));
      }
      if (FN <= F + 1e-4 * dec) {
        accepted = true;
        break;
      }
      step *= 0.5;
      if (step < 1e-12) break;
    }
    if (!accepted) {
      if (!exact) break;
      cnt = 0;
      continue;
    }
    float sf[3], yf[3];
    bool small = true;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const double sd = XN.v[k] - X.v[k];
      sf[k] = (float)sd;
      yf[k] = (float)(GN.v[k] - G.v[k]);
      small = small && (fabs(sd) <= sp.xtol_rel * fabs(XN.v[k]));
    }
    X = XN;
    F = FN;
    G = GN;
    project(X, G, PG, actv);
#pragma unroll
    for (int k = 0; k < 3; ++k) pgf[k] = (float)PG.v[k];
    auto f3 = [](const float* u, const float* v) { return u[0] * v[0] + u[1] * v[1] + u[2] * v[2]; };
    // ---- ONE batched reduction: everything this and the next iteration need ----
    // layout: [0] s.y [1] y.y [2] s.s [3] pg.pg [4] s.pg [5] y.pg, then per surviving stored pair t (5 values):
    // s.y_t, s_t.y, y.y_t, s_t.pg, y_t.pg
    const int drop = cnt == m ? head : -1;  // the slot the new pair would overwrite
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = 0.f;
    v[0] = f3(sf, yf);
    v[1] = f3(yf, yf);
    v[2] = f3(sf, sf);
    v[3] = f3(pgf, pgf);
    v[4] = f3(sf, pgf);
    v[5] = f3(yf, pgf);
#pragma unroll
    for (int j = 0; j < M; ++j) {
      if (6 + 5 * j + 4 < 32) {  // (j = M-1 only exists while the ring is full, and is the dropped pair then)
        if (j < cnt && slot[j] != drop) {
          const float4 s4 = S4[slot[j] * 32 + lane], y4 = Y4[slot[j] * 32 + lane];
          const float st[3] = {s4.x, s4.y, s4.z}, yt[3] = {y4.x, y4.y, y4.z};
          v[6 + 5 * j] = f3(sf, yt);
          v[6 + 5 * j + 1] = f3(st, yf);
          v[6 + 5 * j + 2] = f3(yf, yt);
          v[6 + 5 * j + 3] = f3(st, pgf);
          v[6 + 5 * j + 4] = f3(yt, pgf);
        }
      }
    }
    const float mine = transpose_reduce32(v, lane);  // lane l: the sum of value l
    RED[lane] = mine;
    __syncwarp();
    const float sy = RED[0], yy = RED[1], ss = RED[2];
    pgn2 = RED[3];
    const bool keep = sy > 1e-10f * sqrtf(ss) * sqrtf(yy);
    // Gram update, one lane per value: value 6 + 5j + q belongs to the j-th newest pair
    if (lane >= 6) {
      const int j = (lane - 6) / 5, q = (lane - 6) - 5 * j;
      if (j < cnt) {
        int st = head - 1 - j;
        if (st < 0) st += m;
        if (st != drop) {
          if (q == 3) Ug[st] = mine;
          if (q == 4) Wg[st] = mine;
          if (keep) {
            if (q == 0) SYg[head * M + st] = mine;  // s_new . y_t
            if (q == 1) SYg[st * M + head] = mine;  // s_t . y_new
            if (q == 2) {
              YYg[head * M + st] = mine;
              YYg[st * M + head] = mine;
            }
          }
        }
      }
    } else if (keep) {
      if (lane == 0) {
        SYg[head * M + head] = sy;
        RHO[head] = __fdividef(1.f, sy);
      }
      if (lane == 1) YYg[head * M + head] = yy;
      if (lane == 4) Ug[head] = mine;
      if (lane == 5) Wg[head] = mine;
    }
    if (!keep && cnt == m) {
      // the refused pair leaves the full ring as it is, so the oldest pair (slot head) stays in use -- and the batch
      // above skipped it as the pair about to be dropped: bring its s.pg, y.pg up to date here (warp-uniform, rare)
      const float4 s4 = S4[head * 32 + lane], y4 = Y4[head * 32 + lane];
      const float st[3] = {s4.x, s4.y, s4.z}, yt[3] = {y4.x, y4.y, y4.z};
      const float u = (float)wsum_x(f3(st, pgf)), wv = (float)wsum_x(f3(yt, pgf));
      if (lane == 0) {
        Ug[head] = u;
        Wg[head] = wv;
      }
    }
    if (keep) {
      S4[head * 32 + lane] = make_float4(sf[0], sf[1], sf[2], 0.f);
      Y4[head * 32 + lane] = make_float4(yf[0], yf[1], yf[2], 0.f);
      gamma = __fdividef(sy, yy);
      head = head + 1 == m ? 0 : head + 1;
      if (cnt < m) ++cnt;
    }
    __syncwarp();
    if (!exact && __all_sync(0xffffffffu, small)) break;  // xtol_rel, :173
  }
  {
    __syncwarp();
    V3 XB;
#pragma unroll
    for (int k = 0; k < 3; ++k) XB.v[k] = is_pt ? xb[3 * lane + k] : 0.0;
    if (is_dt) XB.v[0] = xb[nvar - 1];
    const double dtv = opt_time ? __shfl_sync(0xffffffffu, XB.v[0], n) : t.knot_span;
    double fo, gr[3], gdt;
    eval_warp<false>(g, dist, p, t, tc + b, n, mask, XB.v, dtv, lane, fo, gr, gdt);
    if (lane == 0) fbest[b] = fo;
  }
  if (lane == 0) neval_out[b] = neval;
}

}  // namespace

int bspline_optimize_batch_dev_impl(FuelMap* m, int B, int n_pts, int mask, const FuelOptParams* p,
                                    const FuelTrajConst* tc_dev, const FuelSolveParams* sp,
                                    double* x_dev, double* fbest_dev, int32_t* neval_dev) {
  if (B <= 0) return 0;
  const int need = n_pts + ((mask & FUELGPU_MINTIME) ? 1 : 0);
  if (need > 32)
    return fuel_fail(m, FUELGPU_EUNSUPPORTED, "optimize_batch supports at most 32 lanes (n_pts + dt)");
  static int use_vec = -1;  // FUELGPU_SOLVER=vec selects the vector-space two-loop recursion (A/B, debugging)
  if (use_vec < 0) {
    const char* e = getenv("FUELGPU_SOLVER");
    use_vec = (e && !strcmp(e, "vec")) ? 1 : 0;
  }
  if (use_vec || sp->lbfgs_m != 6) {  // the coefficient-space kernel is instantiated for the default history length
    const size_t smem = (size_t)WPB * 2 * sp->lbfgs_m * 96 * sizeof(double);
    FUEL_CUDA(m, cudaFuncSetAttribute(optimize_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    optimize_warp_kernel<<<(B + WPB - 1) / WPB, WPB * 32, smem, m->stream>>>(m->g, m->dist, *p, tc_dev, n_pts, mask, B, *sp,
                                                                        x_dev, fbest_dev, neval_dev);
  } else {
    constexpr int GM = 6;
    const size_t smem = (size_t)WPB * GRAM_FLOATS(GM) * sizeof(float);
    FUEL_CUDA(m, cudaFuncSetAttribute(optimize_gram_kernel<GM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    optimize_gram_kernel<GM><<<(B + WPB - 1) / WPB, WPB * 32, smem, m->stream>>>(m->g, m->dist, *p, tc_dev, n_pts, mask, B, *sp,
                                                                            x_dev, fbest_dev, neval_dev);
  }
  FUEL_LAUNCHES(m, 1);
  FUEL_CUDA(m, cudaGetLastError());
  return 0;
}
