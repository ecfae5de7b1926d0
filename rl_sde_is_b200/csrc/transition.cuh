// Cell probabilities of the tabular transition P[s', s, a], shared by the table builder (K4, tables.cu) and the
// tensor-free Bellman sweep (K6i, dp_implicit.cu): the normal CDF of the erf/erfc path and the constants of the
// Gauss-Legendre density recurrences of the quadrature path.
#pragma once
#include <cmath>

namespace rlsde {

// scipy.special.ndtr (cephes ndtr.c) branch structure, with CUDA's erf / erfc
__device__ __forceinline__ double ndtr(double a) {
  const double kSqrtH = 0.70710678118654752440;
  const double x = a * kSqrtH;
  const double z = fabs(x);
  double y;
  if (z < kSqrtH) {
    y = 0.5 + 0.5 * erf(x);
  } else {
    y = 0.5 * erfc(z);
    if (x > 0) y = 1.0 - y;
  }
  return y;
}

// ---- fast path: uniform state grid with fine cells (cell width <= 0.2 sd) -------------------------------
// P_cell = integral of the N(0,1) density over the cell [m - D/2, m + D/2] by 4-point Gauss-Legendre (truncation error
// 9e-14 at D = 0.25, 1e-14 at D = 0.2: the path is taken up to D = 0.2).  The nodes sit symmetrically at m +- a, m +- b,
// and phi(m +- o) = phi(m) exp(-o^2/2) exp(-+ m o), so
//     P = phi(m) * (Ya + Yb),   Ya = 2 D w_a exp(-a^2/2) cosh(m a),   Yb likewise with (w_b, b).
// Walking s' moves m by the constant step ds, and all three factors follow cheap recurrences:
//     phi(m + ds) = phi(m) r,   r <- r exp(-ds^2)                                (2 DMUL)
//     Y(m + ds)   = Y + dY,     dY <- dY + 4 sinh^2(o ds / 2) Y(m + ds)          (DADD + DFMA each; the second-difference
//                                                                                 form of cosh's three-term recurrence,
//                                                                                 stable because the small quantity is kept)
// 8 FP64 operations per entry, re-anchored with exact exp() every GL_ANCHOR cells and at most GL_SPAN_SD standard
// deviations (measured |P - reference formula| <= 5e-15 at config 3; tests hold 1e-13).
constexpr int GL_ANCHOR = 64;
constexpr double GL_SPAN_SD = 21.0;

struct GlConst {
  double inv_sd, dcell, dstep, rho;        // 1/sd, D, ds, exp(-ds^2)
  double off_a, off_b;                     // node offsets a, b
  double coef_a, coef_b;                   // 2 D w exp(-o^2/2)
  double mu_a, mu_b;                       // 4 sinh^2(o ds / 2)
  double sh_a, sh_b;                       // sinh(o ds / 2)
  double eh_a, eh_b;                       // exp(o ds / 2)
  double half_ds2;                         // ds^2 / 2
};

// the rule that picks the quadrature path: a uniform grid whose cells are at most 0.2 sd wide
static bool gl_path(long long Ns, int uniform_grid, double grid_step, double sigma, double dt, double h) {
  return uniform_grid && grid_step > 0.0 && Ns >= 2 && 2.0 * h / (sigma * sqrt(dt)) <= 0.2;
}

// steps between anchors for a recurrence step of step_sd standard deviations: at most GL_ANCHOR steps and at most
// GL_SPAN_SD standard deviations, so that phi at the anchor does not underflow (|m| < 37) while cells that matter
// (|m| < 9) are still ahead of it, and the relative error of r, which grows with |m ds|, stays small
static long long gl_anchor_steps(double step_sd) {
  const long long steps = (long long)(GL_SPAN_SD / step_sd);
  return steps < 1 ? 1 : (steps > GL_ANCHOR ? GL_ANCHOR : steps);
}

// host side: the constants of the recurrences are the same for every column; they travel as a kernel parameter (round 1
// formed them once per block behind a barrier: 4.1 warps per issue slot stalled there, profiles/r01/ncu_tables_gl_v2.txt)
static GlConst make_gl_const(double grid_step, double sigma, double dt, double h) {
  GlConst C;
  C.inv_sd = 1.0 / (sigma * sqrt(dt));
  C.dcell = 2.0 * h * C.inv_sd;
  C.dstep = grid_step * C.inv_sd;
  C.rho = exp(-C.dstep * C.dstep);
  C.half_ds2 = 0.5 * C.dstep * C.dstep;
  C.off_a = 0.4305681557970263 * C.dcell;
  C.off_b = 0.1699905217924281 * C.dcell;
  C.coef_a = 2.0 * C.dcell * 0.1739274225687269 * exp(-0.5 * C.off_a * C.off_a);
  C.coef_b = 2.0 * C.dcell * 0.3260725774312731 * exp(-0.5 * C.off_b * C.off_b);
  C.sh_a = sinh(0.5 * C.off_a * C.dstep);
  C.sh_b = sinh(0.5 * C.off_b * C.dstep);
  C.mu_a = 4.0 * C.sh_a * C.sh_a;
  C.mu_b = 4.0 * C.sh_b * C.sh_b;
  C.eh_a = exp(0.5 * C.off_a * C.dstep);
  C.eh_b = exp(0.5 * C.off_b * C.dstep);
  return C;
}

}  // namespace rlsde
