// On-device step control of the trust-region loop: everything scipy's trf_no_bounds does
// with scalars on the host (scipy/optimize/_lsq/trf.py:465-578, common.py:171-322,705-717)
// runs here in tiny kernels on the solver stream; the host only polls a status struct.
#pragma once
#include "common.cuh"

namespace lcba {

struct Ctl {
  double cost, cost_new, Delta, reg_term, g_norm, gh2, x_norm, Jg2;
  double c0, c1, predicted, actual, ratio, step_norm, step_h_norm, mu;
  double camp[4];       // camera parts of (|g_h|^2, |x*scl|^2, |x|^2, max|g|)
  double BS[3], gS0, R00, R01, R11, gtgt, gtp, pp;   // 2-D model in the orthonormal basis
  double aa, ab, bb, JAA, JAB, JBB;                  // Gram totals of k_ctl_sub (lcba_debug_step)
  double ftol, xtol;
  int accept, term, chol_fail, nonfinite, first, retry, degenerate, pad;
};

// ---- 2-D trust-region subproblem  min 0.5 p^T B p + g^T p, |p| <= Delta -----------------
// scipy solves the boundary case through the quartic of the tangent half-angle and takes
// the best real root (common.py:171-219); the global minimiser is computed here from the
// 2x2 eigen-decomposition and the secular equation (same point, B is a Gram matrix => PSD).
struct TR2 { double p0, p1; int newton; };

__host__ __device__ inline TR2 solve_tr2d(double B00, double B01, double B11, double g0, double g1,
                                          double Delta) {
  TR2 r;
  r.newton = 0;
  const double d11 = (B00 > 0.0) ? B11 - B01 * B01 / B00 : -1.0;
  if (B00 > 0.0 && d11 > 0.0) {
    const double l00 = sqrt(B00), l10 = B01 / l00, l11 = sqrt(d11);
    const double y0 = -g0 / l00;
    const double y1 = (-g1 - l10 * y0) / l11;
    const double p1 = y1 / l11;
    const double p0 = (y0 - l10 * p1) / l00;
    if (p0 * p0 + p1 * p1 <= Delta * Delta) { r.p0 = p0; r.p1 = p1; r.newton = 1; return r; }
  }
  const double tr = B00 + B11, df = B00 - B11;
  const double rad = hypot(df, 2.0 * B01);
  const double l1 = 0.5 * (tr - rad), l2 = 0.5 * (tr + rad);
  double vx = 1.0, vy = 0.0;            // eigenvector of l2
  if (rad > 0.0) {
    const double ax = B01, ay = l2 - B00;     // (B - l2 I) v = 0, first row
    const double bx = l2 - B11, by = B01;     // second row
    if (ax * ax + ay * ay >= bx * bx + by * by) { vx = ax; vy = ay; } else { vx = bx; vy = by; }
    const double nv = hypot(vx, vy);
    if (nv > 0.0) { vx /= nv; vy /= nv; } else { vx = 1.0; vy = 0.0; }
  }
  const double ux = -vy, uy = vx;       // eigenvector of l1
  const double h1 = ux * g0 + uy * g1, h2 = vx * g0 + vy * g1;
  const double gn = hypot(g0, g1);
  if (gn == 0.0) {                      // flat model: any boundary point along u if l1 < 0
    r.p0 = (l1 < 0.0) ? Delta * ux : 0.0;
    r.p1 = (l1 < 0.0) ? Delta * uy : 0.0;
    return r;
  }
  double lo = fmax(0.0, -l1);
  double hi = gn / Delta - l1;
  if (hi < lo) hi = lo;
  // hard case: no component along the lowest eigenvector and the pole is not reached
  if (l1 + lo <= 0.0) {
    const double e2 = l2 + lo;
    const double q2 = (e2 > 0.0) ? -h2 / e2 : 0.0;
    if (fabs(h1) <= 1e-300 && q2 * q2 <= Delta * Delta) {
      const double tau = sqrt(fmax(0.0, Delta * Delta - q2 * q2));
      r.p0 = q2 * vx + tau * ux;
      r.p1 = q2 * vy + tau * uy;
      return r;
    }
  }
  double mu = lo;
  if (l1 + mu <= 0.0) mu = lo + 1e-16 * fmax(1.0, fabs(hi));
  double blo = lo, bhi = hi;
  for (int it = 0; it < 200; ++it) {
    const double e1 = l1 + mu, e2 = l2 + mu;
    const double q1 = h1 / e1, q2 = h2 / e2;
    const double pn2 = q1 * q1 + q2 * q2;
    const double pn = sqrt(pn2);
    if (pn > Delta) blo = mu; else bhi = mu;
    if (fabs(pn - Delta) <= 4e-16 * Delta) break;
    const double dq = q1 * q1 / e1 + q2 * q2 / e2;       // -0.5 d(pn2)/dmu
    double nxt = mu + (pn - Delta) / Delta * pn2 / dq;
    if (!(nxt > blo && nxt < bhi)) nxt = 0.5 * (blo + bhi);
    if (nxt == mu) break;
    mu = nxt;
  }
  const double q1 = -h1 / (l1 + mu), q2 = -h2 / (l2 + mu);
  double p0 = q1 * ux + q2 * vx, p1 = q1 * uy + q2 * vy;
  const double pn = hypot(p0, p1);
  if (pn > 0.0) { p0 *= Delta / pn; p1 *= Delta / pn; }
  r.p0 = p0;
  r.p1 = p1;
  return r;
}

// Solve the 2-D problem in the orthonormal basis and map it back to coefficients of
// (g_h, gn_h):  step_h = c0 * g_h + c1 * gn_h  (trf.py:496-511).
__device__ inline void ctl_solve_subspace(Ctl* c) {
  double p0, p1;
  if (c->degenerate) {
    // gn_h parallel to g_h: 1-D problem along q1
    const double B = c->BS[0], g = c->gS0;
    double p = (B > 0.0) ? -g / B : -copysign(c->Delta, g);
    if (fabs(p) > c->Delta) p = copysign(c->Delta, p);
    p0 = p; p1 = 0.0;
    c->c1 = 0.0;
    c->c0 = p0 / c->R00;
  } else {
    const TR2 t = solve_tr2d(c->BS[0], c->BS[1], c->BS[2], c->gS0, 0.0, c->Delta);
    p0 = t.p0; p1 = t.p1;
    c->c1 = p1 / c->R11;
    c->c0 = (p0 - c->R01 * c->c1) / c->R00;
  }
  c->predicted = -(0.5 * (c->BS[0] * p0 * p0 + 2.0 * c->BS[1] * p0 * p1 + c->BS[2] * p1 * p1) +
                   c->gS0 * p0);
  c->step_h_norm = hypot(p0, p1);
  const double s2 = c->c0 * c->c0 * c->gtgt + 2.0 * c->c0 * c->c1 * c->gtp + c->c1 * c->c1 * c->pp;
  c->step_norm = sqrt(fmax(0.0, s2));
}

// after k_linearize + reduction: camera scaling (common.py:598-610), g~_c, camera sums
// camsum[c*22 + a] = g_c, camsum[c*22 + 11 + a] = diag(J^T J); camsum[22C] = sum r^2
// cam_fixed (C x 11, may be NULL): entries held constant, like every entry under fix_cameras
__global__ void __launch_bounds__(256)
k_ctl_lin(const double* __restrict__ camsum, const double* __restrict__ cams,
          double* __restrict__ scl_c, double* __restrict__ gt_c, double* __restrict__ g_c, int C,
          Ctl* __restrict__ ctl, int first, int fix_cameras, const uint8_t* __restrict__ cam_fixed,
          int shared_intr) {
  __shared__ double s_red[32];
  __shared__ double s_sh[6];   // shared-intrinsics mode: summed gradient / diag of (f, k1, k2)
  if (shared_intr) {
    if (threadIdx.x < 6) {
      const int a = 6 + threadIdx.x % 3, off = threadIdx.x < 3 ? 0 : 11;
      double sum = 0.0;
      for (int c = 0; c < C; ++c) sum += camsum[c * 22 + off + a];
      s_sh[threadIdx.x] = sum;
    }
    __syncthreads();
  }
  double gh2 = 0, xs2 = 0, x2 = 0, gmax = 0;
  for (int i = threadIdx.x; i < C * NCP; i += blockDim.x) {
    const int c = i / NCP, a = i % NCP;
    if (fix_cameras || (cam_fixed && cam_fixed[i])) {   // constants: no gradient, no scale, no norm share
      scl_c[i] = 1.0; g_c[i] = 0.0; gt_c[i] = 0.0;
      continue;
    }
    const bool sh = shared_intr && a >= 6 && a <= 8;   // one parameter replicated over cameras
    const double g = sh ? s_sh[a - 6] : camsum[c * 22 + a];
    double s = sqrt(sh ? s_sh[3 + a - 6] : camsum[c * 22 + 11 + a]);
    if (first) { if (s == 0.0) s = 1.0; } else s = fmax(s, scl_c[i]);
    if (sh && c > 0) {          // replicas carry the values but count once in the norms
      scl_c[i] = s; g_c[i] = g; gt_c[i] = g / s / s;
      continue;
    }
    scl_c[i] = s;
    g_c[i] = g;
    const double gh = g / s, x = cams[i];
    gt_c[i] = gh / s;
    gh2 = fma(gh, gh, gh2);
    xs2 = fma(x * s, x * s, xs2);
    x2 = fma(x, x, x2);
    gmax = fmax(gmax, fabs(g));
  }
  const double a0 = block_sum(gh2, s_red), a1 = block_sum(xs2, s_red), a2 = block_sum(x2, s_red);
  const double a3 = block_max(gmax, s_red);
  if (threadIdx.x == 0) {
    ctl->camp[0] = a0; ctl->camp[1] = a1; ctl->camp[2] = a2; ctl->camp[3] = a3;
    if (first) ctl->cost = 0.5 * camsum[22 * C];
    const double ss = camsum[22 * C];
    if (!(ss - ss == 0.0)) ctl->nonfinite = 1;
  }
}

// after k_point_prep + reduction (red[0..2] sums, red[3] max)
__global__ void k_ctl_lin2(const double* __restrict__ red, Ctl* __restrict__ ctl, int first) {
  ctl->gh2 = ctl->camp[0] + red[0];
  ctl->x_norm = sqrt(ctl->camp[2] + red[2]);
  ctl->g_norm = fmax(ctl->camp[3], red[3]);
  if (first) {
    double d = sqrt(ctl->camp[1] + red[1]);     // Delta = |x0 * scale_inv| (trf.py:443)
    if (d == 0.0) d = 1.0;
    ctl->Delta = d;
    ctl->mu = 0.0;
  }
}

// reg_term from the 1-D Cauchy model (trf.py:488-492, common.py:251-322).  dhg2 (bounded loop only, else NULL):
// sum diag_h g_h^2, the diagonal's share of the model's curvature (trf.py:327)
__global__ void k_ctl_reg(const double* __restrict__ red, Ctl* __restrict__ ctl, const double* __restrict__ dhg2) {
  const double Jg2 = dhg2 ? red[0] + *dhg2 : red[0];
  ctl->Jg2 = Jg2;
  const double a = 0.5 * Jg2, b = -ctl->gh2;
  const double ub = ctl->Delta / sqrt(ctl->gh2);
  // minimise t*(a*t + b) over {0, ub, extremum in (0, ub)}
  double best = 0.0;
  double y = ub * (a * ub + b);
  if (y < best) best = y;
  if (a != 0.0) {
    const double ex = -0.5 * b / a;
    if (ex > 0.0 && ex < ub) { y = ex * (a * ex + b); if (y < best) best = y; }
  }
  ctl->reg_term = -best / (ctl->Delta * ctl->Delta);
}

// after k_backsub + reduction: red[0..8]; adds the camera parts of the parameter-space
// Gram sums, orthonormalises (g_h, gn_h) through the Cholesky factor of their Gram matrix
// and solves the 2-D problem.
__global__ void __launch_bounds__(256)
k_ctl_sub(const double* __restrict__ red, const double* __restrict__ g_c,
          const double* __restrict__ gt_c, const double* __restrict__ pc,
          const double* __restrict__ scl_c, int C, Ctl* __restrict__ ctl,
          const int* __restrict__ chol_fail, double* __restrict__ coef, int shared_intr) {
  __shared__ double s_red[32];
  double v[6] = {0, 0, 0, 0, 0, 0};
  for (int i = threadIdx.x; i < C * NCP; i += blockDim.x) {
    if (shared_intr && i >= NCP && i % NCP >= 6 && i % NCP <= 8) continue;   // replicas
    const double s = scl_c[i];
    const double ah = g_c[i] / s, bh = pc[i] * s, gt = gt_c[i], p = pc[i];
    v[0] = fma(ah, ah, v[0]); v[1] = fma(ah, bh, v[1]); v[2] = fma(bh, bh, v[2]);
    v[3] = fma(gt, gt, v[3]); v[4] = fma(gt, p, v[4]);  v[5] = fma(p, p, v[5]);
  }
  double w[6];
  for (int k = 0; k < 6; ++k) w[k] = block_sum(v[k], s_red);
  if (threadIdx.x != 0) return;
  const double JAA = red[0], JAB = red[1], JBB = red[2];
  const double aa = red[3] + w[0], ab = red[4] + w[1], bb = red[5] + w[2];
  ctl->gtgt = red[6] + w[3];
  ctl->gtp = red[7] + w[4];
  ctl->pp = red[8] + w[5];
  ctl->aa = aa; ctl->ab = ab; ctl->bb = bb;
  ctl->JAA = JAA; ctl->JAB = JAB; ctl->JBB = JBB;
  ctl->chol_fail = *chol_fail;
  const double chk = JAB + JBB + ab + bb;
  ctl->retry = (!(chk - chk == 0.0) || ctl->chol_fail) ? 1 : 0;
  const double R00 = sqrt(aa), R01 = ab / R00;
  const double d = bb - R01 * R01;
  ctl->R00 = R00; ctl->R01 = R01;
  ctl->gS0 = R00;
  ctl->BS[0] = JAA / aa;
  if (!(d > 1e-24 * bb)) {
    ctl->degenerate = 1;
    ctl->R11 = 0.0; ctl->BS[1] = 0.0; ctl->BS[2] = 0.0;
  } else {
    ctl->degenerate = 0;
    const double R11 = sqrt(d);
    ctl->R11 = R11;
    // B_S = R^-T GJ R^-1 with R^-1 = [[1/R00, -R01/(R00 R11)], [0, 1/R11]]
    const double i00 = 1.0 / R00, i01 = -R01 / (R00 * R11), i11 = 1.0 / R11;
    ctl->BS[1] = i00 * (JAA * i01 + JAB * i11);
    ctl->BS[2] = i01 * (JAA * i01 + JAB * i11) + i11 * (JAB * i01 + JBB * i11);
  }
  ctl_solve_subspace(ctl);
  coef[0] = ctl->c0;
  coef[1] = ctl->c1;
}

// after the trial residual: red[0] = sum r_new^2 (trf.py:503-541)
__global__ void k_ctl_trial(const double* __restrict__ red, Ctl* __restrict__ ctl,
                            double* __restrict__ coef) {
  const double ss = red[0];
  ctl->term = -1;
  ctl->accept = 0;
  if (!(ss - ss == 0.0)) {              // non-finite residuals: shrink and retry (trf.py:519-521)
    ctl->Delta = 0.25 * ctl->step_h_norm;
    ctl->actual = -1.0;
    ctl->cost_new = ss;
    ctl_solve_subspace(ctl);
    coef[0] = ctl->c0; coef[1] = ctl->c1;
    return;
  }
  const double cost_new = 0.5 * ss;
  ctl->cost_new = cost_new;
  const double actual = ctl->cost - cost_new;
  const double pred = ctl->predicted;
  double ratio;
  if (pred > 0.0) ratio = actual / pred;
  else if (pred == 0.0 && actual == 0.0) ratio = 1.0;
  else ratio = 0.0;
  double Delta_new = ctl->Delta;
  if (ratio < 0.25) Delta_new = 0.25 * ctl->step_h_norm;
  else if (ratio > 0.75 && ctl->step_h_norm > 0.95 * ctl->Delta) Delta_new = 2.0 * ctl->Delta;
  ctl->actual = actual;
  ctl->ratio = ratio;
  const bool f_ok = actual < ctl->ftol * ctl->cost && ratio > 0.25;
  const bool x_ok = ctl->step_norm < ctl->xtol * (ctl->xtol + ctl->x_norm);
  int term = -1;
  if (f_ok && x_ok) term = 4; else if (f_ok) term = 2; else if (x_ok) term = 3;
  ctl->term = term;
  if (term < 0) ctl->Delta = Delta_new;
  if (actual > 0.0) {
    ctl->accept = 1;
  } else if (term < 0) {
    ctl_solve_subspace(ctl);            // next trial with the shrunken radius
    coef[0] = ctl->c0; coef[1] = ctl->c1;
  }
}

__global__ void k_ctl_commit(Ctl* __restrict__ ctl) { ctl->cost = ctl->cost_new; }

}  // namespace lcba
