// Box bounds: the reflective half of scipy's TRF (trf_bounds and select_step, scipy/optimize/_lsq/trf.py:129-412,
// helpers in common.py), with the exact Schur solve in place of LSMR.
//
// Per-entry vectors of a bounded solve run over one index space, cameras first: i < nc is camera entry i, i >= nc
// is point coordinate i - nc.  With s the Jacobi column norm and (v, dv) the Coleman-Li vector at (x, g):
//   v <- v * s where dv != 0,  d = sqrt(v) / s,  diag_h = g dv / s,  g~ = d^2 g
// The solver keeps sd = 1 / d where the unbounded loop keeps s (for dv = 0, sd = s), so the Gram sums of the 2-D
// subspace need no change, and the damping of the Gauss-Newton system becomes e = (diag_h + reg_term) sd^2.
// Held entries and entries without a finite bound on the side the gradient points to have dv = 0.
#pragma once
#include "common.cuh"
#include "control.cuh"

namespace lcba {

struct Bnd {
  double dhg2;       // sum diag_h g_h^2: the diagonal's share of the Cauchy model along -g_h
  double ag_bound;   // step_size_to_bound(x, -g~)
  double theta;      // max(0.995, 1 - |g v|_inf)
  double p_stride;   // step_size_to_bound(x, p) of the current trial's subspace step p
  double c_p, c_r, c_ag;   // chosen step: mode 0: c_p p ; 1: p_stride p + c_r r ; 2: -c_ag g~
  int inb, mode, pad[2];
};

// step_size_to_bound (common.py:357-386) of one entry: inf where s == 0.  Every kernel that compares the result with
// a reduced minimum calls this one function, so equal inputs give equal bits.
__device__ __forceinline__ double bnd_step_to_bound(double x, double s, double lb, double ub) {
  if (s == 0.0) return INFINITY;
  return fmax(__ddiv_rn(__dsub_rn(lb, x), s), __ddiv_rn(__dsub_rn(ub, x), s));
}

// CL_scaling_vector (common.py:683-702) and the hat-space quantities of one free entry.
struct BndScaled { double sd, dh, gt, gh, gv, xsv; };
__device__ __forceinline__ BndScaled bnd_scale(double g, double s, double x, double lb, double ub) {
  double v = 1.0, dv = 0.0;
  if (g < 0.0 && isfinite(ub)) { v = ub - x; dv = -1.0; }
  if (g > 0.0 && isfinite(lb)) { v = x - lb; dv = 1.0; }
  BndScaled r;
  r.gv = fabs(g * v);                 // |g v|_inf uses v before the scaling (trf.py:263-265)
  if (dv != 0.0) v *= s;
  const double sv = sqrt(v);
  r.sd = s / sv;
  r.dh = g * dv / s;
  r.gh = g / r.sd;
  r.gt = r.gh / r.sd;
  r.xsv = x * s / sv;                 // Delta0 = |x0 s / sqrt(v)| (trf.py:234)
  return r;
}

// Column ops of the bounded partial sums: [0, nsum) sum, [nsum, nsum + nmax) max of values >= 0, the rest min.
// One CTA per column, fixed order.
__global__ void k_reduce_ops(const double* __restrict__ part, int nblocks, int K, int nsum, int nmax,
                             double* __restrict__ out) {
  __shared__ double s_red[32];
  __shared__ double s_min[256];
  const int j = blockIdx.x;
  const int op = j < nsum ? 0 : (j < nsum + nmax ? 1 : 2);
  double s = op == 2 ? INFINITY : 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) {
    const double v = part[(size_t)b * K + j];
    s = op == 0 ? s + v : (op == 1 ? fmax(s, v) : fmin(s, v));
  }
  if (op == 0) s = block_sum(s, s_red);
  else if (op == 1) s = block_max(s, s_red);
  else {
    s_min[threadIdx.x] = s;
    __syncthreads();
    for (int w = blockDim.x / 2; w > 0; w >>= 1) {
      if (threadIdx.x < w) s_min[threadIdx.x] = fmin(s_min[threadIdx.x], s_min[threadIdx.x + w]);
      __syncthreads();
    }
    s = s_min[0];
  }
  if (threadIdx.x == 0) out[j] = s;
}

// block-wide min of a value (256 threads), result valid in every thread
__device__ __forceinline__ double bnd_block_min(double v, double* s_min) {
  s_min[threadIdx.x] = v;
  __syncthreads();
  for (int w = blockDim.x / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) s_min[threadIdx.x] = fmin(s_min[threadIdx.x], s_min[threadIdx.x + w]);
    __syncthreads();
  }
  const double r = s_min[0];
  __syncthreads();
  return r;
}

// ---- linearisation ---------------------------------------------------------------------------------------------
// Points: k_point_prep of the bounded loop.  part[block][0..5]: sums |g_h|^2, |x s / sqrt(v)|^2, |x|^2,
// sum diag_h g_h^2; max |g v|; min step_size_to_bound(x, -g~).  lb / ub / sd / dh are the point parts.
constexpr int BPP_K = 6;
__global__ void __launch_bounds__(256)
k_bnd_point_prep(double* __restrict__ Vg, const double* __restrict__ pts, double* __restrict__ scl,
                 double* __restrict__ gt, long long P, int first, const uint8_t* __restrict__ pt_fixed,
                 const double* __restrict__ lb, const double* __restrict__ ub, double* __restrict__ sd,
                 double* __restrict__ dh, double* __restrict__ part) {
  __shared__ double s_red[32];
  __shared__ double s_min[256];
  double gh2 = 0, xs2 = 0, x2 = 0, dg2 = 0, gmax = 0, agb = INFINITY;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += stride) {
    if (pt_fixed && pt_fixed[p]) {
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        scl[3 * p + a] = 1.0; gt[3 * p + a] = 0.0; Vg[p * 9 + 6 + a] = 0.0;
        sd[3 * p + a] = 1.0; dh[3 * p + a] = 0.0;
      }
      continue;
    }
    const double* v = Vg + p * 9;
    const double d[3] = {v[0], v[3], v[5]};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const long long i = 3 * p + a;
      double s = sqrt(d[a]);
      if (first) { if (s == 0.0) s = 1.0; } else s = fmax(s, scl[i]);
      scl[i] = s;
      const double x = pts[i];
      const BndScaled b = bnd_scale(v[6 + a], s, x, lb[i], ub[i]);
      sd[i] = b.sd; dh[i] = b.dh; gt[i] = b.gt;
      gh2 = fma(b.gh, b.gh, gh2);
      xs2 = fma(b.xsv, b.xsv, xs2);
      x2 = fma(x, x, x2);
      dg2 = fma(b.dh * b.gh, b.gh, dg2);
      gmax = fmax(gmax, b.gv);
      agb = fmin(agb, bnd_step_to_bound(x, -b.gt, lb[i], ub[i]));
    }
  }
  const double a0 = block_sum(gh2, s_red), a1 = block_sum(xs2, s_red), a2 = block_sum(x2, s_red);
  const double a3 = block_sum(dg2, s_red), a4 = block_max(gmax, s_red);
  const double a5 = bnd_block_min(agb, s_min);
  if (threadIdx.x == 0) {
    double* o = part + (size_t)blockIdx.x * BPP_K;
    o[0] = a0; o[1] = a1; o[2] = a2; o[3] = a3; o[4] = a4; o[5] = a5;
  }
}

// Cameras, then the totals: k_ctl_lin + k_ctl_lin2 of the bounded loop (no fix_cameras, no shared intrinsics).
// red: the reduced point values of k_bnd_point_prep (all-reduced over the ranks).
__global__ void __launch_bounds__(256)
k_bnd_ctl_lin(const double* __restrict__ camsum, const double* __restrict__ cams, double* __restrict__ scl_c,
              double* __restrict__ gt_c, double* __restrict__ g_c, int C, const uint8_t* __restrict__ cam_fixed,
              const double* __restrict__ lb, const double* __restrict__ ub, double* __restrict__ sd,
              double* __restrict__ dh, const double* __restrict__ red, Ctl* __restrict__ ctl,
              Bnd* __restrict__ bnd, int first) {
  __shared__ double s_red[32];
  __shared__ double s_min[256];
  double gh2 = 0, xs2 = 0, x2 = 0, dg2 = 0, gmax = 0, agb = INFINITY;
  for (int i = threadIdx.x; i < C * NCP; i += blockDim.x) {
    const int c = i / NCP, a = i % NCP;
    if (cam_fixed && cam_fixed[i]) {
      scl_c[i] = 1.0; g_c[i] = 0.0; gt_c[i] = 0.0; sd[i] = 1.0; dh[i] = 0.0;
      continue;
    }
    const double g = camsum[c * 22 + a];
    double s = sqrt(camsum[c * 22 + 11 + a]);
    if (first) { if (s == 0.0) s = 1.0; } else s = fmax(s, scl_c[i]);
    scl_c[i] = s;
    g_c[i] = g;
    const double x = cams[i];
    const BndScaled b = bnd_scale(g, s, x, lb[i], ub[i]);
    sd[i] = b.sd; dh[i] = b.dh; gt_c[i] = b.gt;
    gh2 = fma(b.gh, b.gh, gh2);
    xs2 = fma(b.xsv, b.xsv, xs2);
    x2 = fma(x, x, x2);
    dg2 = fma(b.dh * b.gh, b.gh, dg2);
    gmax = fmax(gmax, b.gv);
    agb = fmin(agb, bnd_step_to_bound(x, -b.gt, lb[i], ub[i]));
  }
  const double a0 = block_sum(gh2, s_red), a1 = block_sum(xs2, s_red), a2 = block_sum(x2, s_red);
  const double a3 = block_sum(dg2, s_red), a4 = block_max(gmax, s_red);
  const double a5 = bnd_block_min(agb, s_min);
  if (threadIdx.x != 0) return;
  const double ss = camsum[22 * C];
  if (first) ctl->cost = 0.5 * ss;
  if (!(ss - ss == 0.0)) ctl->nonfinite = 1;
  ctl->gh2 = a0 + red[0];
  ctl->x_norm = sqrt(a2 + red[2]);
  ctl->g_norm = fmax(a4, red[4]);
  if (first) {
    double d = sqrt(a1 + red[1]);
    if (d == 0.0) d = 1.0;
    ctl->Delta = d;
    ctl->mu = 0.0;
  }
  bnd->dhg2 = a3 + red[3];
  bnd->ag_bound = fmin(a5, red[5]);
  bnd->theta = fmax(0.995, 1.0 - ctl->g_norm);
}

// ---- diagonal share of the subspace Gram matrix: S^T diag_h S (trf.py:336) --------------------------------------
// part[block][0..2] = sums of diag_h a^2, diag_h a b, diag_h b^2 with a = g_h, b = gn_h.  Cameras count on one rank.
__global__ void __launch_bounds__(256)
k_bnd_gram(const double* __restrict__ g_c, const double* __restrict__ pc, const double* __restrict__ Vg,
           const double* __restrict__ gn_p, const double* __restrict__ sd, const double* __restrict__ dh, int nc,
           long long n, int count_cams, double* __restrict__ part) {
  __shared__ double s_red[32];
  double v0 = 0, v1 = 0, v2 = 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if (i < nc && !count_cams) continue;
    const double e = dh[i];
    if (e == 0.0) continue;
    const long long j = i - nc;
    const double g = i < nc ? g_c[i] : Vg[(j / 3) * 9 + 6 + j % 3];
    const double gn = i < nc ? pc[i] : gn_p[j];
    const double a = g / sd[i], b = gn * sd[i];
    v0 = fma(e * a, a, v0); v1 = fma(e * a, b, v1); v2 = fma(e * b, b, v2);
  }
  const double a0 = block_sum(v0, s_red), a1 = block_sum(v1, s_red), a2 = block_sum(v2, s_red);
  if (threadIdx.x == 0) {
    double* o = part + (size_t)blockIdx.x * 3;
    o[0] = a0; o[1] = a1; o[2] = a2;
  }
}

__global__ void k_bnd_gram_add(double* __restrict__ red, const double* __restrict__ add) {
  red[0] += add[0]; red[1] += add[1]; red[2] += add[2];
}

// ---- select_step (trf.py:129-224) --------------------------------------------------------------------------------
// A: the subspace step p = c0 g~ + c1 gn into bp; part[block][0] = max of "x + p leaves the box", [1] = min of
// step_size_to_bound(x, p).
__global__ void __launch_bounds__(256)
k_bnd_a(const double* __restrict__ cams, const double* __restrict__ pts, const double* __restrict__ gt_c,
        const double* __restrict__ gt_p, const double* __restrict__ pc, const double* __restrict__ gn_p,
        const double* __restrict__ coef, const double* __restrict__ lb, const double* __restrict__ ub, int nc,
        long long n, double* __restrict__ bp, double* __restrict__ part) {
  __shared__ double s_red[32];
  __shared__ double s_min[256];
  const double c0 = coef[0], c1 = coef[1];
  double out = 0.0, smin = INFINITY;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const bool cm = i < nc;
    const double x = cm ? cams[i] : pts[i - nc];
    const double p = cm ? fma(c1, pc[i], c0 * gt_c[i]) : fma(c1, gn_p[i - nc], c0 * gt_p[i - nc]);
    bp[i] = p;
    const double xp = x + p;
    if (!(xp >= lb[i] && xp <= ub[i])) out = 1.0;
    smin = fmin(smin, bnd_step_to_bound(x, p, lb[i], ub[i]));
  }
  const double a0 = block_max(out, s_red);
  const double a1 = bnd_block_min(smin, s_min);
  if (threadIdx.x == 0) { part[(size_t)blockIdx.x * 2] = a0; part[(size_t)blockIdx.x * 2 + 1] = a1; }
}

__global__ void k_bnd_ctl_a(const double* __restrict__ red, Bnd* __restrict__ bnd) {
  bnd->inb = red[0] == 0.0 ? 1 : 0;
  bnd->p_stride = red[1];
  bnd->mode = 0;
  bnd->c_p = 1.0;
}

__device__ __forceinline__ bool bnd_hit(double x, double p, double lb, double ub, double p_stride) {
  return bnd_step_to_bound(x, p, lb, ub) == p_stride;
}

// B (only when x + p leaves the box): the reflected direction r = p with the hit entries negated into br.
// part[block][0..4] sums: diag_h p_h^2, diag_h p_h r_h, g . r, |p_h|^2 and |p|^2 over the hits; [5] min of
// step_size_to_bound(x + p_stride p, r).  Cameras count in the sums on one rank.
constexpr int BB_K = 6;
__global__ void __launch_bounds__(256)
k_bnd_b(const double* __restrict__ cams, const double* __restrict__ pts, const double* __restrict__ g_c,
        const double* __restrict__ Vg, const double* __restrict__ bp, const double* __restrict__ sd,
        const double* __restrict__ dh, const double* __restrict__ lb, const double* __restrict__ ub, int nc,
        long long n, int count_cams, const Bnd* __restrict__ bnd, double* __restrict__ br,
        double* __restrict__ part) {
  if (bnd->inb) return;
  __shared__ double s_red[32];
  __shared__ double s_min[256];
  const double ps = bnd->p_stride;
  double v[5] = {0, 0, 0, 0, 0};
  double smin = INFINITY;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const bool cm = i < nc;
    const long long j = i - nc;
    const double x = cm ? cams[i] : pts[j];
    const double p = bp[i];
    const bool hit = bnd_hit(x, p, lb[i], ub[i], ps);
    const double r = hit ? -p : p;
    br[i] = r;
    smin = fmin(smin, bnd_step_to_bound(x + ps * p, r, lb[i], ub[i]));
    if (cm && !count_cams) continue;
    const double g = cm ? g_c[i] : Vg[(j / 3) * 9 + 6 + j % 3];
    const double ph = p * sd[i], e = dh[i] * ph * ph;
    v[0] += e;
    v[1] += hit ? -e : e;
    v[2] = fma(g, r, v[2]);
    if (hit) { v[3] = fma(ph, ph, v[3]); v[4] = fma(p, p, v[4]); }
  }
  double o[BB_K];
  for (int k = 0; k < 5; ++k) o[k] = block_sum(v[k], s_red);
  o[5] = bnd_block_min(smin, s_min);
  if (threadIdx.x == 0)
    for (int k = 0; k < BB_K; ++k) part[(size_t)blockIdx.x * BB_K + k] = o[k];
}

// |J r|^2 and (J p).(J r) over the observations (k_jdot with two vectors); only when x + p leaves the box
__global__ void __launch_bounds__(256)
k_bnd_jdot(const double* __restrict__ tab, const double* __restrict__ pts, const uint8_t* __restrict__ cam,
           const int32_t* __restrict__ pt, const double* __restrict__ wgt, const double* __restrict__ bp,
           const double* __restrict__ br, long long N, int C, const Bnd* __restrict__ bnd,
           double* __restrict__ part) {
  if (bnd->inb) return;
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  double* s_p = s_dyn + C * CAMTAB;
  double* s_r = s_p + C * NCP;
  __shared__ double s_red[32];
  load_tables_smem(tab, s_tab, C);
  for (int i = threadIdx.x; i < C * NCP; i += blockDim.x) { s_p[i] = bp[i]; s_r[i] = br[i]; }
  __syncthreads();
  const double* pp = bp + C * NCP;
  const double* rp = br + C * NCP;
  double arr = 0.0, apr = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    const int c = cam[i];
    const long long p = pt[i];
    const double w = wgt ? wgt[i] : 1.0;
    ObsLin L;
    obs_linearize<false>(s_tab + c * CAMTAB, pts[3 * p], pts[3 * p + 1], pts[3 * p + 2], 0.0, 0.0, w, L);
    const double* pc = s_p + c * NCP;
    const double* rc = s_r + c * NCP;
    double p0 = w * pc[9], p1 = w * pc[10], r0 = w * rc[9], r1 = w * rc[10];
#pragma unroll
    for (int a = 0; a < 9; ++a) {
      p0 = fma(L.Jc[0][a], pc[a], p0); p1 = fma(L.Jc[1][a], pc[a], p1);
      r0 = fma(L.Jc[0][a], rc[a], r0); r1 = fma(L.Jc[1][a], rc[a], r1);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double vp = pp[3 * p + a], vr = rp[3 * p + a];
      p0 = fma(L.Jp[0][a], vp, p0); p1 = fma(L.Jp[1][a], vp, p1);
      r0 = fma(L.Jp[0][a], vr, r0); r1 = fma(L.Jp[1][a], vr, r1);
    }
    arr = fma(r0, r0, fma(r1, r1, arr));
    apr = fma(p0, r0, fma(p1, r1, apr));
  }
  const double a0 = block_sum(arr, s_red), a1 = block_sum(apr, s_red);
  if (threadIdx.x == 0) { part[(size_t)blockIdx.x * 2] = a0; part[(size_t)blockIdx.x * 2 + 1] = a1; }
}

// minimize_quadratic_1d (common.py:325-354): min of t (a t + b) + c over [lb, ub]
__device__ inline void bnd_min_quad(double a, double b, double lb, double ub, double c, double& t, double& y) {
  t = lb;
  y = lb * (a * lb + b) + c;
  const double yu = ub * (a * ub + b) + c;
  if (yu < y) { t = ub; y = yu; }
  if (a != 0.0) {
    const double ex = -0.5 * b / a;
    if (lb < ex && ex < ub) {
      const double ye = ex * (a * ex + b) + c;
      if (ye < y) { t = ex; y = ye; }
    }
  }
}

// The three candidates of select_step and the choice; writes the chosen step's predicted reduction and norms into
// ctl, where k_ctl_trial reads them.  rb: k_bnd_b's six values, rj: k_bnd_jdot's two.  In the box the subspace
// step stands as k_ctl_sub / k_ctl_trial left it.
__global__ void k_bnd_select(const double* __restrict__ rb, const double* __restrict__ rj, Ctl* __restrict__ ctl,
                             Bnd* __restrict__ bnd) {
  if (bnd->inb) return;
  const double Delta = ctl->Delta, theta = bnd->theta, ps = bnd->p_stride;
  const double c0 = ctl->c0, c1 = ctl->c1;
  // the subspace step's model: value(t p_h) = 0.5 q t^2 + l t (B_S and g_S include the diagonal)
  const double q = c0 * c0 * ctl->JAA + 2.0 * c0 * c1 * ctl->JAB + c1 * c1 * ctl->JBB;
  const double l = c0 * ctl->aa + c1 * ctl->ab;
  const double hn2 = ctl->step_h_norm * ctl->step_h_norm;   // |p_h|^2 = |r_h|^2
  const double pn2 = ctl->step_norm * ctl->step_norm;       // |p|^2 = |r|^2
  const double DP2 = rb[0], DPR = rb[1], GR = rb[2], H2 = rb[3], Hu2 = rb[4], rbound = rb[5];
  const double Jr2 = rj[0], JpJr = rj[1];
  // reflected direction: intersect_trust_region(ps p_h, r_h, Delta) (common.py:136-168)
  const double ia = hn2, ib = ps * (hn2 - 2.0 * H2), ic = ps * ps * hn2 - Delta * Delta;
  const double idd = sqrt(fmax(ib * ib - ia * ic, 0.0));
  const double iq = -(ib + copysign(idd, ib));
  const double to_tr = fmax(iq / ia, ic / iq);
  double r_stride = fmin(rbound, to_tr), rl, ru;
  if (r_stride > 0.0) {
    rl = (1.0 - theta) * ps / r_stride;
    ru = (r_stride == rbound) ? theta * rbound : to_tr;
  } else {
    rl = 0.0; ru = -1.0;
  }
  double r_value = INFINITY;
  if (rl <= ru) {
    const double a = 0.5 * (Jr2 + DP2);
    const double b = GR + ps * JpJr + ps * DPR;
    const double c = 0.5 * ps * ps * q + ps * l;
    bnd_min_quad(a, b, rl, ru, c, r_stride, r_value);
  }
  // the subspace step pulled back from the bound
  const double tp = theta * ps;
  const double p_value = 0.5 * q * tp * tp + l * tp;
  // anti-gradient
  const double gh = sqrt(ctl->gh2);
  const double ag_tr = Delta / gh, agb = bnd->ag_bound;
  const double ag_up = agb < ag_tr ? theta * agb : ag_tr;
  double ag_stride, ag_value;
  bnd_min_quad(0.5 * ctl->Jg2, -ctl->gh2, 0.0, ag_up, 0.0, ag_stride, ag_value);
  if (p_value < r_value && p_value < ag_value) {
    bnd->mode = 0; bnd->c_p = tp;
    ctl->predicted = -p_value;
    ctl->step_h_norm = tp * ctl->step_h_norm;
    ctl->step_norm = tp * ctl->step_norm;
  } else if (r_value < p_value && r_value < ag_value) {
    bnd->mode = 1; bnd->c_r = r_stride;
    ctl->predicted = -r_value;
    const double rs = r_stride;
    ctl->step_h_norm = sqrt(fmax(0.0, (rs * rs + ps * ps) * hn2 + 2.0 * rs * ps * (hn2 - 2.0 * H2)));
    ctl->step_norm = sqrt(fmax(0.0, (rs * rs + ps * ps) * pn2 + 2.0 * rs * ps * (pn2 - 2.0 * Hu2)));
  } else {
    bnd->mode = 2; bnd->c_ag = ag_stride;
    ctl->predicted = -ag_value;
    ctl->step_h_norm = ag_stride * gh;
    ctl->step_norm = ag_stride * sqrt(ctl->gtgt);
  }
}

// Trial point of the chosen step, moved strictly inside the box by make_strictly_feasible(rstep=0)
// (common.py:387-411).  A zero step keeps x bit for bit (held entries).
__global__ void __launch_bounds__(256)
k_bnd_trial(const double* __restrict__ cams, const double* __restrict__ pts, const double* __restrict__ gt_c,
            const double* __restrict__ gt_p, const double* __restrict__ bp, const double* __restrict__ lb,
            const double* __restrict__ ub, int nc, long long n, const Bnd* __restrict__ bnd,
            double* __restrict__ cams_t, double* __restrict__ pts_t) {
  const int mode = bnd->mode;
  const double cp = bnd->c_p, cr = bnd->c_r, cag = bnd->c_ag, ps = bnd->p_stride;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const bool cm = i < nc;
    const double x = cm ? cams[i] : pts[i - nc];
    const double l = lb[i], u = ub[i];
    double st;
    if (mode == 0) {
      st = cp * bp[i];
    } else if (mode == 1) {
      const double p = bp[i];
      const double r = bnd_hit(x, p, l, u, ps) ? -p : p;
      st = fma(cr, r, ps * p);
    } else {
      st = -cag * (cm ? gt_c[i] : gt_p[i - nc]);
    }
    double xn = x;
    if (st != 0.0) {
      xn = x + st;
      if (xn <= l) xn = nextafter(l, u);
      else if (xn >= u) xn = nextafter(u, l);
      if (xn < l || xn > u) xn = 0.5 * (l + u);
    }
    if (cm) cams_t[i] = xn; else pts_t[i - nc] = xn;
  }
}

}  // namespace lcba
