// Streaming passes of one trust-region iteration (everything except the Schur kernel):
//   k_linearize    : r, J blocks at x -> per-point V (3x3 sym) and g_p, per-camera g_c and
//                    diag(J^T J) (= squared column norms for scipy's x_scale='jac'), cost
//   k_point_prep   : Jacobi scaling with running max (common.py:598-610), g~ = scale^2 g
//   k_jdot         : |J g~|^2 for the Cauchy-model regulariser (trf.py:488-492)
//   k_point_factor : (V + lam Dp^2) = L L^T, stores L^-1 and z = L^-1 g_p
//   k_backsub      : p_p = (V + lam Dp^2)^-1 (g_p - W^T p_c) and the Gram sums of
//                    J[g~, p] for the 2-D subspace problem (trf.py:496-500)
// Work decomposition: "bins" of whole points, <= 256 observations per CTA, one thread per
// observation; per-point reductions go through shared memory (deterministic, no atomics).
#pragma once
#include "common.cuh"
#include "control.cuh"

namespace lcba {

constexpr int LIN_THREADS = 256;
constexpr int LIN_WARPS = LIN_THREADS / 32;
constexpr int CAMSUM = 22;          // per camera: g_c (11) then diag(J^T J) (11)
constexpr int CTAB_LD = 23;         // odd row stride of the warp-private camera tables

// Bin b owns the points whose first observation index lies in [b*B, (b+1)*B); the first
// point and first observation of every bin are precomputed at ingest (k_bin_table): every
// thread reads its bin's range with two uniform 8-byte loads, and the NEXT bin's range is
// prefetched while the current one is processed (no thread-0 lookup + barrier).
struct BinEntry { int32_t p0; uint32_t o0; };

__global__ void k_bin_table(const uint32_t* __restrict__ obs_start, long long P, long long nbins,
                            int B, BinEntry* __restrict__ bins) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b > nbins) return;
  const long long p0 = (b == nbins) ? P : lower_bound_u32(obs_start, P, (unsigned long long)b * B);
  bins[b].p0 = (int32_t)p0;
  bins[b].o0 = obs_start[p0];
}

struct BinRange { long long p0, p1; long long o0; int nobs; };

__device__ __forceinline__ BinRange load_bin(const BinEntry* __restrict__ bins, long long bin,
                                             long long nbins) {
  BinRange r;
  if (bin < nbins) {
    const int2 e0 = *reinterpret_cast<const int2*>(bins + bin);
    const int2 e1 = *reinterpret_cast<const int2*>(bins + bin + 1);
    r.p0 = e0.x;
    r.o0 = (unsigned)e0.y;
    r.p1 = e1.x;
    r.nobs = (int)((unsigned)e1.y - (unsigned)e0.y);
  } else {
    r.p0 = r.p1 = r.o0 = 0;
    r.nobs = 0;
  }
  return r;
}

// dynamic smem layout (doubles): tab[C*CAMTAB | even] pv[256*9] ctab[8*C*23]
__host__ __device__ inline size_t linearize_smem_doubles(int C) {
  return (size_t)((C * CAMTAB + 1) & ~1) + LIN_THREADS * 9 + (size_t)LIN_WARPS * C * CTAB_LD;
}

// Vg[p][0..5] = V (00,01,02,11,12,22), Vg[p][6..8] = g_p.
// cam_part[block][C*22], cost_part[block]
__global__ void __launch_bounds__(LIN_THREADS, 3)
k_linearize(const double* __restrict__ tab, const double* __restrict__ pts,
            const double2* __restrict__ uv, const uint8_t* __restrict__ cam,
            const int32_t* __restrict__ pt, const double* __restrict__ wgt,
            const uint32_t* __restrict__ obs_start, const BinEntry* __restrict__ bins,
            long long nbins, int C, double* __restrict__ Vg, double* __restrict__ cam_part,
            double* __restrict__ cost_part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  double* s_pv = s_dyn + ((C * CAMTAB + 1) & ~1);
  double* s_ctab = s_pv + LIN_THREADS * 9;
  __shared__ double s_red[32];

  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  load_tables_smem(tab, s_tab, C);
  for (int i = t; i < LIN_WARPS * C * CTAB_LD; i += LIN_THREADS) s_ctab[i] = 0.0;
  double cost = 0.0;
  double* my_ctab = s_ctab + (size_t)wid * C * CTAB_LD;
  BinRange nxt = load_bin(bins, blockIdx.x, nbins);
  __syncthreads();

  for (long long bin = blockIdx.x; bin < nbins; bin += gridDim.x) {
    const BinRange cur = nxt;
    nxt = load_bin(bins, bin + gridDim.x, nbins);      // prefetch
    const long long p0 = cur.p0, o0 = cur.o0;
    const long long npts = cur.p1 - p0;
    const int nobs = cur.nobs;
    uint8_t c8 = 255;
    double cv[CAMSUM];
    if (t < nobs) {
      const long long o = o0 + t;
      c8 = cam[o];
      const long long p = pt[o];
      const double2 ob = uv[o];
      const double w = wgt ? wgt[o] : 1.0;
      ObsLin L;
      obs_linearize<true>(s_tab + c8 * CAMTAB, pts[3 * p], pts[3 * p + 1], pts[3 * p + 2], ob.x,
                          ob.y, w, L);
      cost = fma(L.ru, L.ru, fma(L.rv, L.rv, cost));
      double* pv = s_pv + t * 9;
      pv[0] = fma(L.Jp[0][0], L.Jp[0][0], L.Jp[1][0] * L.Jp[1][0]);
      pv[1] = fma(L.Jp[0][0], L.Jp[0][1], L.Jp[1][0] * L.Jp[1][1]);
      pv[2] = fma(L.Jp[0][0], L.Jp[0][2], L.Jp[1][0] * L.Jp[1][2]);
      pv[3] = fma(L.Jp[0][1], L.Jp[0][1], L.Jp[1][1] * L.Jp[1][1]);
      pv[4] = fma(L.Jp[0][1], L.Jp[0][2], L.Jp[1][1] * L.Jp[1][2]);
      pv[5] = fma(L.Jp[0][2], L.Jp[0][2], L.Jp[1][2] * L.Jp[1][2]);
      pv[6] = fma(L.Jp[0][0], L.ru, L.Jp[1][0] * L.rv);
      pv[7] = fma(L.Jp[0][1], L.ru, L.Jp[1][1] * L.rv);
      pv[8] = fma(L.Jp[0][2], L.ru, L.Jp[1][2] * L.rv);
#pragma unroll
      for (int a = 0; a < 9; ++a) {
        cv[a] = fma(L.Jc[0][a], L.ru, L.Jc[1][a] * L.rv);
        cv[11 + a] = fma(L.Jc[0][a], L.Jc[0][a], L.Jc[1][a] * L.Jc[1][a]);
      }
      cv[9] = w * L.ru;
      cv[10] = w * L.rv;
      cv[20] = w * w;
      cv[21] = w * w;
    }
    // per-camera sums into the warp-private table: lanes that share a camera take turns
    // (rank among their peers), all other lanes update their own row concurrently
    {
      const unsigned peers = __match_any_sync(0xffffffffu, (int)c8);
      const int rank = (c8 == 255) ? -1 : __popc(peers & ((1u << lane) - 1u));
      const int maxrank = __reduce_max_sync(0xffffffffu, rank);
      for (int r = 0; r <= maxrank; ++r) {
        if (rank == r) {
          double* row = my_ctab + c8 * CTAB_LD;
#pragma unroll
          for (int v = 0; v < CAMSUM; ++v) row[v] += cv[v];
        }
        __syncwarp();
      }
    }
    __syncthreads();
    // per-point sums (fixed order => deterministic)
    // two lanes per (point, value): even / odd observations, combined with one shuffle
    for (long long base = 0; base < npts * 18; base += LIN_THREADS) {
      const long long idx2 = base + t;
      const bool act = idx2 < npts * 18;
      const long long idx = (act ? idx2 : 0) >> 1;
      const int half = (int)(idx2 & 1);
      const long long q = idx / 9;
      const int e = (int)(idx - q * 9);
      double s = 0.0;
      if (act) {
        const int f0 = (int)(obs_start[p0 + q] - o0), f1 = (int)(obs_start[p0 + q + 1] - o0);
        for (int i = f0 + half; i < f1; i += 2) s += s_pv[i * 9 + e];
      }
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      if (act && half == 0) Vg[(p0 + q) * 9 + e] = s;
    }
    __syncthreads();
  }
  // flush
  __syncthreads();
  double* out = cam_part + (size_t)blockIdx.x * C * CAMSUM;
  for (int i = t; i < C * CAMSUM; i += LIN_THREADS) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < LIN_WARPS; ++w)
      s += s_ctab[(size_t)w * C * CTAB_LD + (i / CAMSUM) * CTAB_LD + (i % CAMSUM)];
    out[i] = s;
  }
  const double cs = block_sum(cost, s_red);
  if (t == 0) cost_part[blockIdx.x] = cs;
}

// out[j] = sum_b part[b*K + j], fixed order.  Block = 32 columns x 8 row lanes: lane r adds rows
// r, r + 8, ... (coalesced 256-byte reads per row), the 8 partial sums are combined in order.
constexpr int RC_COLS = 32, RC_ROWS = 8;
__global__ void __launch_bounds__(RC_COLS * RC_ROWS)
k_reduce_cols(const double* __restrict__ part, int nblocks, int K, double* __restrict__ out) {
  __shared__ double s[RC_ROWS][RC_COLS + 1];
  const int c = threadIdx.x % RC_COLS, r = threadIdx.x / RC_COLS;
  const int j = blockIdx.x * RC_COLS + c;
  double v = 0.0;
  if (j < K)
    for (int b = r; b < nblocks; b += RC_ROWS) v += part[(size_t)b * K + j];
  s[r][c] = v;
  __syncthreads();
  if (r == 0 && j < K) {
    double t = 0.0;
#pragma unroll
    for (int q = 0; q < RC_ROWS; ++q) t += s[q][c];
    out[j] = t;
  }
}

// few columns, many rows: one CTA per column
__global__ void k_reduce_scalars(const double* __restrict__ part, int nblocks, int K,
                                 double* __restrict__ out, int is_max_from) {
  __shared__ double s_red[32];
  const int j = blockIdx.x;
  const bool mx = j >= is_max_from;
  double s = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) {
    const double v = part[(size_t)b * K + j];
    s = mx ? fmax(s, v) : s + v;
  }
  s = mx ? block_max(s, s_red) : block_sum(s, s_red);
  if (threadIdx.x == 0) out[j] = s;
}

// ---- per-point scaling ---------------------------------------------------------------
// scl[p][a] = first ? (sqrt(Vaa) or 1 if 0) : max(sqrt(Vaa), scl) ; gt = g / scl^2.
// partial[block][0..3] sums: |g_h|^2, |x*scl|^2, |x|^2 ; [3] max |g|
// A held point (pt_fixed[p] != 0; pt_fixed may be NULL) is a constant of the problem: scl = 1,
// gt = 0, g_p in Vg set to 0 (so the back-substitution and lcba_get_grad see no gradient), and no
// share of the norms.
constexpr int PP_K = 4;
__global__ void __launch_bounds__(256)
k_point_prep(double* __restrict__ Vg, const double* __restrict__ pts,
             double* __restrict__ scl, double* __restrict__ gt, long long P, int first,
             const uint8_t* __restrict__ pt_fixed, double* __restrict__ part) {
  __shared__ double s_red[32];
  double gh2 = 0, xs2 = 0, x2 = 0, gmax = 0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += stride) {
    if (pt_fixed && pt_fixed[p]) {
#pragma unroll
      for (int a = 0; a < 3; ++a) { scl[3 * p + a] = 1.0; gt[3 * p + a] = 0.0; Vg[p * 9 + 6 + a] = 0.0; }
      continue;
    }
    const double* v = Vg + p * 9;
    const double d[3] = {v[0], v[3], v[5]};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      double s = sqrt(d[a]);
      if (first) { if (s == 0.0) s = 1.0; } else s = fmax(s, scl[3 * p + a]);
      scl[3 * p + a] = s;
      const double g = v[6 + a], x = pts[3 * p + a];
      const double ghh = g / s;
      gt[3 * p + a] = ghh / s;
      gh2 = fma(ghh, ghh, gh2);
      xs2 = fma(x * s, x * s, xs2);
      x2 = fma(x, x, x2);
      gmax = fmax(gmax, fabs(g));
    }
  }
  const double a0 = block_sum(gh2, s_red), a1 = block_sum(xs2, s_red), a2 = block_sum(x2, s_red);
  const double a3 = block_max(gmax, s_red);
  if (threadIdx.x == 0) {
    double* o = part + (size_t)blockIdx.x * PP_K;
    o[0] = a0; o[1] = a1; o[2] = a2; o[3] = a3;
  }
}

// ---- |J g~|^2 ------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_jdot(const double* __restrict__ tab, const double* __restrict__ pts,
       const uint8_t* __restrict__ cam, const int32_t* __restrict__ pt,
       const double* __restrict__ wgt, const double* __restrict__ gt_c,
       const double* __restrict__ gt_p, long long N, int C, double* __restrict__ part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  double* s_gc = s_dyn + C * CAMTAB;
  __shared__ double s_red[32];
  load_tables_smem(tab, s_tab, C);
  for (int i = threadIdx.x; i < C * NCP; i += blockDim.x) s_gc[i] = gt_c[i];
  __syncthreads();
  double acc = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
    const int c = cam[i];
    const long long p = pt[i];
    const double w = wgt ? wgt[i] : 1.0;
    ObsLin L;
    obs_linearize<false>(s_tab + c * CAMTAB, pts[3 * p], pts[3 * p + 1], pts[3 * p + 2], 0.0, 0.0,
                         w, L);
    const double* gc = s_gc + c * NCP;
    double a0 = w * gc[9], a1 = w * gc[10];
#pragma unroll
    for (int a = 0; a < 9; ++a) { a0 = fma(L.Jc[0][a], gc[a], a0); a1 = fma(L.Jc[1][a], gc[a], a1); }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double g = gt_p[3 * p + a];
      a0 = fma(L.Jp[0][a], g, a0);
      a1 = fma(L.Jp[1][a], g, a1);
    }
    acc = fma(a0, a0, fma(a1, a1, acc));
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// ---- per-point factorisation -----------------------------------------------------------
// Lz[p][0..5] = L^-1 (00,10,11,20,21,22), Lz[p][6..8] = z = L^-1 g_p, with
// L L^T = V + lam * diag(scl^2).  Pivots are clamped so that points with < 2 views
// (rank-deficient V; never produced by the reference's pipeline, get_points3d.py:52-56)
// give finite numbers.  lam comes from the device control block (solver loop: no host round
// trip) when `ctl` is given, from the argument otherwise (lcba_linearize debug tap).
// A held point (pt_fixed[p] != 0; pt_fixed may be NULL) gets L^-1 = 0 and z = 0: its Y = W L^-T
// vanishes, so it subtracts nothing from S, and its step L^-T L^-1 (.) is exactly 0.
__global__ void __launch_bounds__(256)
k_point_factor(const double* __restrict__ Vg, const double* __restrict__ scl, double lam,
               const Ctl* __restrict__ ctl, long long P, const uint8_t* __restrict__ pt_fixed,
               double* __restrict__ Lz) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  if (pt_fixed && pt_fixed[p]) {
#pragma unroll
    for (int e = 0; e < 9; ++e) Lz[p * 9 + e] = 0.0;
    return;
  }
  if (ctl) lam = ctl->reg_term;
  const double* v = Vg + p * 9;
  const double s0 = scl[3 * p], s1 = scl[3 * p + 1], s2 = scl[3 * p + 2];
  const double v00 = fma(lam * s0, s0, v[0]), v11 = fma(lam * s1, s1, v[3]),
               v22 = fma(lam * s2, s2, v[5]);
  const double v01 = v[1], v02 = v[2], v12 = v[4];
  const double tiny = 1e-300;
  const double l00 = sqrt(fmax(v00, tiny));
  const double i00 = 1.0 / l00;
  const double l10 = v01 * i00, l20 = v02 * i00;
  const double d11 = v11 - l10 * l10;
  const double l11 = sqrt(fmax(d11, fmax(1e-14 * v11, tiny)));
  const double i11 = 1.0 / l11;
  const double l21 = (v12 - l20 * l10) * i11;
  const double d22 = v22 - l20 * l20 - l21 * l21;
  const double l22 = sqrt(fmax(d22, fmax(1e-14 * v22, tiny)));
  const double i22 = 1.0 / l22;
  const double i10 = -l10 * i00 * i11;
  const double i21 = -l21 * i11 * i22;
  const double i20 = -(l20 * i00 + l21 * i10) * i22;
  double* o = Lz + p * 9;
  o[0] = i00; o[1] = i10; o[2] = i11; o[3] = i20; o[4] = i21; o[5] = i22;
  const double g0 = v[6], g1 = v[7], g2 = v[8];
  o[6] = i00 * g0;
  o[7] = fma(i10, g0, i11 * g1);
  o[8] = fma(i20, g0, fma(i21, g1, i22 * g2));
}

// ---- back-substitution + Gram sums ------------------------------------------------------
// part[block][0..8]: (Jg~.Jg~, Jg~.Jp, Jp.Jp) , scaled-space (a.a, a.b, b.b) with a = g_h,
// b = gn_h (points part), unscaled (g~.g~, g~.p, p.p) (points part)
constexpr int BS_K = 9;
__global__ void __launch_bounds__(LIN_THREADS, 3)
k_backsub(const double* __restrict__ tab, const double* __restrict__ pts,
          const uint8_t* __restrict__ cam, const int32_t* __restrict__ pt,
          const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
          const BinEntry* __restrict__ bins, long long nbins, int C,
          const double* __restrict__ Vg,
          const double* __restrict__ Lz, const double* __restrict__ scl,
          const double* __restrict__ gt_c, const double* __restrict__ gt_p,
          const double* __restrict__ pc /* 11C GN step, cameras */, double* __restrict__ gn_p,
          double* __restrict__ part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  double* s_gc = s_tab + C * CAMTAB;      // g~_c
  double* s_pc = s_gc + C * NCP;          // p_c
  double* s_tv = s_pc + C * NCP;          // [256][3]
  double* s_pp = s_tv + LIN_THREADS * 3;  // [256][3], slot = first local observation of the point
  __shared__ double s_red[32];
  const int t = threadIdx.x;
  load_tables_smem(tab, s_tab, C);
  for (int i = t; i < C * NCP; i += LIN_THREADS) { s_gc[i] = gt_c[i]; s_pc[i] = pc[i]; }
  double acc[BS_K];
#pragma unroll
  for (int k = 0; k < BS_K; ++k) acc[k] = 0.0;

  BinRange nxt = load_bin(bins, blockIdx.x, nbins);
  __syncthreads();
  for (long long bin = blockIdx.x; bin < nbins; bin += gridDim.x) {
    const BinRange cur = nxt;
    nxt = load_bin(bins, bin + gridDim.x, nbins);      // prefetch
    const long long p0 = cur.p0, o0 = cur.o0;
    const long long npts = cur.p1 - p0;
    const int nobs = cur.nobs;
    double jp[2][3];
    double A0 = 0, A1 = 0, b0 = 0, b1 = 0;
    int q_of = 0;
    if (t < nobs) {
      const long long o = o0 + t;
      const int c = cam[o];
      const long long p = pt[o];
      q_of = (int)(obs_start[p] - o0);
      const double w = wgt ? wgt[o] : 1.0;
      ObsLin L;
      obs_linearize<false>(s_tab + c * CAMTAB, pts[3 * p], pts[3 * p + 1], pts[3 * p + 2], 0.0,
                           0.0, w, L);
      const double* gc = s_gc + c * NCP;
      const double* pcc = s_pc + c * NCP;
      A0 = w * gc[9]; A1 = w * gc[10];
      b0 = w * pcc[9]; b1 = w * pcc[10];
#pragma unroll
      for (int a = 0; a < 9; ++a) {
        A0 = fma(L.Jc[0][a], gc[a], A0);  A1 = fma(L.Jc[1][a], gc[a], A1);
        b0 = fma(L.Jc[0][a], pcc[a], b0); b1 = fma(L.Jc[1][a], pcc[a], b1);
      }
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const double g = gt_p[3 * p + a];
        A0 = fma(L.Jp[0][a], g, A0);
        A1 = fma(L.Jp[1][a], g, A1);
        jp[0][a] = L.Jp[0][a];
        jp[1][a] = L.Jp[1][a];
      }
#pragma unroll
      for (int a = 0; a < 3; ++a)
        s_tv[t * 3 + a] = fma(jp[0][a], b0, jp[1][a] * b1);   // J_p^T (J_c p_c)
    }
    __syncthreads();
    for (long long q = t; q < npts; q += LIN_THREADS) {
      const long long p = p0 + q;
      const int f0 = (int)(obs_start[p] - o0), f1 = (int)(obs_start[p + 1] - o0);
      double t0 = 0, t1 = 0, t2 = 0;
      for (int i = f0; i < f1; ++i) {
        t0 += s_tv[i * 3]; t1 += s_tv[i * 3 + 1]; t2 += s_tv[i * 3 + 2];
      }
      const double* v = Vg + p * 9;
      const double* li = Lz + p * 9;
      const double r0 = v[6] - t0, r1 = v[7] - t1, r2 = v[8] - t2;
      // y = L^-1 r ; p = L^-T y
      const double y0 = li[0] * r0;
      const double y1 = fma(li[1], r0, li[2] * r1);
      const double y2 = fma(li[3], r0, fma(li[4], r1, li[5] * r2));
      const double q0 = fma(li[0], y0, fma(li[1], y1, li[3] * y2));
      const double q1 = fma(li[2], y1, li[4] * y2);
      const double q2 = li[5] * y2;
      if (f1 > f0) { s_pp[f0 * 3] = q0; s_pp[f0 * 3 + 1] = q1; s_pp[f0 * 3 + 2] = q2; }
      gn_p[3 * p] = q0; gn_p[3 * p + 1] = q1; gn_p[3 * p + 2] = q2;
      const double pp[3] = {q0, q1, q2};
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        const double s = scl[3 * p + a], g = v[6 + a];
        const double ah = g / s, bh = pp[a] * s, gtl = ah / s;
        acc[3] = fma(ah, ah, acc[3]);
        acc[4] = fma(ah, bh, acc[4]);
        acc[5] = fma(bh, bh, acc[5]);
        acc[6] = fma(gtl, gtl, acc[6]);
        acc[7] = fma(gtl, pp[a], acc[7]);
        acc[8] = fma(pp[a], pp[a], acc[8]);
      }
    }
    __syncthreads();
    if (t < nobs) {
      const double* pp = s_pp + q_of * 3;
#pragma unroll
      for (int a = 0; a < 3; ++a) { b0 = fma(jp[0][a], pp[a], b0); b1 = fma(jp[1][a], pp[a], b1); }
      acc[0] = fma(A0, A0, fma(A1, A1, acc[0]));
      acc[1] = fma(A0, b0, fma(A1, b1, acc[1]));
      acc[2] = fma(b0, b0, fma(b1, b1, acc[2]));
    }
    __syncthreads();
  }
#pragma unroll
  for (int k = 0; k < BS_K; ++k) {
    const double s = block_sum(acc[k], s_red);
    if (t == 0) part[(size_t)blockIdx.x * BS_K + k] = s;
  }
}

// ---- trial point x + c0*g~ + c1*p ------------------------------------------------------
__global__ void k_make_trial(const double* __restrict__ x, const double* __restrict__ gt,
                             const double* __restrict__ gn, const double* __restrict__ coef,
                             long long n, double* __restrict__ xt) {
  const double c0 = coef[0], c1 = coef[1];
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    xt[i] = fma(c1, gn[i], fma(c0, gt[i], x[i]));
}

}  // namespace lcba
