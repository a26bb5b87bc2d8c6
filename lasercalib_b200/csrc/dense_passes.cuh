// Linearisation for DENSE rigs (most cameras see most points; no repeated (camera, point) rows):
// the same arithmetic as k_linearize, organised so that a thread keeps ONE camera for its whole
// life:
//     thread t of a 256-thread block  ->  camera c = t % C, point lane pl = t / C
//     tile = PB = 256 / C consecutive points; observation of (point p, camera c) =
//            obs_start[p] + popc(mask[p] & ((1 << c) - 1))        (point-major, camera-ascending)
// Consequences (what the round-1 ncu capture asked for, profiles/r01_ncu_full_summary.txt):
//   * per-camera sums (g_c, diag(J^T J), and the full camera blocks U_c) accumulate in
//     REGISTERS: no shared-memory read-modify-write per observation (k_linearize: 22 RMWs per
//     observation, shared-memory pipe 69 %, 50.9 M bank conflicts); k_cam_normal's separate model
//     evaluation disappears (U_c comes out of the same pass);
//   * the inputs of the NEXT tile are loaded before the current tile is evaluated (the round-1
//     kernels stalled 50 % on the index -> point -> table load chain);
//   * per-point sums go through one double-buffered shared-memory tile, one barrier per tile,
//     fixed summation order (bit-reproducible, no atomics).
// Invisible (point, camera) pairs idle their thread for that tile, so the sparse rigs keep the
// observation-major kernels of linearize.cuh.
#pragma once
#include "common.cuh"
#include "linearize.cuh"

namespace lcba {

constexpr int DP_THREADS = 256;
// per camera: 66 upper-triangle entries of U_c = sum Jc^T Jc (row-major a <= b), then g_c (11)
constexpr int DP_CAM_VALS = 66 + 11;

// Two-stage prefetch.  The observation index of a (point, camera) item depends on the point's
// mask and CSR offset, so a one-step prefetch still stalls on that dependent load (ncu round 2,
// first version: long-scoreboard stalls 3-11 per issued instruction with 2 warps per scheduler).
// Stage A loads (mask, obs_start) two tiles ahead, stage B turns them into the item's loads one
// tile ahead, stage C computes: no load is consumed in the iteration that issued it.
struct DenseIdx {
  unsigned long long m;
  uint32_t os;
  int ok;
};

struct DenseItem {          // one (point, camera) work item
  double X[3];
  double2 ob;
  double w;
  int live;
};

__device__ __forceinline__ DenseIdx dense_idx(long long p, long long P, bool worker,
                                              const uint32_t* __restrict__ obs_start,
                                              const unsigned long long* __restrict__ mask) {
  DenseIdx d;
  d.ok = worker && p < P;
  d.m = 0ull;
  d.os = 0u;
  if (d.ok) { d.m = mask[p]; d.os = obs_start[p]; }
  return d;
}

__device__ __forceinline__ DenseItem dense_item(const DenseIdx& d, long long p, int c,
                                                const double* __restrict__ pts,
                                                const double2* __restrict__ uv,
                                                const double* __restrict__ wgt) {
  DenseItem it;
  it.w = 0.0;
  it.ob = make_double2(0.0, 0.0);
  it.X[0] = it.X[1] = it.X[2] = 0.0;
  it.live = d.ok && ((d.m >> c) & 1ull);
  if (it.live) {
    const long long o = (long long)d.os + __popcll(d.m & ((1ull << c) - 1ull));
    if (uv) it.ob = uv[o];
    it.w = wgt ? wgt[o] : 1.0;
    it.X[0] = pts[3 * p];
    it.X[1] = pts[3 * p + 1];
    it.X[2] = pts[3 * p + 2];
  }
  return it;
}

// U (66 upper-triangle entries, row-major a <= b) += Jc^T Jc with the structural zeros of the
// cx / cy columns (Jc[0][10] = Jc[1][9] = 0, Jc[0][9] = Jc[1][10] = w) written out by hand.
__device__ __forceinline__ void accumulate_U(double (&acc)[66 + 11], const ObsLin& L, double w) {
  int idx = 0;
#pragma unroll
  for (int a = 0; a < 9; ++a) {
#pragma unroll
    for (int b = a; b < 9; ++b, ++idx)
      acc[idx] = fma(L.Jc[0][a], L.Jc[0][b], fma(L.Jc[1][a], L.Jc[1][b], acc[idx]));
    acc[idx] = fma(L.Jc[0][a], w, acc[idx]); ++idx;      // (a, cx)
    acc[idx] = fma(L.Jc[1][a], w, acc[idx]); ++idx;      // (a, cy)
  }
  acc[idx] = fma(w, w, acc[idx]); idx += 2;              // (cx, cx); (cx, cy) stays 0
  acc[idx] = fma(w, w, acc[idx]);                        // (cy, cy)
}

// ---- linearise: V, g_p per point; U_c, g_c per camera; cost --------------------------------
// Vg[p][0..5] = V (00,01,02,11,12,22), Vg[p][6..8] = g_p   (same layout as k_linearize)
// cam_part[block][C][DP_CAM_VALS], cost_part[block]
// dynamic smem (doubles): tab[C*CAMTAB | even] pv[2][DP_THREADS*9] red[DP_THREADS]
__host__ __device__ inline size_t dense_lin_smem_doubles(int C) {
  return (size_t)((C * CAMTAB + 1) & ~1) + 2 * DP_THREADS * 9 + DP_THREADS;
}

__global__ void __launch_bounds__(DP_THREADS, 1)
k_linearize_dense(const double* __restrict__ tab, const double* __restrict__ pts,
                  const double2* __restrict__ uv, const double* __restrict__ wgt,
                  const uint32_t* __restrict__ obs_start,
                  const unsigned long long* __restrict__ mask, long long P, int C, int PB,
                  double* __restrict__ Vg, double* __restrict__ cam_part,
                  double* __restrict__ cost_part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  double* s_pv = s_dyn + ((C * CAMTAB + 1) & ~1);
  double* s_red = s_pv + 2 * DP_THREADS * 9;
  __shared__ double s_blk[32];
  const int t = threadIdx.x;
  load_tables_smem(tab, s_tab, C);
  const int c = t % C, pl = t / C;
  const bool worker = pl < PB;
  // the thread's camera never changes: volatile keeps the table reads in shared memory (hoisting
  // 29 doubles into registers next to 77 accumulators spills)
  const volatile double* vT = s_tab + c * CAMTAB;
  double acc[DP_CAM_VALS];
#pragma unroll
  for (int i = 0; i < DP_CAM_VALS; ++i) acc[i] = 0.0;
  double cost = 0.0;
  const long long ntiles = (P + PB - 1) / PB;
  long long tile = blockIdx.x;
  const long long G = gridDim.x;
  DenseItem nxt = dense_item(dense_idx(tile * PB + pl, P, worker && tile < ntiles, obs_start, mask),
                             tile * PB + pl, c, pts, uv, wgt);
  DenseIdx idx2 = dense_idx((tile + G) * PB + pl, P, worker && tile + G < ntiles, obs_start, mask);
  __syncthreads();
  int buf = 0;
  for (; tile < ntiles; tile += G, buf ^= 1) {
    const DenseItem cur = nxt;
    nxt = dense_item(idx2, (tile + G) * PB + pl, c, pts, uv, wgt);
    idx2 = dense_idx((tile + 2 * G) * PB + pl, P, worker && tile + 2 * G < ntiles, obs_start, mask);
    double* pv = s_pv + (size_t)buf * DP_THREADS * 9 + t * 9;
    if (cur.live) {
      double T[CAMTAB];
#pragma unroll
      for (int i = 0; i < CAMTAB; ++i) T[i] = vT[i];
      ObsLin L;
      obs_linearize<true>(T, cur.X[0], cur.X[1], cur.X[2], cur.ob.x, cur.ob.y, cur.w, L);
      cost = fma(L.ru, L.ru, fma(L.rv, L.rv, cost));
      pv[0] = fma(L.Jp[0][0], L.Jp[0][0], L.Jp[1][0] * L.Jp[1][0]);
      pv[1] = fma(L.Jp[0][0], L.Jp[0][1], L.Jp[1][0] * L.Jp[1][1]);
      pv[2] = fma(L.Jp[0][0], L.Jp[0][2], L.Jp[1][0] * L.Jp[1][2]);
      pv[3] = fma(L.Jp[0][1], L.Jp[0][1], L.Jp[1][1] * L.Jp[1][1]);
      pv[4] = fma(L.Jp[0][1], L.Jp[0][2], L.Jp[1][1] * L.Jp[1][2]);
      pv[5] = fma(L.Jp[0][2], L.Jp[0][2], L.Jp[1][2] * L.Jp[1][2]);
      pv[6] = fma(L.Jp[0][0], L.ru, L.Jp[1][0] * L.rv);
      pv[7] = fma(L.Jp[0][1], L.ru, L.Jp[1][1] * L.rv);
      pv[8] = fma(L.Jp[0][2], L.ru, L.Jp[1][2] * L.rv);
      accumulate_U(acc, L, cur.w);
#pragma unroll
      for (int a = 0; a < 9; ++a) acc[66 + a] = fma(L.Jc[0][a], L.ru, fma(L.Jc[1][a], L.rv, acc[66 + a]));
      acc[66 + 9] = fma(cur.w, L.ru, acc[66 + 9]);
      acc[66 + 10] = fma(cur.w, L.rv, acc[66 + 10]);
    } else if (worker) {
#pragma unroll
      for (int e = 0; e < 9; ++e) pv[e] = 0.0;
    }
    __syncthreads();
    // per-point sums over the cameras, fixed order; the other threads go on with the next tile
    const long long p0 = tile * PB;
    const int npts = (int)min((long long)PB, P - p0);
    for (int j = t; j < npts * 9; j += DP_THREADS) {     // (more than one round only below 9 cameras)
      const int q = j / 9, e = j - 9 * q;
      const double* src = s_pv + (size_t)buf * DP_THREADS * 9 + (size_t)q * C * 9 + e;
      double s = 0.0;
      for (int k = 0; k < C; ++k) s += src[k * 9];
      Vg[(p0 + q) * 9 + e] = s;
    }
  }
  // block partial of the camera sums: over the PB point lanes of each camera, fixed order
  double* out = cam_part + (size_t)blockIdx.x * C * DP_CAM_VALS;
#pragma unroll
  for (int i = 0; i < DP_CAM_VALS; ++i) {
    __syncthreads();
    if (worker) s_red[pl * C + c] = acc[i];
    __syncthreads();
    if (t < C) {
      double s = 0.0;
      for (int q = 0; q < PB; ++q) s += s_red[q * C + t];
      out[t * DP_CAM_VALS + i] = s;
    }
  }
  const double cs = block_sum(cost, s_blk);
  if (t == 0) cost_part[blockIdx.x] = cs;
}

// camsum[c][0..10] = g_c, [11..21] = diag(J^T J) (the layout k_ctl_lin reads) and U[c][66] from
// the reduced block partials red[c][DP_CAM_VALS]
__global__ void k_dense_cam_unpack(const double* __restrict__ red, int C, double* __restrict__ camsum,
                                   double* __restrict__ U) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C * DP_CAM_VALS) return;
  const int c = i / DP_CAM_VALS, v = i % DP_CAM_VALS;
  const double x = red[i];
  if (v >= 66) { camsum[c * CAMSUM + (v - 66)] = x; return; }
  U[c * 66 + v] = x;
  // diagonal entries of the upper triangle: index of (a, a) = a * 11 - a (a - 1) / 2
  int a = 0, idx = 0;
  while (idx < v) { idx += NCP - a; ++a; }
  if (idx == v) camsum[c * CAMSUM + NCP + a] = x;
}

// ============================== point-parallel passes ==========================================
// Residual, |J g~|^2 and the back-substitution have NO per-camera output, so a thread can own a
// POINT and walk its cameras: all lanes of a warp read the same camera table at the same time
// (one shared-memory broadcast wavefront instead of 2-3 conflicting ones), per-point sums live in
// registers (no shared-memory reduction, no barrier), and the Gram sums of the 2-D subspace
// problem follow from per-point accumulators:
//     sum_k |b_k + Jp_k q|^2 = sum |b_k|^2 + 2 q . (sum Jp_k^T b_k) + q^T V q,  V = sum Jp_k^T Jp_k
// so one walk over the cameras is enough although q = p_p is only known after it.  Any visibility
// pattern works (a lane idles while its point does not see camera k); repeated (camera, point)
// rows keep the observation-major kernels.
constexpr int PT_THREADS = 256;

__global__ void __launch_bounds__(PT_THREADS, 2)
k_residual_pt(const double* __restrict__ tab, const double* __restrict__ pts,
              const double2* __restrict__ uv, const double* __restrict__ wgt,
              const uint32_t* __restrict__ obs_start, const unsigned long long* __restrict__ mask,
              long long P, int C, double* __restrict__ part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  __shared__ double s_red[32];
  load_tables_smem(tab, s_tab, C);
  __syncthreads();
  double acc = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += stride) {
    const unsigned long long m = mask[p];
    long long o = obs_start[p];
    const double X = pts[3 * p], Y = pts[3 * p + 1], Z = pts[3 * p + 2];
    for (int k = 0; k < C; ++k) {
      if (!((m >> k) & 1ull)) continue;
      const double2 ob = uv[o];
      const double w = wgt ? wgt[o] : 1.0;
      ++o;
      double pu, pv;
      project_tab(s_tab + k * CAMTAB, X, Y, Z, pu, pv);
      const double ru = w * (pu - ob.x), rv = w * (pv - ob.y);
      acc = fma(ru, ru, fma(rv, rv, acc));
    }
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// dynamic smem: tab[C*CAMTAB] gc[C*NCP]
__global__ void __launch_bounds__(PT_THREADS, 2)
k_jdot_pt(const double* __restrict__ tab, const double* __restrict__ pts,
          const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
          const unsigned long long* __restrict__ mask, const double* __restrict__ gt_c,
          const double* __restrict__ gt_p, long long P, int C, double* __restrict__ part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  double* s_gc = s_dyn + C * CAMTAB;
  __shared__ double s_red[32];
  load_tables_smem(tab, s_tab, C);
  for (int i = threadIdx.x; i < C * NCP; i += blockDim.x) s_gc[i] = gt_c[i];
  __syncthreads();
  double acc = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += stride) {
    const unsigned long long m = mask[p];
    long long o = obs_start[p];
    const double X = pts[3 * p], Y = pts[3 * p + 1], Z = pts[3 * p + 2];
    const double g0 = gt_p[3 * p], g1 = gt_p[3 * p + 1], g2 = gt_p[3 * p + 2];
    for (int k = 0; k < C; ++k) {
      if (!((m >> k) & 1ull)) continue;
      const double w = wgt ? wgt[o] : 1.0;
      ++o;
      ObsLin L;
      obs_linearize<false>(s_tab + k * CAMTAB, X, Y, Z, 0.0, 0.0, w, L);
      const double* gc = s_gc + k * NCP;
      double a0 = w * gc[9], a1 = w * gc[10];
#pragma unroll
      for (int a = 0; a < 9; ++a) { a0 = fma(L.Jc[0][a], gc[a], a0); a1 = fma(L.Jc[1][a], gc[a], a1); }
      a0 = fma(L.Jp[0][0], g0, fma(L.Jp[0][1], g1, fma(L.Jp[0][2], g2, a0)));
      a1 = fma(L.Jp[1][0], g0, fma(L.Jp[1][1], g1, fma(L.Jp[1][2], g2, a1)));
      acc = fma(a0, a0, fma(a1, a1, acc));
    }
  }
  const double s = block_sum(acc, s_red);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// dynamic smem: tab[C*CAMTAB] gc[C*NCP] pc[C*NCP]
__global__ void __launch_bounds__(PT_THREADS, 2)
k_backsub_pt(const double* __restrict__ tab, const double* __restrict__ pts,
             const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
             const unsigned long long* __restrict__ mask, long long P, int C,
             const double* __restrict__ Vg, const double* __restrict__ Lz,
             const double* __restrict__ scl, const double* __restrict__ gt_c,
             const double* __restrict__ gt_p, const double* __restrict__ pc,
             double* __restrict__ gn_p, double* __restrict__ part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;
  double* s_gc = s_dyn + C * CAMTAB;
  double* s_pc = s_gc + C * NCP;
  __shared__ double s_red[32];
  load_tables_smem(tab, s_tab, C);
  for (int i = threadIdx.x; i < C * NCP; i += blockDim.x) { s_gc[i] = gt_c[i]; s_pc[i] = pc[i]; }
  __syncthreads();
  double acc[BS_K];
#pragma unroll
  for (int k = 0; k < BS_K; ++k) acc[k] = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += stride) {
    const unsigned long long m = mask[p];
    long long o = obs_start[p];
    const double X = pts[3 * p], Y = pts[3 * p + 1], Z = pts[3 * p + 2];
    const double g0 = gt_p[3 * p], g1 = gt_p[3 * p + 1], g2 = gt_p[3 * p + 2];
    double tv0 = 0, tv1 = 0, tv2 = 0, u0 = 0, u1 = 0, u2 = 0, sAA = 0, sAb = 0, sbb = 0;
    for (int k = 0; k < C; ++k) {
      if (!((m >> k) & 1ull)) continue;
      const double w = wgt ? wgt[o] : 1.0;
      ++o;
      ObsLin L;
      obs_linearize<false>(s_tab + k * CAMTAB, X, Y, Z, 0.0, 0.0, w, L);
      const double* gc = s_gc + k * NCP;
      const double* pk = s_pc + k * NCP;
      double A0 = w * gc[9], A1 = w * gc[10], b0 = w * pk[9], b1 = w * pk[10];
#pragma unroll
      for (int a = 0; a < 9; ++a) {
        A0 = fma(L.Jc[0][a], gc[a], A0); A1 = fma(L.Jc[1][a], gc[a], A1);
        b0 = fma(L.Jc[0][a], pk[a], b0); b1 = fma(L.Jc[1][a], pk[a], b1);
      }
      A0 = fma(L.Jp[0][0], g0, fma(L.Jp[0][1], g1, fma(L.Jp[0][2], g2, A0)));
      A1 = fma(L.Jp[1][0], g0, fma(L.Jp[1][1], g1, fma(L.Jp[1][2], g2, A1)));
      tv0 = fma(L.Jp[0][0], b0, fma(L.Jp[1][0], b1, tv0));
      tv1 = fma(L.Jp[0][1], b0, fma(L.Jp[1][1], b1, tv1));
      tv2 = fma(L.Jp[0][2], b0, fma(L.Jp[1][2], b1, tv2));
      u0 = fma(L.Jp[0][0], A0, fma(L.Jp[1][0], A1, u0));
      u1 = fma(L.Jp[0][1], A0, fma(L.Jp[1][1], A1, u1));
      u2 = fma(L.Jp[0][2], A0, fma(L.Jp[1][2], A1, u2));
      sAA = fma(A0, A0, fma(A1, A1, sAA));
      sAb = fma(A0, b0, fma(A1, b1, sAb));
      sbb = fma(b0, b0, fma(b1, b1, sbb));
    }
    const double* v = Vg + p * 9;
    const double* li = Lz + p * 9;
    const double gp0 = v[6], gp1 = v[7], gp2 = v[8];
    const double r0 = gp0 - tv0, r1 = gp1 - tv1, r2 = gp2 - tv2;
    // y = L^-1 r ; q = L^-T y
    const double y0 = li[0] * r0;
    const double y1 = fma(li[1], r0, li[2] * r1);
    const double y2 = fma(li[3], r0, fma(li[4], r1, li[5] * r2));
    const double q0 = fma(li[0], y0, fma(li[1], y1, li[3] * y2));
    const double q1 = fma(li[2], y1, li[4] * y2);
    const double q2 = li[5] * y2;
    gn_p[3 * p] = q0; gn_p[3 * p + 1] = q1; gn_p[3 * p + 2] = q2;
    // sums over this point's observations of (A.A, A.(b + Jp q), |b + Jp q|^2)
    const double Vq0 = fma(v[0], q0, fma(v[1], q1, v[2] * q2));
    const double Vq1 = fma(v[1], q0, fma(v[3], q1, v[4] * q2));
    const double Vq2 = fma(v[2], q0, fma(v[4], q1, v[5] * q2));
    acc[0] += sAA;
    acc[1] += sAb + fma(q0, u0, fma(q1, u1, q2 * u2));
    acc[2] += sbb + 2.0 * fma(q0, tv0, fma(q1, tv1, q2 * tv2)) + fma(q0, Vq0, fma(q1, Vq1, q2 * Vq2));
    const double pp[3] = {q0, q1, q2}, gp[3] = {gp0, gp1, gp2};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const double s = scl[3 * p + a];
      const double ah = gp[a] / s, bh = pp[a] * s, gtl = ah / s;
      acc[3] = fma(ah, ah, acc[3]);
      acc[4] = fma(ah, bh, acc[4]);
      acc[5] = fma(bh, bh, acc[5]);
      acc[6] = fma(gtl, gtl, acc[6]);
      acc[7] = fma(gtl, pp[a], acc[7]);
      acc[8] = fma(pp[a], pp[a], acc[8]);
    }
  }
#pragma unroll
  for (int k = 0; k < BS_K; ++k) {
    const double s = block_sum(acc[k], s_red);
    if (threadIdx.x == 0) part[(size_t)blockIdx.x * BS_K + k] = s;
  }
}

}  // namespace lcba
