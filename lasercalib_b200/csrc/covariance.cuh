// Per-point blocks of the parameter covariance (lcba_covariance): Sigma_pp = L_p^-T (I + Z_p^T Z_p) L_p^-1 with
// Z_p = X Y_p, X = L_S^-1 (k_chol_inverse, held rows / columns 0), Y_p = W_p L_p^-T the (11 C x 3) operand of the
// Schur routes and L_p^-1 from k_point_factor (Lz).  Z = X [Y_1 .. Y_P] is a lower-triangular n x n matrix times
// an n x 3P matrix: n (n + 1) / 2 * 3 P FMA, on the FP64 tensor pipe (DMMA m8n8k4, as k_schur_mma).
//
// One CTA takes a batch of B points (3 B columns of Y) at a time:
//   * all warps evaluate Y of the batch in place (camera tables, points, pair weights, Lz: the arithmetic of
//     mma_produce) into shared memory, column-major [3 B][ld] with ld = 4 (mod 16) doubles, so that the B-fragment
//     loads (lane -> k lane % 4, column lane / 4) are conflict free;
//   * 16-row blocks of Z (two 8-row tiles, K = 16 (b + 1): X is lower triangular and zero above the diagonal) are
//     dealt to the warps in snake order, which balances the triangle; X comes from L2 (<= 4 MB) with a prefetch
//     of four K-steps;
//   * after each block the warp folds its 16 x 3 B slice of Z into per-lane partial Grams (6 entries per point)
//     through a warp-private shared-memory tile; the warps' partials are summed in warp order.  Every sum runs in
//     a fixed order, so the output is bit-identical from run to run.
#pragma once
#include "common.cuh"
#include "eval.cuh"
#include "model.cuh"

namespace lcba {

constexpr int COV_THREADS = 256;
constexpr int COV_WARPS = COV_THREADS / 32;

// rows / columns of X and Y rounded up to the 16-row blocks of k_point_cov
__host__ __device__ inline int cov_npad(int n) { return (n + 15) / 16 * 16; }
__host__ __device__ inline int cov_ld(int n) { return cov_npad(n) + 4; }

// dynamic shared memory of k_point_cov<B> (doubles): tables | Y [3B][ld] | per-warp Z tiles [16][3B+1] | Grams
__host__ __device__ inline size_t cov_smem_doubles(int C, int B) {
  return (size_t)((C * CAMTAB + 1) & ~1) + (size_t)3 * B * cov_ld(NCP * C) + (size_t)COV_WARPS * 16 * (3 * B + 1) +
         (size_t)COV_WARPS * 6 * B;
}

// Y of one (point, camera) item, 11 rows x 3 columns: the arithmetic of mma_produce (schur_mma.cuh)
__device__ __forceinline__ void cov_produce(const double* __restrict__ T, const double (&X)[3], const double (&li)[9],
                                           double w, bool live, double* __restrict__ col0, int ld) {
  ObsLin L;
  obs_linearize<false>(T, X[0], X[1], X[2], 0.0, 0.0, w, L, live);
  double Q[2][3];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    Q[i][0] = L.Jp[i][0] * li[0];
    Q[i][1] = fma(L.Jp[i][0], li[1], L.Jp[i][1] * li[2]);
    Q[i][2] = fma(L.Jp[i][0], li[3], fma(L.Jp[i][1], li[4], L.Jp[i][2] * li[5]));
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    double* o = col0 + (size_t)k * ld;
#pragma unroll
    for (int a = 0; a < 9; ++a) o[a] = fma(L.Jc[0][a], Q[0][k], L.Jc[1][a] * Q[1][k]);
    o[9] = w * Q[0][k];
    o[10] = w * Q[1][k];
  }
}

__device__ __forceinline__ void cov_dmma(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// X: n_pad x n_pad row-major (k_chol_inverse), zero above the diagonal, in held rows / columns and past n.
// out: P x 6 (00 01 02 11 12 22).  B: points per batch (16, or 8 where 16 do not fit in shared memory).
template <int B>
__global__ void __launch_bounds__(COV_THREADS, 1)
k_point_cov(const double* __restrict__ X, const double* __restrict__ tab, const double* __restrict__ pts,
            const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
            const unsigned long long* __restrict__ mask, const double* __restrict__ Lz, long long P, int C,
            double* __restrict__ out) {
  constexpr int NCOL = 3 * B, CT = NCOL / 8, NIT = (6 * B + 31) / 32;
  extern __shared__ __align__(16) double s_dyn[];
  const int n = NCP * C, npad = cov_npad(n), ld = cov_ld(n), nb = npad / 16;
  double* s_tab = s_dyn;
  double* s_Y = s_tab + ((C * CAMTAB + 1) & ~1);
  double* s_Z = s_Y + (size_t)NCOL * ld;
  double* s_G = s_Z + (size_t)COV_WARPS * 16 * (NCOL + 1);
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  double* my_Z = s_Z + (size_t)wid * 16 * (NCOL + 1);
  load_tables_smem(tab, s_tab, C);
  for (int i = t; i < NCOL * (npad - n); i += COV_THREADS) s_Y[(size_t)(i / (npad - n)) * ld + n + i % (npad - n)] = 0.0;
  const int nbatch = (int)((P + B - 1) / B);
  for (int bt = blockIdx.x; bt < nbatch; bt += gridDim.x) {
    const long long p0 = (long long)bt * B;
    __syncthreads();               // tables loaded / the previous batch's Y and Grams consumed
    for (int it = t; it < B * C; it += COV_THREADS) {
      const int pl = it / C, cam = it % C;
      const long long p = p0 + pl;
      double Xp[3] = {0.0, 0.0, 0.0}, li[9];
      bool live = false;
      double w = 0.0;
      if (p < P) {
        const unsigned long long m = mask[p];
        live = (m >> cam) & 1ull;
        if (live) w = wgt ? wgt[(long long)obs_start[p] + __popcll(m & ((1ull << cam) - 1ull))] : 1.0;
#pragma unroll
        for (int a = 0; a < 3; ++a) Xp[a] = pts[3 * p + a];
#pragma unroll
        for (int a = 0; a < 9; ++a) li[a] = Lz[p * 9 + a];
      } else {
#pragma unroll
        for (int a = 0; a < 9; ++a) li[a] = 0.0;
      }
      cov_produce(s_tab + cam * CAMTAB, Xp, li, w, live, s_Y + (size_t)(3 * pl) * ld + NCP * cam, ld);
    }
    __syncthreads();
    double g[NIT];
#pragma unroll
    for (int j = 0; j < NIT; ++j) g[j] = 0.0;
    const double* yb = s_Y + (size_t)(lane >> 2) * ld + (lane & 3);
    for (int r = 0;; ++r) {
      const int b = r * COV_WARPS + ((r & 1) ? COV_WARPS - 1 - wid : wid);
      if (b >= nb) break;
      const double* xa = X + (size_t)(16 * b + (lane >> 2)) * npad + (lane & 3);
      double acc[2][CT][2];
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int u = 0; u < CT; ++u) acc[i][u][0] = acc[i][u][1] = 0.0;
      double an[2][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { an[0][j] = __ldg(xa + 4 * j); an[1][j] = __ldg(xa + (size_t)8 * npad + 4 * j); }
      for (int gk = 0; gk <= b; ++gk) {          // K-steps of 4 in groups of 4: K = 16 (b + 1)
        double ac[2][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { ac[0][j] = an[0][j]; ac[1][j] = an[1][j]; }
        if (gk < b) {
          const double* xn = xa + 16 * (gk + 1);
#pragma unroll
          for (int j = 0; j < 4; ++j) { an[0][j] = __ldg(xn + 4 * j); an[1][j] = __ldg(xn + (size_t)8 * npad + 4 * j); }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k0 = 16 * gk + 4 * j;
          double bf[CT];
#pragma unroll
          for (int u = 0; u < CT; ++u) bf[u] = yb[(size_t)8 * u * ld + k0];
#pragma unroll
          for (int u = 0; u < CT; ++u) {
            cov_dmma(acc[0][u], ac[0][j], bf[u]);
            cov_dmma(acc[1][u], ac[1][j], bf[u]);
          }
        }
      }
      // Z rows 16 b .. 16 b + 15 -> partial Grams: item q * 6 + e of point q, entries (00 01 02 11 12 22)
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int u = 0; u < CT; ++u)
#pragma unroll
          for (int e = 0; e < 2; ++e) my_Z[(8 * i + (lane >> 2)) * (NCOL + 1) + 8 * u + 2 * (lane & 3) + e] = acc[i][u][e];
      __syncwarp();
#pragma unroll
      for (int j = 0; j < NIT; ++j) {
        const int item = lane + 32 * j;
        if (item < 6 * B) {
          const int q = item / 6, e = item % 6;
          const int ea = e < 3 ? 0 : (e < 5 ? 1 : 2), eb = e < 3 ? e : (e < 5 ? e - 2 : 2);
          const double* za = my_Z + 3 * q + ea;
          const double* zb = my_Z + 3 * q + eb;
          double s = g[j];
#pragma unroll
          for (int row = 0; row < 16; ++row) s = fma(za[row * (NCOL + 1)], zb[row * (NCOL + 1)], s);
          g[j] = s;
        }
      }
      __syncwarp();
    }
#pragma unroll
    for (int j = 0; j < NIT; ++j)
      if (lane + 32 * j < 6 * B) s_G[wid * 6 * B + lane + 32 * j] = g[j];
    __syncthreads();
    if (t < B && p0 + t < P) {
      const long long p = p0 + t;
      double G[6];
#pragma unroll
      for (int e = 0; e < 6; ++e) {
        double s = 0.0;
        for (int w = 0; w < COV_WARPS; ++w) s += s_G[w * 6 * B + 6 * t + e];
        G[e] = s;
      }
      // M = I + G; Sigma = Li^T M Li with Li = L^-1 lower (Lz: 00 10 11 20 21 22)
      const double* l = Lz + p * 9;
      const double Li[3][3] = {{l[0], 0.0, 0.0}, {l[1], l[2], 0.0}, {l[3], l[4], l[5]}};
      const double M[3][3] = {{1.0 + G[0], G[1], G[2]}, {G[1], 1.0 + G[3], G[4]}, {G[2], G[4], 1.0 + G[5]}};
      double T3[3][3];
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) T3[a][c] = fma(M[a][0], Li[0][c], fma(M[a][1], Li[1][c], M[a][2] * Li[2][c]));
      double S[3][3];
#pragma unroll
      for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int c = 0; c < 3; ++c) S[a][c] = fma(Li[0][a], T3[0][c], fma(Li[1][a], T3[1][c], Li[2][a] * T3[2][c]));
      double* o = out + p * 6;
      o[0] = S[0][0]; o[1] = S[0][1]; o[2] = S[0][2]; o[3] = S[1][1]; o[4] = S[1][2]; o[5] = S[2][2];
    }
  }
}

// unheld points seen by fewer than two distinct cameras: part[block] = count (as a double)
__global__ void __launch_bounds__(256)
k_cov_views(const unsigned long long* __restrict__ mask, const uint8_t* __restrict__ pt_fixed, long long P,
            double* __restrict__ part) {
  __shared__ double s_red[32];
  double cnt = 0.0;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += (long long)gridDim.x * blockDim.x)
    if (!(pt_fixed && pt_fixed[p]) && __popcll(mask[p]) < 2) cnt += 1.0;
  const double s = block_sum(cnt, s_red);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}

}  // namespace lcba
