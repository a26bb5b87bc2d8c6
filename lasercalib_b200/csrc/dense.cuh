// Dense FP64 Cholesky solve of the reduced camera system (n = 11 C <= 704) on the device:
// blocked right-looking factorisation (32-wide panels) + both triangular solves in ONE
// cooperative launch (k_chol_fused).
// Replaces the LSMR call of scipy's TRF (scipy/optimize/_lsq/trf.py:494-495) for the camera
// block; a non-positive pivot raises fail[0] (the caller adds damping and retries).
#pragma once
#include "common.cuh"

namespace lcba {

constexpr int CH_NB = 32;

// ---- whole solve in one cooperative launch -------------------------------------------
// The solve is latency bound (n <= 704: 9..22 panels).  The first version used two launches
// per panel plus a solve kernel, the diagonal block factored with three CTA barriers per
// column: 0.46 ms at n = 264.  k_chol_fused keeps the right-looking blocked algorithm but
// runs it in ONE cooperative launch (0.135 ms at n = 264, 0.41 ms at n = 704):
//   * A is stored with n + 1 rows, row n = right-hand side: the panel solve and the trailing
//     update treat it like any other row, so the forward substitution comes for free
//     (row n ends as z = L^-1 b);
//   * every CTA factors the 32 x 32 diagonal block redundantly in ONE warp: lane = row, the
//     row in registers, the current column broadcast through shared memory (one __syncwarp
//     per column), every lane tracking all 32 running diagonals so the pivot needs no
//     exchange; the pivot is inverted once (rsqrt) and the DIAGONAL OF THE FACTOR STORES
//     1 / l_jj, so that panel rows and both substitutions multiply instead of divide;
//   * panel rows and trailing tiles are spread over the grid; two grid barriers per panel;
//   * the factored diagonal block goes back to A (CTA 0, from shared memory) only after the
//     panel's first grid barrier, when no CTA can still be reading the original block; so the
//     factor and the solution depend on the input alone, bit-identical for every grid size;
//   * CTA 0 finishes with the blocked back substitution L^T x = z.
// The grid barrier is a monotonic counter in global memory (release add / acquire poll);
// the launch is cooperative so all CTAs are co-resident, and the poll is bounded: a stuck
// barrier raises fail |= 2 instead of hanging the device.
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned target, int* fail) {
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
    unsigned spins = 0;
    while (ld_acquire_u32(counter) < target) {
      if (++spins > (1u << 22)) { atomicOr(fail, 2); break; }
    }
  }
  __syncthreads();
}

// Column J of the in-register 32 x 32 Cholesky (lane = row); compile-time recursion keeps
// every register index static.  a = my row, dg = running diagonals of ALL rows (identical in
// every lane), col = double-buffered broadcast column in shared memory.
template <int J>
__device__ __forceinline__ void chol_cols(double (&a)[CH_NB], double (&dg)[CH_NB], int lane,
                                          double (*col)[CH_NB], bool& bad) {
  if constexpr (J < CH_NB) {
    double d = dg[J];
    if (!(d > 0.0)) { bad = true; d = 1.0; }
    const double r = rsqrt(d);
    dg[J] = r;                                  // 1 / l_JJ
    const double l = a[J] * r;                  // l_{lane,J} for lane > J
    a[J] = l;
    if constexpr (J + 1 < CH_NB) {
      col[J & 1][lane] = l;
      __syncwarp();
#pragma unroll
      for (int c = J + 1; c < CH_NB; ++c) {
        const double lc = col[J & 1][c];
        a[c] = fma(-l, lc, a[c]);
        dg[c] = fma(-lc, lc, dg[c]);
      }
    }
    chol_cols<J + 1>(a, dg, lane, col, bad);
  }
}

constexpr int CH_MAXN = 704;

// A: (n + 1) x n row-major, lower triangle + rhs row; out: n.  sync[0] = fail, sync[1] = counter
// (both zeroed by the caller before the launch).  On return the strict lower triangle of A
// holds L, its diagonal 1 / l_jj, row n holds z.  dbg (may be null): per-phase cycle counters.
__global__ void __launch_bounds__(256)
k_chol_fused(double* A, int n, double* __restrict__ out, int* sync, long long* dbg) {
  __shared__ __align__(16) double D[CH_NB][CH_NB];        // L_kk (strict lower part used)
  __shared__ __align__(16) double Pi[CH_NB][CH_NB];       // rows of the panel, broadcast reads
  __shared__ double Pj[CH_NB][CH_NB + 1];                 // rows of the panel, lane = row
  __shared__ double rinv[CH_NB];
  __shared__ double col[2][CH_NB];
  __shared__ double y[CH_MAXN + CH_NB];
  int* fail = sync;
  unsigned* counter = reinterpret_cast<unsigned*>(sync + 1);
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int G = gridDim.x, b = blockIdx.x;
  unsigned phase = 0;
  long long tm[6] = {0, 0, 0, 0, 0, 0}, tc = dbg ? clock64() : 0;
#define CH_TICK(i) do { if (dbg) { const long long now_ = clock64(); tm[i] += now_ - tc; tc = now_; } } while (0)
  // CTA 0 stores the factored diagonal block of panel k (strict lower L_kk, 1 / l_jj on the
  // diagonal) from shared memory.  Every CTA reads the ORIGINAL block in its own step 1, so the
  // store waits for the first grid barrier of the panel (the closing barrier for the last one);
  // nobody reads the global block in between.
  auto store_diag = [&](int k, int nb) {
    if (b != 0) return;
    for (int e = t; e < CH_NB * CH_NB; e += 256) {
      const int r = e / CH_NB, c = e % CH_NB;
      if (r < nb && c <= r) A[(size_t)(k + r) * n + k + c] = (c < r) ? D[r][c] : rinv[r];
    }
  };

  for (int k = 0; k < n; k += CH_NB) {
    const int nb = min(CH_NB, n - k);
    // 1. diagonal block -> one warp, lane = row
    if (wid == 0) {
      double a[CH_NB], dg[CH_NB];
#pragma unroll
      for (int j = 0; j < CH_NB; ++j) {
        a[j] = (lane < nb && j < lane) ? __ldcg(A + (size_t)(k + lane) * n + k + j) : 0.0;
        dg[j] = (j < nb) ? __ldcg(A + (size_t)(k + j) * n + k + j) : 1.0;
      }
      bool bad = false;
      chol_cols<0>(a, dg, lane, col, bad);
      if (bad && lane == 0 && b == 0) atomicOr(fail, 1);
#pragma unroll
      for (int j = 0; j < CH_NB; ++j) D[lane][j] = (j < lane) ? a[j] : 0.0;
#pragma unroll
      for (int j = 0; j < CH_NB; ++j)
        if (lane == j) rinv[j] = dg[j];
    }
    __syncthreads();
    CH_TICK(0);
    // 2. panel rows below (and the rhs row n):  x L^T = a, one row per thread, rows dealt
    //    round-robin over the CTAs (up to n + 1 - 32 rows: small grids take several per thread)
    {
      const int rows = n + 1 - (k + nb);
      for (int i = t * G + b; i < rows; i += 256 * G) {
        double* row = A + (size_t)(k + nb + i) * n + k;
        double x[CH_NB];
#pragma unroll
        for (int c = 0; c < CH_NB; ++c) x[c] = (c < nb) ? __ldcg(row + c) : 0.0;
#pragma unroll
        for (int m = 0; m < CH_NB; ++m) {
          x[m] *= rinv[m];
#pragma unroll
          for (int c = m + 1; c < CH_NB; ++c) x[c] = fma(-x[m], D[c][m], x[c]);
        }
#pragma unroll
        for (int c = 0; c < CH_NB; ++c)
          if (c < nb) row[c] = x[c];
      }
    }
    const int base = k + CH_NB;
    if (base >= n) break;             // last panel: the rhs row is done, nothing trails
    __syncthreads();
    CH_TICK(1);
    grid_barrier(counter, (++phase) * G, fail);
    CH_TICK(2);
    store_diag(k, nb);
    // 3. trailing update, 32 x 32 tiles (ti >= tj), rows up to n (rhs), columns < n, dealt
    //    round-robin over the CTAs; thread = (column lane, rows wid + 8 m)
    {
      const int ntr = (n + 1 - base + CH_NB - 1) / CH_NB, ntc = (n - base + CH_NB - 1) / CH_NB;
      int turn = b;                      // tiles until this CTA's next one
      for (int ti = 0; ti < ntr; ++ti) {
        const int ncol = min(ti + 1, ntc);
        int tj = turn;
        for (; tj < ncol; tj += G) {
          __syncthreads();
          double old[4];
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const int gi = base + ti * CH_NB + wid + 8 * m, gj = base + tj * CH_NB + lane;
            old[m] = (gi <= n && gj < n && gj <= gi) ? __ldcg(A + (size_t)gi * n + gj) : 0.0;
          }
          for (int e = t; e < CH_NB * CH_NB; e += 256) {
            const int r = e / CH_NB, c = e % CH_NB;
            const int gi = base + ti * CH_NB + r, gj = base + tj * CH_NB + r;
            Pi[r][c] = (gi <= n) ? __ldcg(A + (size_t)gi * n + k + c) : 0.0;
            Pj[r][c] = (gj < n) ? __ldcg(A + (size_t)gj * n + k + c) : 0.0;
          }
          __syncthreads();
          double s[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
          for (int c = 0; c < CH_NB; c += 2) {
            const double q0 = Pj[lane][c], q1 = Pj[lane][c + 1];
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              const double2 pi = *reinterpret_cast<const double2*>(&Pi[wid + 8 * m][c]);
              s[m] = fma(pi.x, q0, s[m]);
              s[m] = fma(pi.y, q1, s[m]);
            }
          }
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            const int gi = base + ti * CH_NB + wid + 8 * m, gj = base + tj * CH_NB + lane;
            if (gi <= n && gj < n && gj <= gi) A[(size_t)gi * n + gj] = old[m] - s[m];
          }
        }
        turn = tj - ncol;
      }
    }
    __syncthreads();
    CH_TICK(3);
    grid_barrier(counter, (++phase) * G, fail);
    CH_TICK(4);
  }
  grid_barrier(counter, (++phase) * G, fail);
  if (b != 0) return;
  store_diag(CH_NB * ((n - 1) / CH_NB), n - CH_NB * ((n - 1) / CH_NB));
  __syncthreads();
  CH_TICK(4);
  // 4. back substitution L^T x = z (z = row n), CTA 0; the diagonal holds 1 / l_jj
  for (int i = t; i < n; i += 256) y[i] = __ldcg(A + (size_t)n * n + i);
  __syncthreads();
  const int nblk = (n + CH_NB - 1) / CH_NB;
  double lcol[CH_NB];   // lcol[j] = L[kb+j][kb+lane], j > lane ; lcol[lane] = 1 / l
  auto load_lcol = [&](int bi) {
    const int kb = bi * CH_NB, nb = min(CH_NB, n - kb);
#pragma unroll
    for (int j = 0; j < CH_NB; ++j)
      lcol[j] = (lane < nb && j >= lane && j < nb) ? __ldcg(A + (size_t)(kb + j) * n + kb + lane)
                                                    : ((j == lane) ? 1.0 : 0.0);
  };
  if (wid == 0) load_lcol(nblk - 1);
  for (int bi = nblk - 1; bi >= 0; --bi) {
    const int kb = bi * CH_NB;
    const int nb = min(CH_NB, n - kb);
    if (wid == 0) {
      double v = (lane < nb) ? y[kb + lane] : 0.0;
#pragma unroll
      for (int jj = 0; jj < CH_NB; ++jj) {
        const int j = CH_NB - 1 - jj;
        if (lane == j) v *= lcol[j];
        const double xj = __shfl_sync(0xffffffffu, v, j);
        if (lane < j) v = fma(-lcol[j], xj, v);
      }
      if (lane < nb) y[kb + lane] = v;
      if (bi > 0) load_lcol(bi - 1);      // in flight while the other warps update y below
    }
    __syncthreads();
    for (int i = t; i < kb; i += 256) {
      double s = y[i];
#pragma unroll 8
      for (int c = 0; c < nb; ++c) s = fma(-__ldcg(A + (size_t)(kb + c) * n + i), y[kb + c], s);
      y[i] = s;
    }
    __syncthreads();
  }
  for (int i = t; i < n; i += 256) out[i] = y[i];
  CH_TICK(5);
  if (dbg && t == 0)
    for (int i = 0; i < 6; ++i) dbg[i] = tm[i];
#undef CH_TICK
}

// A_out (n + 1 rows) = [A_in + mu * diag(d^2) ; rhs]
__global__ void k_copy_damped_rhs(const double* __restrict__ Ain, int n, double mu,
                                  const double* __restrict__ d, const double* __restrict__ rhs,
                                  double* __restrict__ Aout) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)(n + 1) * n) return;
  const int r = (int)(idx / n), c = (int)(idx % n);
  if (r == n) { Aout[idx] = rhs[c]; return; }
  double v = Ain[idx];
  if (r == c && mu != 0.0) v = fma(mu * d[r], d[r], v);
  Aout[idx] = v;
}

}  // namespace lcba
