// Reduced camera system: per point eliminate the 3x3 block and accumulate
//   S_jk += [j==k] Jc_j^T Jc_j - Y_j Y_k^T ,  rhs_j -= Y_j z ,   Y_j = (Jc_j^T Jp_j) L^-T
// over all camera pairs (j >= k) that see the point (V + lam Dp^2 = L L^T, z = L^-1 g_p).
// This is the FP64-pipe-bound kernel of the iteration (SURVEY.md section 8d): ~363 DFMA
// per (point, camera pair).  J is never materialised; Y lives in shared memory only.
//
// Decomposition.  Cameras are grouped in duos; a half-warp owns one 2x2 duo block
// (4 camera pairs) with its 4 x 9 accumulators in registers: lane (rr,cc) of the 4x4
// half-warp grid holds rows 3rr..3rr+2 x cols 3cc..3cc+2 of every 11x11 (padded to 12)
// pair block.  A CTA ("kind") owns up to 32 duo blocks and streams a slice of the points:
//   phase 1: threads = (point, camera slot) -> Jacobian blocks -> Y (and Jc for the
//            diagonal pairs) into shared memory, K-major [slice][row-group][4];
//   phase 2: half-warps run the rank-3 (+ rank-2 on the diagonal) updates for the pairs
//            whose two cameras both see the point (visibility mask test, no divergence
//            inside a half-warp).
// Partials per point-slice are written without atomics and summed in a fixed order.
#pragma once
#include <stdlib.h>
#include <algorithm>
#include <vector>
#include "common.cuh"
#include "control.cuh"

namespace lcba {

constexpr int SCHUR_MAX_HW_A = 20;   // config A: 10 consumer + 2 producer warps x 160 registers
constexpr int SCHUR_MAX_HW_B = 24;   // config B: 12 consumer + 4 producer warps x 128 registers
constexpr int SCHUR_MAX_HW = 24;     // consumer half-warps (duo blocks) per CTA: 12 consumer + 4 producer
                                     // warps x 128 registers: 3 consumers + 1 producer per SM sub-partition
constexpr int SCHUR_STAGES = 2;
constexpr int Y_LD = 50;             // doubles per (point, slot): 3 K-slices x 4 row groups x 4, +2 pad
constexpr int JC_LD = 34;            // doubles per (point, diag slot): 2 K-slices x 16, +2 pad
// (both strides are = 4 banks mod 32 and multiples of 16 B: conflict-free 128-bit stores from
//  consecutive lanes in phase 1, aligned 128-bit loads in phase 2)

struct SchurHw {          // one duo block = 2x2 camera pairs
  int8_t s[4];            // shared-memory slots of cams j0, j1, k0, k1
  int8_t c[4];            // camera ids   j0, j1, k0, k1 (0 when absent; see valid)
  uint8_t valid;          // bit (2*ja + kb): pair (j_ja, k_kb) is a lower-triangle pair
  uint8_t diag;           // same bit layout: pair is a diagonal pair (same camera)
  int8_t ds[2];           // Jc slots of j0, j1 (diagonal blocks only)
  uint8_t pad[4];
};

struct SchurKind {
  int nslots, nhw, hw_base, threads;
  int ndiag, qpr, pad0, pad1;             // diagonal (Jc) slots; first producer thread; points per stage
  uint8_t slot_cam[LCBA_MAX_CAMERAS];
  int8_t slot_dslot[LCBA_MAX_CAMERAS];    // Jc slot of a camera slot or -1
};

struct SchurPlan {
  int C = 0, nkinds = 0, nslices = 0, pc = 0, max_threads = 0, max_slots = 0;
  int npairs = 0;
  int cfg = 0;              // 0 = config A (12 warps x 160 regs), 1 = config B (16 warps x 128 regs)
  size_t part_stride = 0;   // doubles per slice partial: npairs*121 + 11*C
  size_t smem_bytes = 0;
  std::vector<SchurKind> kinds;
  std::vector<SchurHw> hws;
};

inline int pair_index(int j, int k) { return j * (j + 1) / 2 + k; }

inline size_t schur_smem_bytes(int C, int pc, int nslots, int ndiag) {
  return ((size_t)pc * nslots * Y_LD + (size_t)pc * ndiag * JC_LD + (size_t)pc * 2 +
          (size_t)C * CAMTAB) * 8 + 64;
}

inline SchurPlan make_schur_plan_cfg(int C, int sm_count, size_t smem_limit, int cfg) {
  SchurPlan pl;
  pl.C = C;
  pl.cfg = cfg;
  const int max_hw = cfg == 1 ? SCHUR_MAX_HW_B : (cfg == 2 ? 16 : SCHUR_MAX_HW_A);
  const int prod_warps = cfg == 0 ? 2 : 4;
  const int nb = (C + 1) / 2;
  pl.npairs = C * (C + 1) / 2;
  pl.part_stride = (size_t)pl.npairs * 121 + (size_t)NCP * C;
  // Partition the lower-triangular duo-block matrix into kinds.  Greedy clustering over camera
  // duos: a kind keeps a duo set D and takes every free block inside D x D; when none is left it
  // adds the duo that unlocks the most free blocks.  Kinds become compact cliques / rectangles
  // (few cameras each), so their producers compute few (point, camera) Jacobians.
  std::vector<std::vector<char>> freeb(nb, std::vector<char>(nb, 0));
  size_t nfree = 0;
  for (int j = 0; j < nb; ++j)
    for (int k = 0; k <= j; ++k) { freeb[j][k] = 1; ++nfree; }
  pl.pc = 0;
  while (nfree > 0) {
    SchurKind K{};
    K.hw_base = (int)pl.hws.size();
    bool used[LCBA_MAX_CAMERAS] = {false}, isdiag[LCBA_MAX_CAMERAS] = {false};
    std::vector<char> inD(nb, 0);
    std::vector<std::pair<int, int>> blks;
    int nd = 0;
    bool full = false;
    while (nfree > 0 && !full) {
      // 1. a free block inside D x D (row-major)
      int bj = -1, bk = -1;
      for (int j = 0; j < nb && bj < 0; ++j) {
        if (!inD[j]) continue;
        for (int k = 0; k <= j; ++k)
          if (inD[k] && freeb[j][k]) { bj = j; bk = k; break; }
      }
      if (bj < 0) {
        // 2. grow D by the duo that unlocks the most free blocks
        int best = -1, gain_best = 0;
        for (int d = 0; d < nb; ++d) {
          if (inD[d]) continue;
          int gain = freeb[d][d] ? 1 : 0;
          for (int x = 0; x < nb; ++x)
            if (inD[x]) gain += (x < d) ? freeb[d][x] : freeb[x][d];
          if (gain > gain_best) { gain_best = gain; best = d; }
        }
        if (best < 0) {   // D empty or exhausted: seed with the first free block
          for (int j = 0; j < nb && best < 0; ++j)
            for (int k = 0; k <= j; ++k)
              if (freeb[j][k]) { inD[j] = 1; inD[k] = 1; best = j; break; }
        } else {
          inD[best] = 1;
        }
        continue;
      }
      const int dg = (bj == bk) ? 1 : 0;
      // a kind with an odd number of diagonal blocks needs one idle half-warp
      if ((int)blks.size() + 1 + ((nd + dg) & 1) > max_hw) { full = true; break; }
      nd += dg;
      freeb[bj][bk] = 0;
      --nfree;
      blks.push_back({bj, bk});
      for (int d = 0; d < 2; ++d) {
        if (2 * bj + d < C) used[2 * bj + d] = true;
        if (2 * bk + d < C) used[2 * bk + d] = true;
        if (bj == bk && 2 * bj + d < C) isdiag[2 * bj + d] = true;
      }
    }
    int slot_of[LCBA_MAX_CAMERAS], dslot_of[LCBA_MAX_CAMERAS];
    K.nslots = 0;
    K.ndiag = 0;
    for (int c = 0; c < C; ++c)
      if (used[c]) {
        slot_of[c] = K.nslots;
        dslot_of[c] = isdiag[c] ? K.ndiag++ : -1;
        K.slot_dslot[K.nslots] = (int8_t)dslot_of[c];
        K.slot_cam[K.nslots++] = (uint8_t)c;
      }
    // diagonal duo blocks first and in pairs, so that a warp is either all-diagonal (3 pairs +
    // the rank-2 U update) or all-regular (4 pairs): balanced work per warp
    std::stable_sort(blks.begin(), blks.end(), [](const std::pair<int, int>& a, const std::pair<int, int>& b) {
      return (a.first == a.second) > (b.first == b.second);
    });
    int ndblk = 0;
    for (auto& bl : blks) ndblk += bl.first == bl.second;
    if (ndblk & 1) blks.insert(blks.begin() + ndblk, std::make_pair(-1, -1));   // idle half-warp
    for (auto& bl : blks) {
      SchurHw h{};
      if (bl.first < 0) { pl.hws.push_back(h); continue; }
      const int cj[2] = {2 * bl.first, 2 * bl.first + 1};
      const int ck[2] = {2 * bl.second, 2 * bl.second + 1};
      for (int d = 0; d < 2; ++d) {
        h.c[d] = (int8_t)(cj[d] < C ? cj[d] : 0);
        h.s[d] = (int8_t)(cj[d] < C ? slot_of[cj[d]] : 0);
        h.c[2 + d] = (int8_t)(ck[d] < C ? ck[d] : 0);
        h.s[2 + d] = (int8_t)(ck[d] < C ? slot_of[ck[d]] : 0);
        h.ds[d] = (int8_t)((bl.first == bl.second && cj[d] < C) ? dslot_of[cj[d]] : 0);
      }
      for (int ja = 0; ja < 2; ++ja)
        for (int kb = 0; kb < 2; ++kb)
          if (cj[ja] < C && ck[kb] < C && ck[kb] <= cj[ja]) {
            h.valid |= (uint8_t)(1u << (2 * ja + kb));
            if (ck[kb] == cj[ja]) h.diag |= (uint8_t)(1u << (2 * ja + kb));
          }
      pl.hws.push_back(h);
    }
    K.nhw = (int)blks.size();
    const int cons_threads = 32 * ((K.nhw + 1) / 2);
    K.threads = cons_threads + 32 * prod_warps;
    K.qpr = cons_threads;                       // first producer thread
    pl.max_threads = std::max(pl.max_threads, K.threads);
    pl.max_slots = std::max(pl.max_slots, K.nslots);
    // points per stage: SCHUR_STAGES stages must fit shared memory
    {
      const size_t per_pt = ((size_t)K.nslots * Y_LD + (size_t)K.ndiag * JC_LD + 2) * 8;
      const size_t fixed = (size_t)C * CAMTAB * 8 + 64;
      const int sp = (int)((smem_limit - fixed) / (per_pt * SCHUR_STAGES));
      K.pad0 = std::max(1, std::min(16, sp));
    }
    pl.smem_bytes = std::max(pl.smem_bytes,
                             schur_smem_bytes(C, K.pad0 * SCHUR_STAGES, K.nslots, K.ndiag));
    pl.kinds.push_back(K);
  }
  pl.nkinds = (int)pl.kinds.size();
  pl.nslices = std::max(1, sm_count / pl.nkinds);
  return pl;
}

// Config B holds 20 % more duo blocks per CTA but each CTA runs ~1.27x slower (measured on
// B200): take it only when it saves enough kinds (e.g. 18 cameras: 2 kinds instead of 3).
inline SchurPlan make_schur_plan(int C, int sm_count, size_t smem_limit) {
  SchurPlan a = make_schur_plan_cfg(C, sm_count, smem_limit, 0);
  SchurPlan b = make_schur_plan_cfg(C, sm_count, smem_limit, 1);
  if (getenv("LCBA_SCHUR_CFG")) {
    const int c = atoi(getenv("LCBA_SCHUR_CFG"));
    return make_schur_plan_cfg(C, sm_count, smem_limit, c);
  }
  return (1.27 * b.nkinds < 1.0 * a.nkinds) ? b : a;
}

__device__ __forceinline__ void ld3(const double* __restrict__ p, double (&v)[3]) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  v[0] = a.x; v[1] = a.y; v[2] = p[2];
}

template <bool SUB>
__device__ __forceinline__ void outer9(double (&acc)[9], const double (&a)[3], const double (&b)[3]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      acc[3 * i + j] = SUB ? fma(-a[i], b[j], acc[3 * i + j]) : fma(a[i], b[j], acc[3 * i + j]);
}

__device__ __forceinline__ void st4(double* p, double a, double b, double c, double d) {
  *reinterpret_cast<double2*>(p) = make_double2(a, b);
  *reinterpret_cast<double2*>(p + 2) = make_double2(c, d);
}

// Phase 1 for one (point, camera slot): Y = (Jc^T Jp) L^-T into Ys, Jc into Js (diagonal slots).
// Invisible cameras produce exact zeros (w = 0, masked divide) so that phase 2 needs no
// per-pair visibility test.
struct ProdIn {
  const double* T;
  double X[3], li[9], w;
  double *Y, *Js;
  bool live;
};

__device__ __forceinline__ void schur_produce(const ProdIn& in) {
  ObsLin L;
  obs_linearize<false>(in.T, in.X[0], in.X[1], in.X[2], 0.0, 0.0, in.w, L, in.live);
  const double w = in.w;
  const double* li = in.li;
  double* Y = in.Y;
  double Q[2][3];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    Q[i][0] = L.Jp[i][0] * li[0];
    Q[i][1] = fma(L.Jp[i][0], li[1], L.Jp[i][1] * li[2]);
    Q[i][2] = fma(L.Jp[i][0], li[3], fma(L.Jp[i][1], li[4], L.Jp[i][2] * li[5]));
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    double y[9];
#pragma unroll
    for (int a = 0; a < 9; ++a) y[a] = fma(L.Jc[0][a], Q[0][k], L.Jc[1][a] * Q[1][k]);
    st4(Y + k * 16 + 0, y[0], y[1], y[2], 0.0);
    st4(Y + k * 16 + 4, y[3], y[4], y[5], 0.0);
    st4(Y + k * 16 + 8, y[6], y[7], y[8], 0.0);
    // row 11 is padding for the 12x12 lane grid: it carries z = L^-1 g_p, so that column 11
    // of the diagonal pair block accumulates -Y_j z = the reduced right-hand side for free
    st4(Y + k * 16 + 12, w * Q[0][k], w * Q[1][k], li[6 + k], 0.0);
  }
  if (in.Js) {
    double* Js = in.Js;
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      st4(Js + i * 16 + 0, L.Jc[i][0], L.Jc[i][1], L.Jc[i][2], 0.0);
      st4(Js + i * 16 + 4, L.Jc[i][3], L.Jc[i][4], L.Jc[i][5], 0.0);
      st4(Js + i * 16 + 8, L.Jc[i][6], L.Jc[i][7], L.Jc[i][8], 0.0);
      st4(Js + i * 16 + 12, i == 0 ? w : 0.0, i == 1 ? w : 0.0, 0.0, 0.0);
    }
  }
}

// SKIP: test the visibility mask per (point, duo block) and skip blocks nobody sees
// (sparse rigs); without it every block is computed (zeros contribute nothing).
//
// Warp-specialised: the last SCHUR_PROD_WARPS warps are producers (phase 1: latency-bound
// Jacobian + Y into a 2-stage shared-memory ring), the others consumers (phase 2: the DFMA
// stream).  Stages are handed over with named barriers: producers bar.arrive FULL[s] /
// bar.sync EMPTY[s], consumers bar.sync FULL[s] / bar.arrive EMPTY[s].
__device__ __forceinline__ void nbar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void nbar_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}

template <bool SKIP, int NREG>
__global__ void __maxnreg__(NREG)
k_schur(const double* __restrict__ tab, const double* __restrict__ pts,
        const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
        const unsigned long long* __restrict__ mask, const double* __restrict__ Lz, long long P,
        long long N, int C, const SchurKind* __restrict__ kinds, const SchurHw* __restrict__ hws,
        int nslices, size_t part_stride, int npairs, double* __restrict__ part,
        long long* __restrict__ stats) {
  extern __shared__ __align__(16) double s_dyn[];
  const SchurKind& K = kinds[blockIdx.y];
  const long long t_start = clock64();
  long long t_wait = 0;
  const int nthreads = K.threads;
  const int tid = threadIdx.x;
  if (tid >= nthreads) return;          // uniform per warp (threads multiple of 32)
  const int nslots = K.nslots, ndiag = K.ndiag, SP = K.pad0, prod0 = K.qpr;
  // per stage: Y[SP][nslots][Y_LD] J[SP][ndiag][JC_LD] mask[SP] pad[SP] (even => 16 B)
  const size_t stage_doubles = (size_t)SP * nslots * Y_LD + (size_t)SP * ndiag * JC_LD + SP * 2;
  double* s_tab = s_dyn + SCHUR_STAGES * stage_doubles;      // C * CAMTAB
  enum { BAR_FULL = 2, BAR_EMPTY = BAR_FULL + SCHUR_STAGES, BAR_PROD = BAR_EMPTY + SCHUR_STAGES };

  // slice boundaries balanced by observation count
  const int slice = blockIdx.x;
  long long pa, pb;
  {
    const unsigned long long ta = (unsigned long long)N * slice / nslices;
    const unsigned long long tb = (unsigned long long)N * (slice + 1) / nslices;
    pa = (slice == 0) ? 0 : lower_bound_u32(obs_start, P, ta);
    pb = (slice == nslices - 1) ? P : lower_bound_u32(obs_start, P, tb);
  }
  const long long nchunks = (pb - pa + SP - 1) / SP;

  if (tid >= prod0) {
    // =============================== producers ===============================
    const int ptid = tid - prod0, nprod = nthreads - prod0;
    for (int i = ptid; i < C * CAMTAB; i += nprod) s_tab[i] = tab[i];
    nbar_sync(BAR_PROD, nprod);
    for (long long c = 0; c < nchunks + SCHUR_STAGES; ++c) {
      const int st = (int)(c % SCHUR_STAGES);
      if (c >= SCHUR_STAGES) { const long long t0 = clock64(); nbar_sync(BAR_EMPTY + st, nthreads); t_wait += clock64() - t0; }
      if (c >= nchunks) continue;
      double* s_Y = s_dyn + st * stage_doubles;
      double* s_J = s_Y + (size_t)SP * nslots * Y_LD;
      unsigned long long* s_mask =
          reinterpret_cast<unsigned long long*>(s_J + (size_t)SP * ndiag * JC_LD);
      const long long q0 = pa + c * SP;
      const int npc = (int)min((long long)SP, pb - q0);
      const int total = npc * nslots;
      for (int idx = ptid; idx < total; idx += nprod) {
        ProdIn in;
        const int q = idx / nslots, sl = idx - q * nslots;
        const long long p = q0 + q;
        const unsigned long long m = mask[p];
        const int cam = K.slot_cam[sl];
        const int ds = K.slot_dslot[sl];
        in.live = (m >> cam) & 1ull;
        in.w = 0.0;
        if (in.live)
          in.w = wgt ? wgt[(long long)obs_start[p] + __popcll(m & ((1ull << cam) - 1ull))] : 1.0;
        in.T = s_tab + cam * CAMTAB;
#pragma unroll
        for (int a = 0; a < 3; ++a) in.X[a] = pts[3 * p + a];
#pragma unroll
        for (int a = 0; a < 9; ++a) in.li[a] = Lz[p * 9 + a];
        in.Y = s_Y + ((size_t)q * nslots + sl) * Y_LD;
        in.Js = ds >= 0 ? s_J + ((size_t)q * ndiag + ds) * JC_LD : nullptr;
        schur_produce(in);
      }
      for (int q = ptid; q < npc; q += nprod) s_mask[q] = mask[q0 + q];
      __threadfence_block();
      nbar_arrive(BAR_FULL + st, nthreads);
    }
    if (stats && tid == prod0) {
      long long* o = stats + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 4;
      o[2] = t_wait;
      o[3] = clock64() - t_start;
    }
    return;
  }

  // =============================== consumers ===============================
  const int hw = tid >> 4, l16 = tid & 15, rr = l16 >> 2, cc = l16 & 3;
  SchurHw D{};
  if (hw < K.nhw) D = hws[K.hw_base + hw];
  const unsigned valid = D.valid, diag = D.diag;
  const int oj0 = D.s[0] * Y_LD + rr * 4, oj1 = D.s[1] * Y_LD + rr * 4;
  const int ok0 = D.s[2] * Y_LD + cc * 4, ok1 = D.s[3] * Y_LD + cc * 4;
  unsigned long long bm_j = 0, bm_k = 0;      // cameras of the block, for the SKIP test
  if (valid) {
    bm_j = (1ull << D.c[0]) | ((valid & 12u) ? (1ull << D.c[1]) : 0ull);
    bm_k = (1ull << D.c[2]) | ((valid & 10u) ? (1ull << D.c[3]) : 0ull);
  }
  // all-diagonal warp: pairs 00, 10, 11 (+ U); all-regular warp: pairs 00, 01, 10, 11
  const bool dwarp = __any_sync(0xffffffffu, diag != 0);
  double acc[4][9];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 9; ++j) acc[i][j] = 0.0;

  for (long long c = 0; c < nchunks; ++c) {
    const int st = (int)(c % SCHUR_STAGES);
    const double* s_Y = s_dyn + st * stage_doubles;
    const double* s_J = s_Y + (size_t)SP * nslots * Y_LD;
    const unsigned long long* s_mask =
        reinterpret_cast<const unsigned long long*>(s_J + (size_t)SP * ndiag * JC_LD);
    const int npc = (int)min((long long)SP, pb - (pa + c * SP));
    { const long long t0 = clock64(); nbar_sync(BAR_FULL + st, nthreads); t_wait += clock64() - t0; }
    if (valid) {
      const double* Yq = s_Y;
      for (int q = 0; q < npc; ++q, Yq += nslots * Y_LD) {
        if (SKIP) {
          const unsigned long long m = s_mask[q];
          if (!(m & bm_j) || !(m & bm_k)) continue;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          double a0[3], a1[3], b0[3], b1[3];
          ld3(Yq + oj0 + k * 16, a0);
          ld3(Yq + oj1 + k * 16, a1);
          ld3(Yq + ok0 + k * 16, b0);
          ld3(Yq + ok1 + k * 16, b1);
          // DFMA issue order chosen for register-operand reuse: a DFMA with three fresh
          // 64-bit register operands issues every 3 cycles on B200, every 2 with one operand
          // held in the reuse cache (tools/fp64_operands.cu: 24.7 vs 34.1 TFLOP/s).  Six
          // consecutive products share a[i]; the sweep direction over b alternates so that the
          // first product of a row group reuses the last b of the previous one.
          if (!dwarp) {
#pragma unroll
            for (int i = 0; i < 3; ++i) {
#pragma unroll
              for (int jj = 0; jj < 6; ++jj) {
                const int j6 = (i & 1) ? 5 - jj : jj;
                const int j = j6 % 3;
                if (j6 < 3) acc[0][3 * i + j] = fma(-a0[i], b0[j], acc[0][3 * i + j]);
                else        acc[1][3 * i + j] = fma(-a0[i], b1[j], acc[1][3 * i + j]);
              }
            }
          } else {
            outer9<true>(acc[0], a0, b0);
          }
#pragma unroll
          for (int i = 0; i < 3; ++i) {
#pragma unroll
            for (int jj = 0; jj < 6; ++jj) {
              const int j6 = (i & 1) ? jj : 5 - jj;
              const int j = j6 % 3;
              if (j6 < 3) acc[2][3 * i + j] = fma(-a1[i], b0[j], acc[2][3 * i + j]);
              else        acc[3][3 * i + j] = fma(-a1[i], b1[j], acc[3][3 * i + j]);
            }
          }
        }
        if (dwarp) {   // U_j = sum Jc^T Jc on the diagonal pairs
          const double* Jq = s_J + (size_t)q * ndiag * JC_LD;
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            double a[3], b[3];
            ld3(Jq + D.ds[0] * JC_LD + k * 16 + rr * 4, a);
            ld3(Jq + D.ds[0] * JC_LD + k * 16 + cc * 4, b);
            outer9<false>(acc[0], a, b);
            ld3(Jq + D.ds[1] * JC_LD + k * 16 + rr * 4, a);
            ld3(Jq + D.ds[1] * JC_LD + k * 16 + cc * 4, b);
            outer9<false>(acc[3], a, b);
          }
        }
      }
    }
    nbar_arrive(BAR_EMPTY + st, nthreads);
  }
  if (stats && tid == 0) {
    long long* o = stats + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 4;
    o[0] = t_wait;
    o[1] = clock64() - t_start;
  }
  // ---------------- write the slice partial (every lower-triangle entry exactly once) ----
  if (valid) {
    double* out = part + (size_t)slice * part_stride;
#pragma unroll
    for (int pr = 0; pr < 4; ++pr) {
      if (!((valid >> pr) & 1u)) continue;
      const int cj = D.c[pr >> 1], ck = D.c[2 + (pr & 1)];
      double* blk = out + (size_t)(cj * (cj + 1) / 2 + ck) * 121;
#pragma unroll
      for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
          const int a = 3 * rr + i, b = 3 * cc + j;
          if (a < NCP && b < NCP) blk[a * NCP + b] = acc[pr][3 * i + j];
        }
    }
    if (cc == 3) {   // column 11 of the diagonal pair blocks = reduced right-hand side
      double* rout = out + (size_t)npairs * 121;
#pragma unroll
      for (int d = 0; d < 2; ++d) {
        if (!((diag >> (3 * d)) & 1u)) continue;
        const int cj = D.c[d];
#pragma unroll
        for (int i = 0; i < 3; ++i)
          if (3 * rr + i < NCP) rout[cj * NCP + 3 * rr + i] = acc[3 * d][3 * i + 2];
      }
    }
  }
}

// S (n x n, both triangles) = reduced blocks + lam * diag(scl_c^2) ; rhs = g_c + rhs_red.
// lam: the device control block's reg_term when `ctl` is given, the argument otherwise.
// A held camera entry (cam_fixed[i] != 0; cam_fixed may be NULL) turns row and column i into
// those of the identity and rhs[i] into 0: dropping camera columns commutes with eliminating the
// points, so the free block is the reduced system of the free parameters, and the Cholesky returns
// an exact 0 for entry i (scl_c[i] = 1 there, so the retries' mu damping keeps the row diagonal).
__global__ void k_assemble_S(const double* __restrict__ red, int C, int npairs,
                             const double* __restrict__ camsum, const double* __restrict__ scl_c,
                             double lam, const Ctl* __restrict__ ctl,
                             const uint8_t* __restrict__ cam_fixed, double* __restrict__ S,
                             double* __restrict__ rhs) {
  if (ctl) lam = ctl->reg_term;
  const int n = C * NCP;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * n) return;
  const int r = (int)(idx / n), c = (int)(idx % n);
  if (cam_fixed && (cam_fixed[r] || cam_fixed[c])) {
    S[idx] = r == c ? 1.0 : 0.0;
    if (r == c) rhs[r] = 0.0;
    return;
  }
  const int hi = max(r, c), lo = min(r, c);
  const int j = hi / NCP, a = hi % NCP, k = lo / NCP, b = lo % NCP;
  double v;
  if (j == k) {
    // diagonal block is stored in full (both halves computed from the same products)
    v = red[(size_t)(j * (j + 1) / 2 + j) * 121 + (r % NCP) * NCP + (c % NCP)];
  } else {
    v = red[(size_t)(j * (j + 1) / 2 + k) * 121 + a * NCP + b];
  }
  if (r == c) {
    const double s = scl_c[r];
    v = fma(lam * s, s, v);
    rhs[r] = camsum[(r / NCP) * 22 + (r % NCP)] + red[(size_t)npairs * 121 + r];
  }
  S[idx] = v;
}


// ---- shared intrinsics (PySBA.bundleAdjust_sharedcam, pySBA.py:252-325) -------------------
// Reduced parameter order of the reference: [f k1 k2 | 6 extrinsics per camera | cx cy per
// camera].  J_red = J_full T with a 0/1 matrix T, so S_red = T^T S_full T (+ damping once per
// reduced parameter) and rhs_red = T^T rhs_full.
__host__ __device__ inline int shared_red_index(int c, int a, int C) {
  return a < 6 ? 3 + 6 * c + a : (a < 9 ? a - 6 : 3 + 6 * C + 2 * c + (a - 9));
}

__device__ __forceinline__ double sfull_entry(const double* __restrict__ red, int r, int c) {
  const int hi = max(r, c), lo = min(r, c);
  const int j = hi / NCP, a = hi % NCP, k = lo / NCP, b = lo % NCP;
  if (j == k) return red[(size_t)(j * (j + 1) / 2 + j) * 121 + (r % NCP) * NCP + (c % NCP)];
  return red[(size_t)(j * (j + 1) / 2 + k) * 121 + a * NCP + b];
}

// preimage of reduced index i: cameras [c0, c1) and the full parameter slot a
__device__ __forceinline__ void shared_preimage(int i, int C, int& c0, int& c1, int& a) {
  if (i < 3) { c0 = 0; c1 = C; a = 6 + i; }
  else if (i < 3 + 6 * C) { c0 = (i - 3) / 6; c1 = c0 + 1; a = (i - 3) % 6; }
  else { c0 = (i - 3 - 6 * C) / 2; c1 = c0 + 1; a = 9 + (i - 3 - 6 * C) % 2; }
}

__global__ void k_assemble_S_shared(const double* __restrict__ red, int C, int npairs,
                                    const double* __restrict__ camsum,
                                    const double* __restrict__ scl_c, const Ctl* __restrict__ ctl,
                                    double lam_host, int use_ctl, double* __restrict__ S,
                                    double* __restrict__ rhs, double* __restrict__ scl_red) {
  const double lam = use_ctl ? ctl->reg_term : lam_host;
  const int n = 3 + 8 * C;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n * n) return;
  const int i = (int)(idx / n), j = (int)(idx % n);
  int ic0, ic1, ia, jc0, jc1, ja;
  shared_preimage(i, C, ic0, ic1, ia);
  shared_preimage(j, C, jc0, jc1, ja);
  double v = 0.0;
  for (int c = ic0; c < ic1; ++c)
    for (int d = jc0; d < jc1; ++d) v += sfull_entry(red, c * NCP + ia, d * NCP + ja);
  if (i == j) {
    const double s = scl_c[ic0 * NCP + ia];
    scl_red[i] = s;
    v = fma(lam * s, s, v);
    double r = 0.0;
    for (int c = ic0; c < ic1; ++c)
      r += camsum[c * 22 + ia] + red[(size_t)npairs * 121 + c * NCP + ia];
    rhs[i] = r;
  }
  S[idx] = v;
}

__global__ void k_expand_shared(const double* __restrict__ p_red, int C, double* __restrict__ pc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < C * NCP) pc[i] = p_red[shared_red_index(i / NCP, i % NCP, C)];
}

}  // namespace lcba
