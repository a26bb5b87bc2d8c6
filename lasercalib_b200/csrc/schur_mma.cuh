// Reduced camera system on the FP64 tensor path (DMMA, mma.sync m8n8k4 f64) for dense rigs.
//
// S - U = - sum_p Y_p Y_p^T is a symmetric rank-3P update: a SYRK with K = 3 P.  The DFMA
// kernel (schur.cuh) is bound by the shared-memory crossbar (12 operand doubles per 36 DFMA
// and lane) and by FP64 issue slots; with DMMA a lane loads ONE double per 8 x 8 x 4 fragment
// and the operand broadcast happens inside the tensor datapath: 12 doubles per 36 DMMA =
// 288 FMA per lane (8x less shared-memory traffic, 8x fewer issue slots).  Measured on B200
// (tools/dmma_syrk.cu, fragment loads included): 33.6 TFLOP/s with one warp per SM
// sub-partition, 36.9 with two.
//
// Decomposition.  The matrix that is accumulated is [Y; z] [Y; z]^T with the 11 C rows of Y
// UNPADDED and one extra row z = L^-1 g_p (its products with Y are the reduced right-hand
// side): 11 C + 1 rows = nt tiles of 8.  Only tiles on or below the diagonal are computed.
// Tile rows are grouped by 6; a consumer WARP owns one unit = (row group, column group): a
// 6 x 6 rectangle of tiles (72 FP64 accumulators per lane), a lower triangle of 21 on the
// diagonal, smaller at the last group.  Units are packed into CTAs ("kinds") of 8 consumer
// warps + 4 producer warps, balanced first over the kinds, then over the four SM
// sub-partitions of a kind (warp w runs on sub-partition w % 4: DMMA time is per
// sub-partition).  12 warps are launched with 168 registers; the producer warpgroup gives
// registers back (setmaxnreg.dec 88) and the two consumer warpgroups take them (inc 208).
//   producer: (point, camera) -> Y = (Jc^T Jp) L^-T (11 rows) into a 2-stage ring laid out
//             [kappa = 3 q + k][12 c + r | z 0 0 0], row stride = 4 (mod 16) doubles, so that
//             the fragment loads (lane -> row lane/4, kappa lane%4) are conflict free;
//   consumer: per K-step (4 kappa = 4/3 point) <= 12 LDS.64 + <= 36 DMMA.
// Invisible (point, camera) pairs and the tail of the last chunk are exact zeros.  The
// camera blocks U_j = sum Jc^T Jc are accumulated by k_cam_normal (one thread per (point,
// camera), fixed camera per thread, 66 register accumulators) and added to the diagonal pair
// blocks before the all-reduce, so everything downstream is unchanged.
#pragma once
#include <algorithm>
#include <vector>
#include "common.cuh"
#include "schur.cuh"

namespace lcba {

constexpr int MMA_CONS_WARPS = 8;     // consumer warps per CTA (two warpgroups)
constexpr int MMA_PROD_WARPS = 4;     // producer warps (one warpgroup)
constexpr int MMA_THREADS = 32 * (MMA_CONS_WARPS + MMA_PROD_WARPS);
constexpr int MMA_MAX_CAMERAS = 64;   // = LCBA_MAX_CAMERAS (every kind stages all cameras: 4 points per ring stage at 64)
#define MMA_CONS_REGS "208"
#define MMA_PROD_REGS "88"

struct MmaUnit {          // tile rectangle [tr0, tr0 + nr) x [tc0, tc0 + nc); nr = 0: idle warp
  int16_t tr0, tc0;
  int8_t nr, nc, tri, pad;
};

struct MmaKind {
  int nactive, rp, sp, pad0;            // active consumer warps; ring row stride; points per stage
  MmaUnit unit[MMA_CONS_WARPS];
};

struct MmaPlan {
  int C = 0, nkinds = 0, nslices = 0;
  size_t smem_bytes = 0;
  std::vector<MmaKind> kinds;
};

// need_tab: the producers evaluate Y in place and keep the camera tables in shared memory; with
// Y precomputed (k_make_Y) that space goes to the ring (24 cameras: 16 instead of 12 points per stage)
inline MmaPlan make_mma_plan(int C, int sm_count, size_t smem_limit, bool need_tab = true) {
  MmaPlan pl;
  pl.C = C;
  const int nrows = NCP * C + 1, nt = (nrows + 7) / 8, ng = (nt + 5) / 6;
  struct U { MmaUnit u; int cost; };
  std::vector<U> units;
  long long total = 0;
  for (int gi = 0; gi < ng; ++gi)
    for (int gj = 0; gj <= gi; ++gj) {
      U x{};
      x.u.tr0 = (int16_t)(6 * gi);
      x.u.tc0 = (int16_t)(6 * gj);
      x.u.nr = (int8_t)std::min(6, nt - 6 * gi);
      x.u.nc = (int8_t)std::min(6, nt - 6 * gj);
      x.u.tri = gi == gj;
      x.cost = x.u.tri ? x.u.nr * (x.u.nr + 1) / 2 : x.u.nr * x.u.nc;
      total += x.cost;
      units.push_back(x);
    }
  const int nk = (int)((units.size() + MMA_CONS_WARPS - 1) / MMA_CONS_WARPS);
  // spare warp slots: split full 6 x 6 units into two 3 x 6 halves (finer grain for the balance
  // over the sub-partitions; 24 cameras: max load 54 tiles instead of 60)
  for (size_t i = 0; i < units.size() && (int)units.size() < nk * MMA_CONS_WARPS; ++i) {
    if (units[i].u.tri || units[i].u.nr != 6 || units[i].u.nc != 6) continue;
    U lo = units[i];
    lo.u.nr = 3;
    lo.cost = 18;
    U hi = lo;
    hi.u.tr0 = (int16_t)(lo.u.tr0 + 3);
    units[i] = lo;
    units.push_back(hi);
  }
  std::sort(units.begin(), units.end(), [](const U& a, const U& b) { return a.cost > b.cost; });
  std::vector<std::vector<U>> per_kind(nk);
  std::vector<long long> kcost(nk, 0);
  for (const U& x : units) {   // longest processing time first, into the lightest kind with room
    int best = -1;
    for (int k = 0; k < nk; ++k)
      if ((int)per_kind[k].size() < MMA_CONS_WARPS && (best < 0 || kcost[k] < kcost[best])) best = k;
    per_kind[best].push_back(x);
    kcost[best] += x.cost;
  }
  int rp = C * 12 + 2;
  while (rp % 16 != 4) ++rp;
  const size_t fixed = (need_tab ? (size_t)C * CAMTAB * 8 : 0) + 64;
  int sp = (int)((smem_limit - fixed) / ((size_t)3 * rp * 8 * SCHUR_STAGES));
  sp = std::max(4, std::min(16, sp / 4 * 4));
  pl.smem_bytes = (size_t)3 * sp * rp * 8 * SCHUR_STAGES + fixed;
  for (int k = 0; k < nk; ++k) {
    MmaKind K{};
    K.rp = rp;
    K.sp = sp;
    // units of the kind over the sub-partitions (2 warp slots each): lightest one with room
    long long load[4] = {0, 0, 0, 0};
    int used[4] = {0, 0, 0, 0};
    for (const U& x : per_kind[k]) {   // already sorted by decreasing cost
      int best = -1;
      for (int q = 0; q < 4; ++q)
        if (used[q] < 2 && (best < 0 || load[q] < load[best])) best = q;
      K.unit[best + 4 * used[best]] = x.u;
      load[best] += x.cost;
      ++used[best];
      ++K.nactive;
    }
    pl.kinds.push_back(K);
  }
  pl.nkinds = nk;
  pl.nslices = std::max(1, sm_count / pl.nkinds);
  return pl;
}

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// One (point, camera) item: Y (11 rows + a zero) x 3 kappa, rows rp doubles apart.
__device__ __forceinline__ void mma_produce(const double* __restrict__ T, const double (&X)[3],
                                            const double (&li)[9], double w, bool live,
                                            double* __restrict__ Yk0, int rp) {
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
    double y[9];
#pragma unroll
    for (int a = 0; a < 9; ++a) y[a] = fma(L.Jc[0][a], Q[0][k], L.Jc[1][a] * Q[1][k]);
    double2* o = reinterpret_cast<double2*>(Yk0 + (size_t)k * rp);
    o[0] = make_double2(y[0], y[1]);
    o[1] = make_double2(y[2], y[3]);
    o[2] = make_double2(y[4], y[5]);
    o[3] = make_double2(y[6], y[7]);
    o[4] = make_double2(y[8], w * Q[0][k]);
    o[5] = make_double2(w * Q[1][k], 0.0);
  }
}

// Ring offset of matrix row rho: camera rows are stored with stride 12, then z, then zeros.
__device__ __forceinline__ int mma_row_offset(int rho, int C) {
  const int n = NCP * C;
  if (rho < n) return (rho / NCP) * 12 + rho % NCP;
  return C * 12 + (rho == n ? 0 : 1);
}

// ---- Y precomputed in HBM ------------------------------------------------------------------
// Inside k_schur_mma the producers' FP64 instructions have to squeeze in between the DMMAs of
// two consumer warps per sub-partition: every dependent step of the ~200-instruction Jacobian
// chain waits for a pipe slot and the producers, not the tensor pipe, set the pace (ncu: 29 %
// barrier stalls, tensor pipe 53 % active).  k_make_Y therefore evaluates Y once per iteration
// at full occupancy and stores it in exactly the ring layout ([point][kappa][rp] doubles, z
// and the zero column included): the producers of every kind then only copy contiguous rows
// with cp.async (no FP64 work, no registers).  Costs 288 B per (point, camera) of HBM write
// and one read (the kinds of a slice run concurrently and share it in L2; ncu: 7.0 GB read for
// 7.0 GB written at 24 cameras x 1 M points); the Schur pass is compute bound, HBM is idle
// otherwise.
// Block = 128 / C points at a time (small blocks: several per SM overlap their two phases):
// thread (camera t % C, point t / C) evaluates its item into a
// shared-memory tile that has the global layout, then the whole tile (contiguous in Yg) goes
// out as one TMA bulk store.
constexpr int MAKEY_THREADS = 128;
__global__ void __launch_bounds__(MAKEY_THREADS)
k_make_Y(const double* __restrict__ tab, const double* __restrict__ pts,
         const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
         const unsigned long long* __restrict__ mask, const double* __restrict__ Lz, long long P,
         int C, int rp, double* __restrict__ Yg) {
  extern __shared__ __align__(16) double s_dyn[];
  double* s_tab = s_dyn;
  double* tile = s_dyn + ((C * CAMTAB + 1) & ~1);          // [3 * PB][rp]
  const int t = threadIdx.x, PB = MAKEY_THREADS / C;
  load_tables_smem(tab, s_tab, C);
  __syncthreads();
  const int cam = t % C, pl = t / C;
  for (long long p0 = (long long)blockIdx.x * PB; p0 < P; p0 += (long long)gridDim.x * PB) {
    const int npts = (int)min((long long)PB, P - p0);
    if (pl < npts) {
      const long long p = p0 + pl;
      const unsigned long long m = mask[p];
      const bool live = (m >> cam) & 1ull;
      double w = 0.0;
      if (live) w = wgt ? wgt[(long long)obs_start[p] + __popcll(m & ((1ull << cam) - 1ull))] : 1.0;
      double X[3], li[9];
#pragma unroll
      for (int a = 0; a < 3; ++a) X[a] = pts[3 * p + a];
#pragma unroll
      for (int a = 0; a < 9; ++a) li[a] = Lz[p * 9 + a];
      double* row0 = tile + (size_t)3 * pl * rp;
      mma_produce(s_tab + cam * CAMTAB, X, li, w, live, row0 + cam * 12, rp);
      if (cam == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          double* o = row0 + (size_t)k * rp + C * 12;
          o[0] = li[6 + k];
          for (int e = 1; e < rp - C * 12; ++e) o[e] = 0.0;
        }
      }
    }
    // the tile is one contiguous range of Yg: a single TMA bulk store (cp.async.bulk shared ->
    // global) issued by one thread; the other blocks of the SM keep computing meanwhile
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (t == 0) {
      const unsigned src = (unsigned)__cvta_generic_to_shared(tile);
      const unsigned bytes = (unsigned)(3 * npts * rp * 8);
      double* dst = Yg + (size_t)p0 * 3 * rp;
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes)
                   : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");     // tile may be rewritten
    }
    __syncthreads();
  }
  if (t == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}

// Consumer body for one unit shape (NR x NC tiles, TRI: lower triangle): everything static,
// the DMMA stream is branch free.
template <int NR, int NC, bool TRI>
__device__ __forceinline__ void mma_consume(const MmaUnit& U, const double* s_dyn, size_t stage_doubles,
                                            int rp, int ksteps, long long nchunks, int nthreads,
                                            int bar_full, int bar_empty, int C, int lane,
                                            double* __restrict__ out, double* __restrict__ rout) {
  int offA[NR], offB[NC];
#pragma unroll
  for (int t = 0; t < NR; ++t) offA[t] = mma_row_offset(8 * (U.tr0 + t) + (lane >> 2), C) + (lane & 3) * rp;
#pragma unroll
  for (int u = 0; u < NC; ++u) offB[u] = mma_row_offset(8 * (U.tc0 + u) + (lane >> 2), C) + (lane & 3) * rp;
  double acc[NR][NC][2];
#pragma unroll
  for (int t = 0; t < NR; ++t)
#pragma unroll
    for (int u = 0; u < NC; ++u) acc[t][u][0] = acc[t][u][1] = 0.0;
  for (long long c = 0; c < nchunks; ++c) {
    const int st = (int)(c % SCHUR_STAGES);
    const double* s_Y = s_dyn + st * stage_doubles;
    nbar_sync(bar_full + st, nthreads);
#pragma unroll 1
    for (int ks = 0; ks < ksteps; ++ks) {
      const double* base = s_Y + (size_t)ks * 4 * rp;
      double a[NR], b[NC];
#pragma unroll
      for (int t = 0; t < NR; ++t) a[t] = base[offA[t]];
#pragma unroll
      for (int u = 0; u < NC; ++u) b[u] = base[offB[u]];
#pragma unroll
      for (int t = 0; t < NR; ++t)
#pragma unroll
        for (int u = 0; u < NC; ++u)
          if (!TRI || u <= t) dmma884(acc[t][u], a[t], b[u]);
    }
    nbar_arrive(bar_empty + st, nthreads);
  }
  // slice partial: every lower-triangle pair entry exactly once (same-camera blocks are stored
  // with both triangles: the mirror is written alongside)
  const int n = NCP * C;
#pragma unroll
  for (int t = 0; t < NR; ++t) {
    const int rho = 8 * (U.tr0 + t) + (lane >> 2);
    if (rho > n) continue;
#pragma unroll
    for (int u = 0; u < NC; ++u) {
      if (TRI && u > t) continue;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int sig = 8 * (U.tc0 + u) + 2 * (lane & 3) + e;
        if (sig >= n || sig > rho) continue;
        const double v = -acc[t][u][e];
        const int ck = sig / NCP, cb = sig % NCP;
        if (rho == n) { rout[ck * NCP + cb] = v; continue; }          // z row: reduced rhs
        const int cj = rho / NCP, ra = rho % NCP;
        double* blk = out + (size_t)(cj * (cj + 1) / 2 + ck) * 121;
        blk[ra * NCP + cb] = v;
        if (cj == ck && ra != cb) blk[cb * NCP + ra] = v;
      }
    }
  }
}

// part[slice][npairs*121 + 11 C]: - sum Y Y^T per pair block (11 x 11) and the reduced rhs.
// LAST = number of tile rows of the last group (compile time, so that every unit shape is).
// PRE: Y comes from k_make_Y (Yg), the producers only copy; otherwise they evaluate it in place.
template <int LAST, bool PRE>
__global__ void __launch_bounds__(MMA_THREADS, 1)
k_schur_mma(const double* __restrict__ Yg, const double* __restrict__ tab, const double* __restrict__ pts,
            const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
            const unsigned long long* __restrict__ mask, const double* __restrict__ Lz,
            long long P, long long N, int C, const MmaKind* __restrict__ kinds, int nslices,
            size_t part_stride, int npairs, double* __restrict__ part,
            long long* __restrict__ stats, const int* __restrict__ gate = nullptr /* non-null: run only if *gate */) {
  if (gate && *gate == 0) return;
  extern __shared__ __align__(16) double s_dyn[];
  const MmaKind& K = kinds[blockIdx.y];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int nthreads = 32 * (K.nactive + MMA_PROD_WARPS);   // barrier participants
  const int SP = K.sp, rp = K.rp;
  const size_t stage_doubles = (size_t)3 * SP * rp;
  double* s_tab = s_dyn + SCHUR_STAGES * stage_doubles;
  enum { BAR_FULL = 2, BAR_EMPTY = BAR_FULL + SCHUR_STAGES, BAR_PROD = BAR_EMPTY + SCHUR_STAGES };
  const long long t_start = clock64();

  const int slice = blockIdx.x;
  long long pa, pb;
  {
    const unsigned long long ta = (unsigned long long)N * slice / nslices;
    const unsigned long long tb = (unsigned long long)N * (slice + 1) / nslices;
    pa = (slice == 0) ? 0 : lower_bound_u32(obs_start, P, ta);
    pb = (slice == nslices - 1) ? P : lower_bound_u32(obs_start, P, tb);
  }
  const long long nchunks = (pb - pa + SP - 1) / SP;

  if (wid >= MMA_CONS_WARPS) {
    // ================================ producer warpgroup ================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 " MMA_PROD_REGS ";");
    const int ptid = tid - 32 * MMA_CONS_WARPS, nprod = 32 * MMA_PROD_WARPS;
    if (!PRE) {
      for (int i = ptid; i < C * CAMTAB; i += nprod) s_tab[i] = tab[i];
      nbar_sync(BAR_PROD, nprod);
    }
    const int total = SP * C;
    for (long long c = 0; c < nchunks + SCHUR_STAGES; ++c) {
      const int st = (int)(c % SCHUR_STAGES);
      if (c >= SCHUR_STAGES) nbar_sync(BAR_EMPTY + st, nthreads);
      if (c >= nchunks) continue;
      double* s_Y = s_dyn + st * stage_doubles;
      const long long q0 = pa + c * SP;
      if (PRE) {
        // contiguous rows of Yg -> ring stage (16-byte chunks); the tail of the last chunk is zeroed
        const int npc = (int)min((long long)SP, pb - q0);
        const int nch = 3 * npc * rp / 2, nall = 3 * SP * rp / 2;
        const double2* src = reinterpret_cast<const double2*>(Yg + (size_t)q0 * 3 * rp);
        double2* dst2 = reinterpret_cast<double2*>(s_Y);
        for (int i = ptid; i < nch; i += nprod) cp_async16(dst2 + i, src + i);
        for (int i = nch + ptid; i < nall; i += nprod) dst2[i] = make_double2(0.0, 0.0);
        asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
        __threadfence_block();
        nbar_arrive(BAR_FULL + st, nthreads);
        continue;
      }
      for (int idx = ptid; idx < total + SP; idx += nprod) {
        if (idx >= total) {   // the z row of point q (and the zero row behind it)
          const int q = idx - total;
          const long long p = q0 + q;
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            double* o = s_Y + (size_t)(3 * q + k) * rp + C * 12;
            o[0] = (p < pb) ? Lz[p * 9 + 6 + k] : 0.0;
            o[1] = 0.0;
          }
          continue;
        }
        const int q = idx / C, cam = idx - q * C;
        const long long p = q0 + q;
        double* Yk0 = s_Y + (size_t)3 * q * rp + cam * 12;
        if (p >= pb) {
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            double2* o = reinterpret_cast<double2*>(Yk0 + (size_t)k * rp);
#pragma unroll
            for (int e = 0; e < 6; ++e) o[e] = make_double2(0.0, 0.0);
          }
          continue;
        }
        const unsigned long long m = mask[p];
        const bool live = (m >> cam) & 1ull;
        double w = 0.0;
        if (live) w = wgt ? wgt[(long long)obs_start[p] + __popcll(m & ((1ull << cam) - 1ull))] : 1.0;
        double X[3], li[9];
#pragma unroll
        for (int a = 0; a < 3; ++a) X[a] = pts[3 * p + a];
#pragma unroll
        for (int a = 0; a < 9; ++a) li[a] = Lz[p * 9 + a];
        mma_produce(s_tab + cam * CAMTAB, X, li, w, live, Yk0, rp);
      }
      __threadfence_block();
      nbar_arrive(BAR_FULL + st, nthreads);
    }
    if (stats && ptid == 0) {
      long long* o = stats + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 4;
      o[2] = 0;
      o[3] = clock64() - t_start;
    }
    return;
  }

  // ================================ consumer warpgroups ================================
  asm volatile("setmaxnreg.inc.sync.aligned.u32 " MMA_CONS_REGS ";");
  const MmaUnit U = K.unit[wid];
  if (U.nr == 0) return;                             // idle warp slot of this kind
  double* out = part + (size_t)slice * part_stride;
  double* rout = out + (size_t)npairs * 121;
  const int ksteps = 3 * SP / 4;
#define MMA_CONSUME(NR, NC, TRI)                                                                   \
  mma_consume<NR, NC, TRI>(U, s_dyn, stage_doubles, rp, ksteps, nchunks, nthreads, BAR_FULL, BAR_EMPTY, \
                           C, lane, out, rout)
  if (U.nr == 6)                { if (U.tri) MMA_CONSUME(6, 6, true); else MMA_CONSUME(6, 6, false); }
  else if (U.nr == 3 && !U.tri) MMA_CONSUME(3, 6, false);            // half of a split 6 x 6 unit
  else                          { if (U.tri) MMA_CONSUME(LAST, LAST, true); else MMA_CONSUME(LAST, 6, false); }
#undef MMA_CONSUME
  if (stats && lane == 0 && wid == 0) {
    long long* o = stats + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 4;
    o[0] = 0;
    o[1] = clock64() - t_start;
  }
}

// ---- camera blocks U_c = sum_obs Jc^T Jc ------------------------------------------------
// thread = (camera c = t % C fixed, point lane t / C); 66 register accumulators (upper
// triangle); block partial -> part[block][C * 66].
constexpr int CAMN_VALS = 66;
__global__ void __launch_bounds__(256, 1)
k_cam_normal(const double* __restrict__ tab, const double* __restrict__ pts,
             const double* __restrict__ wgt, const uint32_t* __restrict__ obs_start,
             const unsigned long long* __restrict__ mask, long long P, int C, int PB,
             double* __restrict__ part) {
  extern __shared__ double s_dyn[];
  double* s_tab = s_dyn;                                   // C * CAMTAB
  double* s_red = s_dyn + ((C * CAMTAB + 1) & ~1);         // PB * C  (one value at a time)
  const int t = threadIdx.x;
  load_tables_smem(tab, s_tab, C);
  __syncthreads();
  const int c = t % C, pl = t / C;
  const bool worker = pl < PB;
  double acc[CAMN_VALS];
#pragma unroll
  for (int i = 0; i < CAMN_VALS; ++i) acc[i] = 0.0;
  if (worker) {
    for (long long p = (long long)blockIdx.x * PB + pl; p < P; p += (long long)gridDim.x * PB) {
      const unsigned long long m = mask[p];
      if (!((m >> c) & 1ull)) continue;
      const double w = wgt ? wgt[(long long)obs_start[p] + __popcll(m & ((1ull << c) - 1ull))] : 1.0;
      ObsLin L;
      obs_linearize<false>(s_tab + c * CAMTAB, pts[3 * p], pts[3 * p + 1], pts[3 * p + 2], 0.0, 0.0, w, L);
      double J0[11], J1[11];
#pragma unroll
      for (int a = 0; a < 9; ++a) { J0[a] = L.Jc[0][a]; J1[a] = L.Jc[1][a]; }
      J0[9] = w; J0[10] = 0.0; J1[9] = 0.0; J1[10] = w;
      int idx = 0;
#pragma unroll
      for (int a = 0; a < 11; ++a)
#pragma unroll
        for (int b = a; b < 11; ++b, ++idx) acc[idx] = fma(J0[a], J0[b], fma(J1[a], J1[b], acc[idx]));
    }
  }
  // reduce over the PB point lanes of each camera (fixed order)
  double* out = part + (size_t)blockIdx.x * C * CAMN_VALS;
#pragma unroll
  for (int i = 0; i < CAMN_VALS; ++i) {
    __syncthreads();
    if (worker) s_red[pl * C + c] = acc[i];
    __syncthreads();
    if (t < C) {
      double s = 0.0;
      for (int q = 0; q < PB; ++q) s += s_red[q * C + t];
      out[t * CAMN_VALS + i] = s;
    }
  }
}

// Sred diagonal pair blocks += U (symmetric expansion of the 66 upper-triangle values)
__global__ void k_add_cam_blocks(const double* __restrict__ U, int C, double* __restrict__ Sred) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C * 121) return;
  const int c = i / 121, e = i % 121, a = e / NCP, b = e % NCP;
  const int lo = a < b ? a : b, hi = a < b ? b : a;
  const int idx = lo * NCP - lo * (lo - 1) / 2 + (hi - lo);
  Sred[(size_t)(c * (c + 1) / 2 + c) * 121 + e] += U[c * CAMN_VALS + idx];
}

}  // namespace lcba
