// Reduced camera system on the 5th-generation tensor cores: the SYRK  - sum_p [Y; z][Y; z]^T  through
// an error-free integer split ("Ozaki scheme"), tcgen05.mma kind::i8 with int32 accumulators in TMEM.
// Prototype, measurements and the accuracy model: tools/ozaki_syrk.cu, profiles/r02_ozaki.txt.
//
//   y_rk = 2^e_r * sum_{i<6} d_i(r,k) 2^-8(i+1)     d_i: balanced base-256 digits (int8), e_r from max_k |y_rk|
//   (Y Y^T)_rc = 2^(e_r+e_c) * sum_{i+j<=6} 2^-8(i+j+2) (D_i D_j^T)_rc       D_i D_j^T exact in int32
// 48 bits per entry relative to the row maximum; the 26 digit products kept include every coherent
// term (i = j) down to 2^-64: FP64-grade (numpy model on the oracle's Y: 1e-15 of max|S|).
//
// Passes (all in this file):
//   k_i8_rowmax   : max |Y| per matrix row (thread = fixed camera, 11 running maxima in registers)
//   k_i8_rowexp   : e_r
//   k_i8_make     : Y in FP64 -> 48-bit integers -> digit planes in HBM, laid out exactly as the UMMA
//                   shared-memory operand (K-major, no swizzle, 8 x 16-byte core matrices):
//                   [K block of 64 kappa = 21 points + 1 zero][slice][row group of 8][k-step 2][k half 2][8][16]
//   k_i8_syrk     : one CTA = one output tile (128 rows x <= 64 columns, the 7 anti-diagonals d = i + j
//                   side by side in TMEM) x a range of K blocks; warps 0-3 epilogue (TMEM -> FP64 registers
//                   before an int32 can overflow), warp 4 producer (up to three TMA tensor loads per K block =
//                   2 k-steps: all six slices of A (4-D, or 5-D for two row ranges), B1, B2), warp 5 MMA
//                   issuer (elect.sync, compile-time MMA plan: slice i of the rows against slices 0..6-i of
//                   the columns in ONE instruction, N <= 256, A kept in the collector, widest last); tiles
//                   from the strip or the cover plan, CTAs per tile weighted
//                   by the measured cost of a K block, K blocks dealt K-major in chunks so that all tiles read a
//                   K block at about the same time, a progress window between the CTAs (i8_deal)
//   k_i8_gather   : per-CTA partials -> the pair-block layout of Sred (fixed order, no atomics)
//   k_i8_check    : resolution guard: rows whose maximum lies far above their Schur diagonal hand the pass to
//                   the DMMA kernel (k_schur_mma, gated) and k_i8_fallback_finish
#pragma once
#include <cuda.h>
#include <algorithm>
#include <vector>
#include "common.cuh"
#include "schur_mma.cuh"

namespace lcba {

constexpr int I8_NS = 6;                  // digits per entry
constexpr int I8_DMAX = 6;                // anti-diagonals kept: i + j <= 6
constexpr int I8_ND = I8_DMAX + 1;
constexpr int I8_PTS = 21;                // points per K block (63 kappa + 1 zero column)
constexpr int I8_STAGES = 3;              // ring stages of one K block (72 KB each)
constexpr int I8_FLUSH = 224;             // K blocks between TMEM flushes: 6 pairs * 64 * 128^2 * 224 < 2^31
constexpr int I8_THREADS = 192;
constexpr int I8_RG_BYTES = 512;          // one row group of one slice of one K block
constexpr int I8_GROUP_CAMS = 8;          // cameras per k_i8_make block: 88 rows = 11 row groups exactly
constexpr int I8_GROUP_RG = 13;           // row groups of the last group at most: 8 cameras + z + even padding
constexpr int I8_GROUP_ROWS = I8_GROUP_RG * 8;
constexpr int I8_KC = 8;                  // K blocks per chunk of the K-major schedule (0.8 MB of planes at 24 cameras)
constexpr size_t I8_WINDOW_BYTES = 32u << 20;   // planes between the slowest and the fastest CTA of k_i8_syrk
constexpr int I8_POLL_CAP = 2048;         // window polls after which a CTA stops waiting for the others

// One CTA of k_i8_syrk: rows = row groups [m_rg0, m_rg0 + m_nrg) and, optionally, a second range
// [m2_rg0, +m2_nrg) stacked below them (the A operand, <= 16 row groups in all), columns = block 1
// [n_rg0, +n_nrg) and, optionally, block 2 [n2_rg0, +n2_nrg): the few rows left over behind the last full
// 128-row tile of the strip plan, handled as COLUMNS (the tile entry is S[column][row]); n_nrg + n2_nrg <= 8.
// In the partial tile [128][64] block 1 occupies columns [0, 8 n_nrg), block 2 the LAST 8 n2_nrg columns.
// The K blocks of a CTA: positions [kb0, kb1) of its tile's K order, i.e. the K blocks
// kfirst + (i / kc) kstride + i % kc for i < kb1 - kb0 (runs of kc K blocks, kstride apart).
struct I8Work {
  int m_rg0, m_nrg, m2_rg0, m2_nrg, n_rg0, n_nrg, n2_rg0, n2_nrg;
  int kb0, kb1;
  int map_a, map_b1, map_b2;              // tensor-map index of the three operand loads
  int kfirst, kc, kstride;
};
// TMA tensor maps over the digit planes, one per (box height, range distance) that the plan uses.
// delta = 0: a 4-D tensor (128 u32 = one 512-byte row group, NRG row groups, 6 digits, K blocks); a box of
// (128, h, 6, 1) lands in shared memory as [digit][h row groups][512 B] = the UMMA operand of all six digits
// in ONE instruction.
// delta > 0: the two-range A operand, a 5-D tensor (128 u32, NRG - delta row groups, 2 ranges delta row
// groups apart, 6 digits, K blocks); a box of (128, h, 2, 6, 1) lands as [digit][2 h row groups][512 B], the same
// layout as one range of 2 h row groups.
constexpr int I8_MAX_MAPS = 16;
struct alignas(64) I8Maps { CUtensorMap m[I8_MAX_MAPS]; };
struct I8Tile { int m_rg0, m_nrg, m2_rg0, m2_nrg, n_rg0, n_nrg, n2_rg0, n2_nrg, w0, nw; };

struct I8Plan {
  int C = 0, R = 0, NRG = 0;
  long long nkb = 0;
  int map_heights[I8_MAX_MAPS] = {};                   // box heights (row groups per range) of the tensor maps
  int map_delta[I8_MAX_MAPS] = {};                     // 0: one range; > 0: two ranges this many row groups apart
  int nmaps = 0;                                       // > I8_MAX_MAPS: too many shapes, i8_encode_maps fails
  bool cover = false;                                  // made by make_i8_cover_plan
  bool kmajor = true;                                  // K-major schedule (else one contiguous K range per CTA)
  int window = 0;                                      // K-major: K blocks a CTA may run ahead of the slowest
  double model_cycles = 0.0;                           // slowest CTA in the cost model (MMA-warp cycles)
  std::vector<I8Tile> tiles;
  std::vector<I8Work> work;
  size_t plane_bytes = 0, smem_bytes = 0;
};

// Cost of one K block of a tile, in cycles of the MMA warp (measured per tile kind with LCBA_SCHUR_STATS=1,
// tools/i8_stats.py, ring24 x 1 M): a fixed part (stage hand-over, waiting for operands) + one part per column
// block that grows with its width -- narrow instructions are far from free: a 16-column block costs half a
// 48-column one.  The row ranges of A do not enter: M is 128 in every instruction.
inline double i8_block_cost(int nrg) {
  return nrg <= 0 ? 0.0 : (nrg <= 2 ? 592.0 : (nrg <= 4 ? 812.0 : (nrg <= 6 ? 1181.0 : 1550.0)));
}
inline double i8_tile_cost(const I8Tile& t) { return 507.0 + i8_block_cost(t.n_nrg) + i8_block_cost(t.n2_nrg); }

// CTAs per tile: one CTA per SM in total, dealt so that the slowest tile finishes as early as possible
// (greedy over the cost model; the first version gave every main tile the same number of ranges: the tile that
// carries a second column block was 13 % slower than the rest and set the kernel's time).  The K blocks of a
// tile's n CTAs:
//   - range schedule (kmajor = false): CTA q takes the contiguous range [nkb q / n, nkb (q + 1) / n).  CTAs of
//     tiles with different n read different K blocks at any moment, so only tiles with the same n share their
//     operands through L2 (ring24 x 1 M: 13.9 GB of DRAM reads for 5.0 GB of planes, strip plan);
//   - K-major schedule: the K blocks form chunks of kc = I8_KC; CTA q takes the chunks j = q mod n in
//     increasing j.  n is roughly proportional to a tile's cost per K block, so every tile sweeps K at about
//     the same rate and all tiles read a chunk at about the same time; k_i8_syrk's window bounds the drift
//     that the rounding of the deal leaves (up to 4.5 % at 24 cameras: 2100 K blocks by the end of a launch).
// Fills pl.work, the tensor-map shapes, the buffer sizes, the window and the model's slowest-CTA cycles.
inline void i8_deal(I8Plan& pl, int sm_count) {
  std::vector<double> cost(pl.tiles.size());
  std::vector<long long> nr(pl.tiles.size(), 1);
  for (size_t ti = 0; ti < pl.tiles.size(); ++ti) cost[ti] = i8_tile_cost(pl.tiles[ti]);
  for (long long left = (long long)sm_count - (long long)pl.tiles.size(); left > 0; --left) {
    size_t worst = 0;
    double tw = -1.0;
    for (size_t ti = 0; ti < pl.tiles.size(); ++ti) {
      const double tt = nr[ti] < pl.nkb ? cost[ti] / (double)nr[ti] : -1.0;
      if (tt > tw) { tw = tt; worst = ti; }
    }
    if (tw < 0.0) break;                                    // every tile already has one CTA per K block
    ++nr[worst];
  }
  pl.model_cycles = 0.0;
  long long spread = 0;                                     // K-major: K blocks between a tile's first and last CTA
  for (size_t ti = 0; ti < pl.tiles.size(); ++ti) {
    I8Tile& t = pl.tiles[ti];
    const long long n = std::min<long long>(nr[ti], pl.nkb);
    t.w0 = (int)pl.work.size();
    t.nw = (int)n;
    auto map_of = [&](int h, int delta) {
      if (h == 0) return 0;
      for (int i = 0; i < pl.nmaps && i < I8_MAX_MAPS; ++i)
        if (pl.map_heights[i] == h && pl.map_delta[i] == delta) return i;
      if (pl.nmaps < I8_MAX_MAPS) { pl.map_heights[pl.nmaps] = h; pl.map_delta[pl.nmaps] = delta; }
      return pl.nmaps++;
    };
    const int ma = map_of(t.m_nrg, t.m2_nrg > 0 ? t.m2_rg0 - t.m_rg0 : 0), mb1 = map_of(t.n_nrg, 0), mb2 = map_of(t.n2_nrg, 0);
    // kc <= nkb / n: every CTA gets at least one chunk
    const long long kc = pl.kmajor ? std::max(1LL, std::min<long long>(I8_KC, pl.nkb / n)) : 0;
    const long long nch = pl.kmajor ? (pl.nkb + kc - 1) / kc : 0;
    long long pos = 0, most = 0;
    for (long long q = 0; q < n; ++q) {
      I8Work w{t.m_rg0, t.m_nrg, t.m2_rg0, t.m2_nrg, t.n_rg0, t.n_nrg, t.n2_rg0, t.n2_nrg, 0, 0, ma, mb1, mb2, 0, 0, 0};
      long long cnt;
      if (pl.kmajor) {
        cnt = ((nch - 1 - q) / n + 1) * kc - ((nch - 1) % n == q ? nch * kc - pl.nkb : 0);   // the last chunk may be short
        w.kfirst = (int)(q * kc);
        w.kc = (int)kc;
        w.kstride = (int)(n * kc);
      } else {
        cnt = pl.nkb * (q + 1) / n - pl.nkb * q / n;
        w.kfirst = (int)(pl.nkb * q / n);
        w.kc = (int)std::max(1LL, cnt);
      }
      w.kb0 = (int)pos;
      w.kb1 = (int)(pos + cnt);
      pos += cnt;
      most = std::max(most, cnt);
      pl.work.push_back(w);
    }
    pl.model_cycles = std::max(pl.model_cycles, cost[ti] * (double)most);
    spread = std::max(spread, n * kc);
  }
  // the window: about I8_WINDOW_BYTES of planes, and at least twice the spread of the CTAs of one tile, which
  // are that far apart by construction
  const long long kb_bytes = (long long)I8_NS * pl.NRG * I8_RG_BYTES;
  pl.window = pl.kmajor ? (int)std::min(pl.nkb, std::max((long long)(I8_WINDOW_BYTES / kb_bytes), 2 * spread)) : 0;
  pl.plane_bytes = (size_t)pl.nkb * I8_NS * pl.NRG * I8_RG_BYTES;
  pl.smem_bytes = (size_t)I8_STAGES * I8_NS * (16 + 8) * I8_RG_BYTES + 1024;
}

inline I8Plan i8_plan_base(int C, long long P, bool kmajor) {
  I8Plan pl;
  pl.kmajor = kmajor;
  pl.C = C;
  pl.R = NCP * C + 1;
  pl.NRG = (pl.R + 7) / 8;
  pl.NRG += pl.NRG & 1;                                   // MMA N is a multiple of 16
  pl.nkb = (P + I8_PTS - 1) / I8_PTS;
  return pl;
}

// The strip plan.  Row tiles of 16 row groups (128 rows), each with its column tiles up to and including the
// diagonal block, which is computed as a square (k_i8_gather drops its upper half).  When the last row tile
// would hold <= 4 row groups (24 cameras: 34 = 16 + 16 + 2) those rows are not given a 128-row tile of their
// own: they ride as column block 2 of ONE tile of every full row tile (the operand rows A are the same, only
// 1-2 KB of extra B per K block are loaded) plus a small corner tile; the column tiles are then
// 8 - last row groups wide so that block 1 + block 2 <= 64 columns (7 anti-diagonals x 64 = 448 TMEM columns).
// (First version: separate 16-column tiles with their own K ranges streamed K positions nobody else was
// reading: 40 % of the kernel's DRAM traffic for 11 % of its work, ncu r02.)
inline I8Plan make_i8_plan(int C, long long P, int sm_count, bool kmajor = true) {
  I8Plan pl = i8_plan_base(C, P, kmajor);
  const int NRG = pl.NRG;
  const int nmt = (NRG + 15) / 16;
  const int last_m = NRG - 16 * (nmt - 1);
  const bool fold = nmt > 1 && last_m <= 4;
  const int nfull = fold ? nmt - 1 : nmt;
  const int col_w = fold ? 8 - last_m : 8;
  const int c0 = 16 * (nmt - 1);
  for (int mt = 0; mt < nfull; ++mt) {
    const int m0 = 16 * mt, mn = std::min(16, NRG - m0);
    for (int n0 = 0; n0 < m0 + mn; n0 += col_w) {
      const int nn = std::min(col_w, m0 + mn - n0);
      const bool last = n0 + col_w >= m0 + mn;
      I8Tile t{m0, mn, 0, 0, n0, nn, fold && last ? c0 : 0, fold && last ? last_m : 0, 0, 0};
      pl.tiles.push_back(t);
    }
  }
  if (fold) {
    I8Tile t{c0, last_m, 0, 0, c0, last_m, 0, 0, 0, 0};  // the corner: left-over rows x left-over rows
    pl.tiles.push_back(t);
  }
  i8_deal(pl, sm_count);
  return pl;
}

// The cover plan: only full 128 x 64 tiles where the strip plan computes square diagonal blocks and folds.
// The row groups form G groups of 8 (g = row groups [8g, 8g + 8)) and a ragged rest E of NRG - 8G < 8 row
// groups.  A tile (I, J) has the column group J (<= 8 row groups) and up to two row groups I (the two
// ranges of A, 8 row groups each); S is symmetric, so a tile serves either orientation:
//   - I = {x, z}, J = z: the triangle of z and the block x-z;  I = {x, y}, J = z: the blocks x-z and y-z.
// Give every cross pair {x, z} of groups a column group (an orientation) so that each group z has an odd
// number of pairs pointing to it: its own triangle and those pairs then fill whole tiles.  Start from
// "pair {a, b}, a < b, points to b" (indegree of z = z) and flip the pair between two groups of the wrong
// parity; at most one group stays even when G (G - 1) / 2 and G differ in parity.  E stays a column block
// (<= 48 columns): its triangle rides with the last group (one contiguous range), the other groups go two at a
// time.  k_i8_gather keeps each entry once: inside I and J both (the square of z) only rho >= sig.
// 24 cameras (NRG = 34, G = 4): 8 tiles, 13 582 model cycles per K block against 16 517 for the strip plan.
inline I8Plan make_i8_cover_plan(int C, long long P, int sm_count, bool kmajor = true) {
  I8Plan pl = i8_plan_base(C, P, kmajor);
  pl.cover = true;
  const int G = pl.NRG / 8, r = pl.NRG - 8 * G;
  std::vector<std::vector<int>> to(G);                  // to[z]: the groups x whose pair {x, z} has columns z
  for (int b = 0; b < G; ++b)
    for (int a = 0; a < b; ++a) to[b].push_back(a);
  std::vector<int> even;
  for (int z = 0; z < G; ++z) if (to[z].size() % 2 == 0) even.push_back(z);
  for (size_t k = 0; k + 1 < even.size(); k += 2) {     // flip {u, v}, u < v: it pointed to v, now to u
    const int u = even[k], v = even[k + 1];
    to[v].erase(std::find(to[v].begin(), to[v].end(), u));
    to[u].push_back(v);
  }
  auto tile = [&](int x, int y, int j0, int jn) {       // rows: group x (and group y >= 0), columns [j0, j0 + jn)
    int a = std::min(x, y < 0 ? x : y), b = std::max(x, y);
    I8Tile t{8 * a, 8, 0, 0, j0, jn, 0, 0, 0, 0};
    if (y >= 0 && b == a + 1) t.m_nrg = 16;             // adjacent groups: one range of 16
    else if (y >= 0) { t.m2_rg0 = 8 * b; t.m2_nrg = 8; }
    pl.tiles.push_back(t);
  };
  for (int z = 0; z < G; ++z) {
    std::vector<int> items(1, z);                       // z's own triangle, then the pairs pointing to z
    items.insert(items.end(), to[z].begin(), to[z].end());
    std::sort(items.begin() + 1, items.end());
    for (size_t k = 0; k < items.size(); k += 2) tile(items[k], k + 1 < items.size() ? items[k + 1] : -1, 8 * z, 8);
  }
  if (r > 0) {
    // E's triangle with the last group: rows [8 (G - 1), NRG) in one range
    if (G > 0) pl.tiles.push_back(I8Tile{8 * (G - 1), 8 + r, 0, 0, 8 * G, r, 0, 0, 0, 0});
    else pl.tiles.push_back(I8Tile{0, r, 0, 0, 0, r, 0, 0, 0, 0});
    for (int x = 0; x + 1 < G; x += 2) tile(x, x + 2 < G ? x + 1 : -1, 8 * G, r);
  }
  i8_deal(pl, sm_count);
  return pl;
}

// The plan k_i8_syrk runs: the cover plan where the cost model puts its slowest CTA below the strip plan's.
// which: 0 = by the model, 1 = strip, 2 = cover (LCBA_I8_PLAN); kmajor: the schedule (LCBA_I8_SCHED=range: false).
inline I8Plan make_i8_best_plan(int C, long long P, int sm_count, int which, bool kmajor = true) {
  if (which == 1) return make_i8_plan(C, P, sm_count, kmajor);
  I8Plan cv = make_i8_cover_plan(C, P, sm_count, kmajor);
  if (which == 2) return cv;
  I8Plan st = make_i8_plan(C, P, sm_count, kmajor);
  return cv.model_cycles < st.model_cycles ? cv : st;
}

// int8 ops (1 MAC = 2) one k_i8_syrk launch of a plan issues: 26 digit products of 128 rows x the plan's
// columns x 64 kappa per K block.
inline double i8_executed_ops(const I8Plan& pl) {
  long long cols = 0;
  for (const I8Tile& t : pl.tiles) cols += 8 * (t.n_nrg + t.n2_nrg);
  return 26.0 * 2.0 * 128.0 * (double)cols * 64.0 * (double)pl.nkb;
}

// Encode the tensor maps of a plan over `planes` (host).  Returns false when the driver entry point is
// missing, an encode fails or the plan has more shapes than I8_MAX_MAPS (the plans need at most 16).
inline bool i8_encode_maps(const I8Plan& pl, void* planes, I8Maps* out) {
  if (pl.nmaps <= 0 || pl.nmaps > I8_MAX_MAPS) return false;
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) {
    cudaGetLastError();
    return false;
  }
  const cuuint64_t rg = I8_RG_BYTES, slice = (cuuint64_t)pl.NRG * I8_RG_BYTES, blk = (cuuint64_t)I8_NS * slice;
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  memset(out, 0, sizeof(*out));
  for (int i = 0; i < pl.nmaps; ++i) {
    const cuuint32_t h = (cuuint32_t)pl.map_heights[i];
    CUresult r;
    if (pl.map_delta[i] == 0) {
      const cuuint64_t gdim[4] = {128, (cuuint64_t)pl.NRG, (cuuint64_t)I8_NS, (cuuint64_t)pl.nkb};
      const cuuint64_t gstr[3] = {rg, slice, blk};
      const cuuint32_t box[4] = {128, h, (cuuint32_t)I8_NS, 1};
      r = ((EncodeFn)fn)(&out->m[i], CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, planes, gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
      // the row-group extent ends delta before NRG, so that the second range of any box stays inside the slice
      const cuuint64_t gdim[5] = {128, (cuuint64_t)(pl.NRG - pl.map_delta[i]), 2, (cuuint64_t)I8_NS, (cuuint64_t)pl.nkb};
      const cuuint64_t gstr[4] = {rg, (cuuint64_t)pl.map_delta[i] * rg, slice, blk};
      const cuuint32_t box[5] = {128, h, 2, (cuuint32_t)I8_NS, 1};
      r = ((EncodeFn)fn)(&out->m[i], CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, planes, gdim, gstr, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r != CUDA_SUCCESS) return false;
  }
  return true;
}

// ------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ void i8_tma_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}
__device__ __forceinline__ void i8_tma_5d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t i8_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void i8_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void i8_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void i8_mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a protocol error must end in an error code, never in a hung GPU.
template <bool BACKOFF>
__device__ __forceinline__ void i8_mbar_wait(uint32_t bar, uint32_t parity, int* fail) {
  const long long t0 = clock64();
  while (true) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) return;
    if (BACKOFF) __nanosleep(128);      // waiting warps must not compete with the MMA issuer for issue slots
    if (clock64() - t0 > 6000000000LL) { atomicOr(fail, 4); asm volatile("trap;"); }
  }
}
// COLL: what happens to the A operand in the tensor core's collector: 0 nothing kept (the default), 1 ::fill (read
// from shared memory and kept), 2 ::use (taken from the collector, kept), 3 ::lastuse (taken from the collector)
template <int COLL>
__device__ __forceinline__ void i8_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
#define I8_MMA_ASM(Q)                                                                                      \
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"                                          \
               "tcgen05.mma.cta_group::1.kind::i8" Q " [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"         \
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc), "r"(0u) : "memory")
  if (COLL == 1) I8_MMA_ASM(".collector::a::fill");
  else if (COLL == 2) I8_MMA_ASM(".collector::a::use");
  else if (COLL == 3) I8_MMA_ASM(".collector::a::lastuse");
  else I8_MMA_ASM("");
#undef I8_MMA_ASM
}
__device__ __forceinline__ void i8_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool i8_elect_one() {
  uint32_t p;
  asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(p));
  return p != 0;
}
__device__ __forceinline__ void i8_tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr) : "memory");
}

// ------------------------------------------------------------------------------ Y of one (point, camera)
// y[k][a], a < 11: the 11 rows of the camera for kappa = k (same arithmetic as mma_produce)
__device__ __forceinline__ void i8_item_values(const double* __restrict__ T, const double (&X)[3],
                                               const double (&li)[9], double w, bool live, double (&y)[3][NCP]) {
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
#pragma unroll
    for (int a = 0; a < 9; ++a) y[k][a] = fma(L.Jc[0][a], Q[0][k], L.Jc[1][a] * Q[1][k]);
    y[k][9] = w * Q[0][k];
    y[k][10] = w * Q[1][k];
  }
}

// FP32 twin of i8_item_values for the row maxima only (an exponent needs 1e-4, not 1e-16; FP32 runs
// at twice the FP64 rate with half the registers).  m[a] = max(m[a], max_k |y[k][a]|).
__device__ __forceinline__ void i8_item_absmax_f32(const float* __restrict__ T, float X, float Y, float Z,
                                                   const float (&li)[6], float w, float (&m)[NCP]) {
  const float* R = T + CT_R;
  const float xc = fmaf(R[0], X, fmaf(R[1], Y, fmaf(R[2], Z, T[3])));
  const float yc = fmaf(R[3], X, fmaf(R[4], Y, fmaf(R[5], Z, T[4])));
  const float zc = fmaf(R[6], X, fmaf(R[7], Y, fmaf(R[8], Z, T[5])));
  const float iz = 1.0f / zc;
  const float x = xc * iz, y = yc * iz;
  const float n = x * x + y * y;
  const float f = T[6], k1 = T[7], k2 = T[8];
  const float d = 1.0f + n * (k1 + k2 * n);
  const float dp = k1 + 2.0f * k2 * n;
  const float wf = w * f;
  const float e00 = wf * (d + 2.0f * x * x * dp), e01 = wf * (2.0f * x * y * dp), e11 = wf * (d + 2.0f * y * y * dp);
  float G[2][3] = {{e00 * iz, e01 * iz, -(e00 * x + e01 * y) * iz}, {e01 * iz, e11 * iz, -(e01 * x + e11 * y) * iz}};
  float Jc[2][9], Jp[2][3];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) Jp[i][j] = fmaf(G[i][0], R[j], fmaf(G[i][1], R[3 + j], G[i][2] * R[6 + j]));
  const float* Jr = T + CT_JR;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float c0 = Jr[k], c1 = Jr[3 + k], c2 = Jr[6 + k];
    const float m0 = fmaf(Y, c2, -Z * c1), m1 = fmaf(Z, c0, -X * c2), m2 = fmaf(X, c1, -Y * c0);
    Jc[0][k] = -fmaf(Jp[0][0], m0, fmaf(Jp[0][1], m1, Jp[0][2] * m2));
    Jc[1][k] = -fmaf(Jp[1][0], m0, fmaf(Jp[1][1], m1, Jp[1][2] * m2));
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) { Jc[i][3] = G[i][0]; Jc[i][4] = G[i][1]; Jc[i][5] = G[i][2]; }
  const float wd = w * d, wfn = wf * n, wfn2 = wfn * n;
  Jc[0][6] = wd * x;   Jc[1][6] = wd * y;
  Jc[0][7] = wfn * x;  Jc[1][7] = wfn * y;
  Jc[0][8] = wfn2 * x; Jc[1][8] = wfn2 * y;
  float Q[2][3];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    Q[i][0] = Jp[i][0] * li[0];
    Q[i][1] = fmaf(Jp[i][0], li[1], Jp[i][1] * li[2]);
    Q[i][2] = fmaf(Jp[i][0], li[3], fmaf(Jp[i][1], li[4], Jp[i][2] * li[5]));
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
#pragma unroll
    for (int a = 0; a < 9; ++a) m[a] = fmaxf(m[a], fabsf(fmaf(Jc[0][a], Q[0][k], Jc[1][a] * Q[1][k])));
    m[9] = fmaxf(m[9], fabsf(w * Q[0][k]));
    m[10] = fmaxf(m[10], fabsf(w * Q[1][k]));
  }
}

// Work decomposition of k_i8_rowmax / k_i8_make: block = (K block kb, camera group g of 8 cameras);
// thread t < 21 * gc: point lane q = t / gc, camera g*8 + t % gc.  blockIdx.y = g, blockIdx.x strides kb.
// rmax_part[blockIdx.x][NRG * 8]
__global__ void __launch_bounds__(192, 4)
k_i8_rowmax(const double* __restrict__ tab, const double* __restrict__ pts, const double* __restrict__ wgt,
            const uint32_t* __restrict__ obs_start, const unsigned long long* __restrict__ mask,
            const double* __restrict__ Lz, long long P, int C, int RP, double* __restrict__ rmax_part) {
  extern __shared__ double s_dyn[];
  float* s_tab = reinterpret_cast<float*>(s_dyn);                 // 8 * CAMTAB floats
  float* s_red = s_tab + I8_GROUP_CAMS * CAMTAB;                  // 192
  const int t = threadIdx.x, g = blockIdx.y;
  const int c0 = g * I8_GROUP_CAMS, gc = min(I8_GROUP_CAMS, C - c0);
  for (int i = t; i < gc * CAMTAB; i += blockDim.x) s_tab[i] = (float)tab[c0 * CAMTAB + i];
  __syncthreads();
  const bool worker = t < I8_PTS * gc;
  const int q = worker ? t / gc : 0, cl = worker ? t % gc : 0, cam = c0 + cl;
  const bool zthread = (g == gridDim.y - 1) && t >= 168 && t < 168 + I8_PTS;      // z row: one thread per point lane
  float mx[NCP], mz = 0.0f;
#pragma unroll
  for (int a = 0; a < NCP; ++a) mx[a] = 0.0f;
  const long long nkb = (P + I8_PTS - 1) / I8_PTS;
  for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x) {
    if (worker) {
      const long long p = kb * I8_PTS + q;
      if (p < P) {
        const unsigned long long m = mask[p];
        if ((m >> cam) & 1ull) {
          const float w = wgt ? (float)wgt[(long long)obs_start[p] + __popcll(m & ((1ull << cam) - 1ull))] : 1.0f;
          float li[6];
#pragma unroll
          for (int a = 0; a < 6; ++a) li[a] = (float)Lz[p * 9 + a];
          i8_item_absmax_f32(s_tab + cl * CAMTAB, (float)pts[3 * p], (float)pts[3 * p + 1], (float)pts[3 * p + 2], li, w, mx);
        }
      }
    }
    if (zthread) {
      const long long p = kb * I8_PTS + (t - 168);
      if (p < P) mz = fmaxf(mz, fmaxf(fabsf((float)Lz[p * 9 + 6]), fmaxf(fabsf((float)Lz[p * 9 + 7]), fabsf((float)Lz[p * 9 + 8]))));
    }
  }
  // block partial: max over the 21 point lanes of each camera (order irrelevant for a maximum)
  double* out = rmax_part + (size_t)blockIdx.x * RP;
#pragma unroll
  for (int a = 0; a < NCP; ++a) {
    __syncthreads();
    s_red[t] = worker ? mx[a] : 0.0f;
    __syncthreads();
    if (t < gc) {
      float m = 0.0f;
      for (int qq = 0; qq < I8_PTS; ++qq) m = fmaxf(m, s_red[qq * gc + t]);
      out[(c0 + t) * NCP + a] = (double)m;
    }
  }
  if (g == gridDim.y - 1) {
    __syncthreads();
    s_red[t] = zthread ? mz : 0.0f;
    __syncthreads();
    if (t == 0) {
      float m = 0.0f;
      for (int i = 168; i < 168 + I8_PTS; ++i) m = fmaxf(m, s_red[i]);
      out[NCP * C] = (double)m;
    }
  }
}

// e_row[r]: |y| 2^-e < 0.25 (two bits of headroom: the top digit stays below 65); rows without data: 0.
// m_row[r]: the row maximum itself (for k_i8_check)
__global__ void k_i8_rowexp(const double* __restrict__ rmax_part, int nb, int R, int RP, int* __restrict__ e_row,
                            double* __restrict__ m_row) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= RP) return;
  double m = 0.0;
  if (r < R) for (int b = 0; b < nb; ++b) m = fmax(m, rmax_part[(size_t)b * RP + r]);
  int e = 0;
  if (m > 0.0 && m < 1e300) { frexp(m * 1.001, &e); e += 2; }    // maxima come from an FP32 evaluation: 1e-3 of slack
  e_row[r] = e;
  m_row[r] = m;
}

// 48-bit integer T -> the 6 balanced digits as the bytes of one word: digit i (0 = most significant)
// is byte (5 - i) of (T + 0x808080808080) ^ 0x808080808080  (adding 128 to every base-256 digit makes
// them unsigned, so they are the bytes of the sum; ^ 0x80 maps d + 128 back to int8 d).
__device__ __forceinline__ unsigned long long i8_encode(double v, double scale) {
  const long long T = __double2ll_rn(v * scale);
  return (unsigned long long)(T + 0x808080808080LL) ^ 0x808080808080ULL;
}

// i8_encode without the FP64 -> int64 conversion (F2I.S64.F64 issues at a fraction of the DFMA rate): for
// finite |x| < 2^51, x + 1.5 * 2^52 rounded to nearest even holds rint(x) + 2^51 in its 52 fraction bits, so its
// low 48 bits, the only ones the planes use, are those of __double2ll_rn(x) (here |x| < 2^47).  v * scale is exact
// (scale is a power of two), so one FMA rounds exactly like the product followed by the addition.  A non-finite
// Y gives other bytes than i8_encode (whose conversion saturates); both are meaningless, and k_i8_rowexp's fmax
// passes a NaN by in either case.
__device__ __forceinline__ unsigned long long i8_encode_fma(double v, double scale) {
  const unsigned long long T = (unsigned long long)__double_as_longlong(fma(v, scale, 6755399441055744.0));
  return (T + 0x808080808080ULL) ^ 0x808080808080ULL;
}

constexpr int I8_VAL_LD = 65;             // row stride (64-bit words) of the staging tile: conflict-free both ways
inline size_t i8_make_ref_smem_bytes() {
  return (size_t)I8_GROUP_CAMS * CAMTAB * 8 + (size_t)I8_GROUP_ROWS * 8 + (size_t)I8_GROUP_ROWS * I8_VAL_LD * 8;
}

// The first k_i8_make, kept as the reference the tests compare k_i8_make's planes with (lcba_debug_i8_make).
// planes[((kb * NS + i) * NRG + rg) * 512 + a * 256 + kh * 128 + r8 * 16 + kbyte], kappa_local = 32 a + 16 kh + kbyte.
// block (kb stride, g).  Phase 1: thread = (point lane, camera) evaluates Y in FP64 and writes the 33
// encoded integers to the staging tile [row][kappa] (one 64-bit store each).  Phase 2: a warp takes one
// (row group, k-step, k half): lane = (row r8, kappa quad) reads 4 integers, picks byte 5 - i of each with
// PRMT and stores one 32-bit word per slice: 128 contiguous bytes per warp and slice, straight to HBM.
__global__ void __launch_bounds__(192, 3)
k_i8_make_ref(const double* __restrict__ tab, const double* __restrict__ pts, const double* __restrict__ wgt,
          const uint32_t* __restrict__ obs_start, const unsigned long long* __restrict__ mask,
          const double* __restrict__ Lz, long long P, int C, int NRG, const int* __restrict__ e_row,
          unsigned char* __restrict__ planes) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  double* s_tab = reinterpret_cast<double*>(s_raw);                                        // 8 * CAMTAB
  double* s_scale = s_tab + I8_GROUP_CAMS * CAMTAB;                                        // I8_GROUP_ROWS: 2^(48 - e_row)
  unsigned long long* s_val = reinterpret_cast<unsigned long long*>(s_scale + I8_GROUP_ROWS);   // [rows][I8_VAL_LD]
  const int t = threadIdx.x, g = blockIdx.y, lane = t & 31, wid = t >> 5;
  const int c0 = g * I8_GROUP_CAMS, gc = min(I8_GROUP_CAMS, C - c0);
  const int rg0 = 11 * g;                                    // 8 cameras = 88 rows = 11 row groups
  const int nrgl = (g == (int)gridDim.y - 1) ? NRG - rg0 : 11;
  for (int i = t; i < gc * CAMTAB; i += blockDim.x) s_tab[i] = tab[c0 * CAMTAB + i];
  for (int i = t; i < I8_GROUP_ROWS; i += blockDim.x)
    s_scale[i] = (rg0 * 8 + i < NRG * 8) ? ldexp(1.0, 8 * I8_NS - e_row[rg0 * 8 + i]) : 0.0;
  for (int i = t; i < I8_GROUP_ROWS * I8_VAL_LD; i += blockDim.x) s_val[i] = 0ull;       // padding rows / column 63 stay 0
  __syncthreads();
  const bool worker = t < I8_PTS * gc;
  // point lane of a thread: slots 2j, 2j + 1 (the two point lanes of a half-warp when gc = 8) take lanes j and j + 8:
  // their staging columns then differ by 24 words = 8 banks and the 64-bit stores of phase 1 are conflict-free
  // (with neighbouring lanes, 3 words apart, one bank of the 16 was hit twice by every store: 2 wavefronts each)
  const int slot = worker ? t / gc : 0;
  const int q = slot < 16 ? (slot >> 1) + 8 * (slot & 1) : slot, cl = worker ? t % gc : 0, cam = c0 + cl;
  const bool zthread = (g == (int)gridDim.y - 1) && t >= 168 && t < 168 + I8_PTS;
  const int zrow = NCP * C - rg0 * 8;                        // local row of z in the last group
  const long long nkb = (P + I8_PTS - 1) / I8_PTS;
  // inputs of the next K block are loaded before the current one is evaluated (first version: 3 blocks
  // of 6 warps per SM stalled on the mask -> point -> factor loads: long-scoreboard 3 per issue)
  unsigned long long n_m = 0ull;
  double n_X[3] = {0, 0, 0}, n_li[6] = {0, 0, 0, 0, 0, 0};
  auto prefetch = [&](long long kb) {
    n_m = 0ull;
    const long long p = kb * I8_PTS + q;
    if (worker && kb < nkb && p < P) {
      n_m = mask[p];
#pragma unroll
      for (int a = 0; a < 3; ++a) n_X[a] = pts[3 * p + a];
#pragma unroll
      for (int a = 0; a < 6; ++a) n_li[a] = Lz[p * 9 + a];
    }
  };
  prefetch(blockIdx.x);
  for (long long kb = blockIdx.x; kb < nkb; kb += gridDim.x) {
    // ---- phase 1
    if (worker) {
      const long long p = kb * I8_PTS + q;
      const unsigned long long m = n_m;
      const bool live = (m >> cam) & 1ull;
      double X[3], li[6];
#pragma unroll
      for (int a = 0; a < 3; ++a) X[a] = n_X[a];
#pragma unroll
      for (int a = 0; a < 6; ++a) li[a] = n_li[a];
      prefetch(kb + gridDim.x);
      unsigned long long* dst = s_val + (size_t)(cl * NCP) * I8_VAL_LD + 3 * q;
      if (live) {
        const double w = wgt ? wgt[(long long)obs_start[p] + __popcll(m & ((1ull << cam) - 1ull))] : 1.0;
        ObsLin L;
        obs_linearize<false>(s_tab + cl * CAMTAB, X[0], X[1], X[2], 0.0, 0.0, w, L);
        const double* sc = s_scale + cl * NCP;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          double q0, q1;                                   // column k of Q = Jp L^-T
          if (k == 0) { q0 = L.Jp[0][0] * li[0]; q1 = L.Jp[1][0] * li[0]; }
          else if (k == 1) { q0 = fma(L.Jp[0][0], li[1], L.Jp[0][1] * li[2]); q1 = fma(L.Jp[1][0], li[1], L.Jp[1][1] * li[2]); }
          else { q0 = fma(L.Jp[0][0], li[3], fma(L.Jp[0][1], li[4], L.Jp[0][2] * li[5]));
                 q1 = fma(L.Jp[1][0], li[3], fma(L.Jp[1][1], li[4], L.Jp[1][2] * li[5])); }
#pragma unroll
          for (int a = 0; a < 9; ++a) dst[a * I8_VAL_LD + k] = i8_encode(fma(L.Jc[0][a], q0, L.Jc[1][a] * q1), sc[a]);
          dst[9 * I8_VAL_LD + k] = i8_encode(w * q0, sc[9]);
          dst[10 * I8_VAL_LD + k] = i8_encode(w * q1, sc[10]);
        }
      } else {
        // invisible pairs and the ragged tail are exact zeros
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
          for (int a = 0; a < NCP; ++a) dst[a * I8_VAL_LD + k] = 0ull;
      }
    }
    if (zthread) {
      const int qq = t - 168;
      const long long p = kb * I8_PTS + qq;
#pragma unroll
      for (int k = 0; k < 3; ++k)
        s_val[(size_t)zrow * I8_VAL_LD + 3 * qq + k] = p < P ? i8_encode(Lz[p * 9 + 6 + k], s_scale[zrow]) : 0ull;
    }
    __syncthreads();
    // ---- phase 2: warp = (row group, k-step), lane = (k half, row r8, 8-kappa half): 8 integers -> one
    // 8-byte store per slice (a warp writes 2 x 128 contiguous bytes per slice)
    {
      const int kh = lane >> 4, r8 = (lane >> 1) & 7, hf = lane & 1;
      const size_t sstride = (size_t)NRG * I8_RG_BYTES;
      unsigned char* lane_dst = planes + (((size_t)kb * I8_NS) * NRG + rg0) * I8_RG_BYTES + kh * 128 + r8 * 16 + hf * 8;
      const unsigned long long* lane_src = s_val + (size_t)r8 * I8_VAL_LD + kh * 16 + hf * 8;
      for (int task = wid; task < nrgl * 2; task += 6) {
        const int rgl = task >> 1, a = task & 1;
        const unsigned long long* src = lane_src + (size_t)rgl * 8 * I8_VAL_LD + a * 32;
        unsigned lo[8], hi[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) { const unsigned long long v = src[e]; lo[e] = (unsigned)v; hi[e] = (unsigned)(v >> 32); }
        unsigned char* dst = lane_dst + (size_t)rgl * I8_RG_BYTES + a * 256;
        // slices 0, 1 = bytes 5, 4 (bytes 1, 0 of the high words); slices 2..5 = bytes 3..0 of the low words
#pragma unroll
        for (int i = 0; i < I8_NS; ++i) {
          const unsigned sel = i == 0 ? 0x0051u : i == 1 ? 0x0040u : i == 2 ? 0x0073u : i == 3 ? 0x0062u : i == 4 ? 0x0051u : 0x0040u;
          unsigned w[2];
#pragma unroll
          for (int h2 = 0; h2 < 2; ++h2) {
            const unsigned* x = (i < 2) ? hi + 4 * h2 : lo + 4 * h2;
            w[h2] = __byte_perm(__byte_perm(x[0], x[1], sel), __byte_perm(x[2], x[3], sel), 0x5410);
          }
          *reinterpret_cast<uint2*>(dst + (size_t)i * sstride) = make_uint2(w[0], w[1]);
        }
      }
    }
    __syncthreads();
  }
}

// k_i8_make: the same planes as k_i8_make_ref, byte for byte, with evaluation and draining overlapped.
// Warps 0-5 evaluate (thread = (point lane q, camera), as in k_i8_make_ref but q = slot: the 4 point lanes
// of a warp then differ mod 4 and the 32-bit staging stores are conflict-free); warps 6-7 drain.  The
// staging tile is double-buffered and split into the low 32 and the top 16 bits of each encoded integer
// (48 bits of data, 6 B staged per entry instead of 8); the row strides (68 words, 72 halves = 36 words,
// both 4 mod 32) make the drain's 16-byte loads of 8 rows conflict-free.  Named barriers hand a buffer
// over: FULL[b] (evaluators arrive, drainers wait), EMPTY[b] (drainers arrive, evaluators wait two blocks
// later), so an evaluator never waits for stores and a drainer never for FP64.  A drain lane = (row r8,
// k half kh, k-step a) packs 16 kappa of one row, one core-matrix row per digit, and stores 16 B per
// slice: a warp writes one whole 512-byte row group per slice.  The weight chain obs_start -> wgt is
// prefetched in two stages (index two blocks ahead, weight one block ahead) with the mask, point and factor.
constexpr int I8_MK_EVAL = 192;           // evaluator threads (warps 0-5)
constexpr int I8_MK_DRAIN = 64;           // drainer threads (warps 6-7)
constexpr int I8_MK_THREADS = I8_MK_EVAL + I8_MK_DRAIN;
constexpr int I8_MK_LDL = 68;             // row stride of the low words (u32)
constexpr int I8_MK_LDH = 72;             // row stride of the top halves (u16)
constexpr int I8_MK_LO = I8_GROUP_ROWS * I8_MK_LDL;    // u32 per buffer
constexpr int I8_MK_HI = I8_GROUP_ROWS * I8_MK_LDH;    // u16 per buffer
inline size_t i8_make_smem_bytes() {
  return (size_t)I8_GROUP_CAMS * CAMTAB * 8 + (size_t)I8_GROUP_ROWS * 8 + 2 * ((size_t)I8_MK_LO * 4 + (size_t)I8_MK_HI * 2);
}
// named barriers with immediate ids (a register id makes ptxas reserve all 16)
template <int ID> __device__ __forceinline__ void i8_bar_sync() { asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(I8_MK_THREADS) : "memory"); }
template <int ID> __device__ __forceinline__ void i8_bar_arrive() { asm volatile("bar.arrive %0, %1;" ::"n"(ID), "n"(I8_MK_THREADS) : "memory"); }

__global__ void __launch_bounds__(I8_MK_THREADS, 2)
k_i8_make(const double* __restrict__ tab, const double* __restrict__ pts, const double* __restrict__ wgt,
          const uint32_t* __restrict__ obs_start, const unsigned long long* __restrict__ mask,
          const double* __restrict__ Lz, long long P, int C, int NRG, const int* __restrict__ e_row,
          unsigned char* __restrict__ planes) {
  extern __shared__ __align__(16) unsigned char s_raw[];
  double* s_tab = reinterpret_cast<double*>(s_raw);                                        // 8 * CAMTAB
  double* s_scale = s_tab + I8_GROUP_CAMS * CAMTAB;                                        // I8_GROUP_ROWS: 2^(48 - e_row)
  uint32_t* s_lo = reinterpret_cast<uint32_t*>(s_scale + I8_GROUP_ROWS);                   // [2][rows][I8_MK_LDL]
  uint16_t* s_hi = reinterpret_cast<uint16_t*>(s_lo + 2 * I8_MK_LO);                       // [2][rows][I8_MK_LDH]
  constexpr int BAR_FULL = 1, BAR_EMPTY = 3;                                               // + buffer
  const int t = threadIdx.x, g = blockIdx.y;
  const int c0 = g * I8_GROUP_CAMS, gc = min(I8_GROUP_CAMS, C - c0);
  const int rg0 = 11 * g;
  const int nrgl = (g == (int)gridDim.y - 1) ? NRG - rg0 : 11;
  for (int i = t; i < gc * CAMTAB; i += blockDim.x) s_tab[i] = tab[c0 * CAMTAB + i];
  for (int i = t; i < I8_GROUP_ROWS; i += blockDim.x)
    s_scale[i] = (rg0 * 8 + i < NRG * 8) ? ldexp(1.0, 8 * I8_NS - e_row[rg0 * 8 + i]) : 0.0;
  {
    uint4* z = reinterpret_cast<uint4*>(s_lo);                 // padding rows / column 63 stay 0 in both buffers
    const int n16 = (2 * I8_MK_LO * 4 + 2 * I8_MK_HI * 2) / 16;
    for (int i = t; i < n16; i += blockDim.x) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();
  const long long nkb = (P + I8_PTS - 1) / I8_PTS;
  const long long G = gridDim.x;

  if (t < I8_MK_EVAL) {
    // ---------------------------------------------------------------- evaluators
    const bool worker = t < I8_PTS * gc;
    const int q = worker ? t / gc : 0, cl = worker ? t % gc : 0, cam = c0 + cl;
    const bool zthread = (g == (int)gridDim.y - 1) && t >= 168 && t < 168 + I8_PTS;
    const int zrow = NCP * C - rg0 * 8;
    const unsigned long long below = (1ull << cam) - 1ull;
    // stage 2 (two blocks ahead): mask and CSR offset; stage 1 (one block ahead): point, factor and weight
    unsigned long long a_m = 0ull;
    uint32_t a_os = 0u;
    auto prefetch2 = [&](long long kb) {
      a_m = 0ull;
      const long long p = kb * I8_PTS + q;
      if (worker && kb < nkb && p < P) { a_m = mask[p]; a_os = wgt ? obs_start[p] : 0u; }
    };
    unsigned long long n_m = 0ull;
    double n_X[3] = {0, 0, 0}, n_li[6] = {0, 0, 0, 0, 0, 0}, n_w = 1.0;
    auto prefetch1 = [&](long long kb) {     // takes the stage-2 values of block kb
      n_m = a_m;
      const long long p = kb * I8_PTS + q;
      if (worker && kb < nkb && p < P) {
#pragma unroll
        for (int a = 0; a < 3; ++a) n_X[a] = pts[3 * p + a];
#pragma unroll
        for (int a = 0; a < 6; ++a) n_li[a] = Lz[p * 9 + a];
        if (wgt && ((n_m >> cam) & 1ull)) n_w = wgt[(long long)a_os + __popcll(n_m & below)];
      }
    };
    prefetch2(blockIdx.x);
    prefetch1(blockIdx.x);
    prefetch2(blockIdx.x + G);
    int it = 0;
    for (long long kb = blockIdx.x; kb < nkb; kb += G, ++it) {
      const int b = it & 1;
      const unsigned long long m = n_m;
      const bool live = (m >> cam) & 1ull;
      const double w = n_w;
      double X[3], li[6];
#pragma unroll
      for (int a = 0; a < 3; ++a) X[a] = n_X[a];
#pragma unroll
      for (int a = 0; a < 6; ++a) li[a] = n_li[a];
      prefetch1(kb + G);
      prefetch2(kb + 2 * G);
      if (it >= 2) { if (b) i8_bar_sync<BAR_EMPTY + 1>(); else i8_bar_sync<BAR_EMPTY>(); }                  // the drain of block kb - 2 G has read buffer b
      uint32_t* lo = s_lo + b * I8_MK_LO;
      uint16_t* hi = s_hi + b * I8_MK_HI;
      if (worker) {
        uint32_t* dlo = lo + (cl * NCP) * I8_MK_LDL + 3 * q;
        uint16_t* dhi = hi + (cl * NCP) * I8_MK_LDH + 3 * q;
        if (live) {
          ObsLin L;
          obs_linearize<false>(s_tab + cl * CAMTAB, X[0], X[1], X[2], 0.0, 0.0, w, L);
          const double* sc = s_scale + cl * NCP;
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            double q0, q1;                                   // column k of Q = Jp L^-T
            if (k == 0) { q0 = L.Jp[0][0] * li[0]; q1 = L.Jp[1][0] * li[0]; }
            else if (k == 1) { q0 = fma(L.Jp[0][0], li[1], L.Jp[0][1] * li[2]); q1 = fma(L.Jp[1][0], li[1], L.Jp[1][1] * li[2]); }
            else { q0 = fma(L.Jp[0][0], li[3], fma(L.Jp[0][1], li[4], L.Jp[0][2] * li[5]));
                   q1 = fma(L.Jp[1][0], li[3], fma(L.Jp[1][1], li[4], L.Jp[1][2] * li[5])); }
#pragma unroll
            for (int a = 0; a < NCP; ++a) {
              const double y = a < 9 ? fma(L.Jc[0][a], q0, L.Jc[1][a] * q1) : (a == 9 ? w * q0 : w * q1);
              const unsigned long long v = i8_encode_fma(y, sc[a]);
              dlo[a * I8_MK_LDL + k] = (uint32_t)v;
              dhi[a * I8_MK_LDH + k] = (uint16_t)(v >> 32);
            }
          }
        } else {
          // invisible pairs and the ragged tail are exact zeros
#pragma unroll
          for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int a = 0; a < NCP; ++a) { dlo[a * I8_MK_LDL + k] = 0u; dhi[a * I8_MK_LDH + k] = 0u; }
        }
      }
      if (zthread) {
        const int qq = t - 168;
        const long long pz = kb * I8_PTS + qq;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const unsigned long long v = pz < P ? i8_encode_fma(Lz[pz * 9 + 6 + k], s_scale[zrow]) : 0ull;
          lo[zrow * I8_MK_LDL + 3 * qq + k] = (uint32_t)v;
          hi[zrow * I8_MK_LDH + 3 * qq + k] = (uint16_t)(v >> 32);
        }
      }
      __threadfence_block();
      if (b) i8_bar_arrive<BAR_FULL + 1>(); else i8_bar_arrive<BAR_FULL>();
    }
  } else {
    // ---------------------------------------------------------------- drainers
    const int lane = t & 31, dw = (t - I8_MK_EVAL) >> 5;
    const int r8 = lane & 7, kh = (lane >> 3) & 1, a = lane >> 4;
    const int kap = 32 * a + 16 * kh;
    const size_t sstride = (size_t)NRG * I8_RG_BYTES;
    int it = 0;
    for (long long kb = blockIdx.x; kb < nkb; kb += G, ++it) {
      const int b = it & 1;
      if (b) i8_bar_sync<BAR_FULL + 1>(); else i8_bar_sync<BAR_FULL>();
      const uint32_t* lo = s_lo + b * I8_MK_LO + r8 * I8_MK_LDL + kap;
      const uint16_t* hi = s_hi + b * I8_MK_HI + r8 * I8_MK_LDH + kap;
      unsigned char* lane_dst = planes + (((size_t)kb * I8_NS) * NRG + rg0) * I8_RG_BYTES + a * 256 + kh * 128 + r8 * 16;
      for (int rgl = dw; rgl < nrgl; rgl += I8_MK_DRAIN / 32) {
        const uint4* sl = reinterpret_cast<const uint4*>(lo + rgl * 8 * I8_MK_LDL);
        const uint4* sh = reinterpret_cast<const uint4*>(hi + rgl * 8 * I8_MK_LDH);
        uint32_t x[16], hw[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) { const uint4 u = sl[j]; x[4 * j] = u.x; x[4 * j + 1] = u.y; x[4 * j + 2] = u.z; x[4 * j + 3] = u.w; }
#pragma unroll
        for (int j = 0; j < 2; ++j) { const uint4 u = sh[j]; hw[4 * j] = u.x; hw[4 * j + 1] = u.y; hw[4 * j + 2] = u.z; hw[4 * j + 3] = u.w; }
        // out[i][j]: slice i, kappa 4 j .. 4 j + 3.  Slices 0, 1 = bytes 1, 0 of the top halves (two per word);
        // slices 2..5 = bytes 3..0 of the low words (a 4 x 4 byte transpose per kappa quad)
        uint32_t out[I8_NS][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          out[0][j] = __byte_perm(hw[2 * j], hw[2 * j + 1], 0x7531);
          out[1][j] = __byte_perm(hw[2 * j], hw[2 * j + 1], 0x6420);
          const uint32_t t0 = __byte_perm(x[4 * j], x[4 * j + 1], 0x5140), t1 = __byte_perm(x[4 * j + 2], x[4 * j + 3], 0x5140);
          const uint32_t t2 = __byte_perm(x[4 * j], x[4 * j + 1], 0x7362), t3 = __byte_perm(x[4 * j + 2], x[4 * j + 3], 0x7362);
          out[2][j] = __byte_perm(t2, t3, 0x7632);
          out[3][j] = __byte_perm(t2, t3, 0x5410);
          out[4][j] = __byte_perm(t0, t1, 0x7632);
          out[5][j] = __byte_perm(t0, t1, 0x5410);
        }
        unsigned char* dst = lane_dst + (size_t)rgl * I8_RG_BYTES;
#pragma unroll
        for (int i = 0; i < I8_NS; ++i)
          *reinterpret_cast<uint4*>(dst + (size_t)i * sstride) = make_uint4(out[i][0], out[i][1], out[i][2], out[i][3]);
      }
      if (kb + 2 * G < nkb) { if (b) i8_bar_arrive<BAR_EMPTY + 1>(); else i8_bar_arrive<BAR_EMPTY>(); }      // the evaluators refill buffer b for block kb + 2 G
    }
  }
}

// ------------------------------------------------------------------------------ MMA issue plan
struct I8Op { int i, j, nj, fresh, coll; };
// The digit products of one k-step as tcgen05.mma instructions.  For a fixed slice i of A the slices j = 0..jmax of B
// are adjacent in shared memory and their anti-diagonals i + j adjacent in TMEM, so up to 256 / NCOL of them go into
// ONE instruction (N = nj NCOL).  Order: narrow instructions first, the widest last -- what sits in the tensor
// pipe's queue while the issuing thread crosses a stage boundary (commit, mbarrier wait, fence) must be long enough
// to cover it.  FIRST (the k-step after a flush): one instruction per product, the first to touch an
// anti-diagonal overwrites it.
template <int NCOL, bool FIRST>
struct I8KstepPlan {
  I8Op ops[32];
  int n;
  constexpr I8KstepPlan() : ops{}, n(0) {
    bool touched[I8_ND] = {};
    for (int i = I8_NS - 1; i >= 0; --i) {
      if (i > I8_DMAX) continue;
      const int jmax = (I8_NS - 1 < I8_DMAX - i) ? I8_NS - 1 : I8_DMAX - i;
      if (FIRST) {
        for (int j = 0; j <= jmax; ++j) {
          ops[n].i = i; ops[n].j = j; ops[n].nj = 1; ops[n].fresh = touched[i + j] ? 0 : 1; ops[n].coll = 0;
          touched[i + j] = true;
          ++n;
        }
      } else {
        const int per = 256 / NCOL, cnt = jmax + 1;
        int j = 0, rem = cnt % per;                     // the left-over (narrow) instruction goes first
        while (j <= jmax) {
          const int nj = (rem > 0) ? rem : per;
          rem = 0;
          ops[n].i = i; ops[n].j = j; ops[n].nj = nj; ops[n].fresh = 0; ops[n].coll = 0;
          ++n;
          j += nj;
        }
      }
    }
    // consecutive MMAs on the same slice i of A: the first keeps A in the collector, the others take it from there
    for (int q = 0; q < n; ++q) {
      const bool prev = q > 0 && ops[q - 1].i == ops[q].i, next = q + 1 < n && ops[q + 1].i == ops[q].i;
      ops[q].coll = prev ? (next ? 2 : 3) : (next ? 1 : 0);
    }
  }
};

// one k-step (32 kappa): sA / sB = operand bases of this k-step inside the stage
template <int NCOL, bool FIRST>
__device__ __forceinline__ void i8_issue_kstep(uint32_t tmem, uint32_t sA, uint32_t sB, uint32_t a_bytes, uint32_t b_bytes) {
  constexpr I8KstepPlan<NCOL, FIRST> plan{};
  constexpr uint32_t DESC_HI = ((uint32_t)I8_RG_BYTES >> 4) | (1u << 14);          // SBO = 512 B, descriptor version 1
  constexpr uint32_t DESC_LO = (128u >> 4) << 16;                                  // LBO = 128 B, no swizzle
  constexpr uint32_t IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);   // s32 += s8 x s8, M = 128
#pragma unroll
  for (int q = 0; q < plan.n; ++q) {
    const uint64_t adesc = ((uint64_t)DESC_HI << 32) | (DESC_LO | (((sA + plan.ops[q].i * a_bytes) >> 4) & 0x3FFF));
    const uint64_t bdesc = ((uint64_t)DESC_HI << 32) | (DESC_LO | (((sB + plan.ops[q].j * b_bytes) >> 4) & 0x3FFF));
    const uint32_t dcol = tmem + (uint32_t)((plan.ops[q].i + plan.ops[q].j) * NCOL);
    const uint32_t idesc = IDESC | ((uint32_t)(plan.ops[q].nj * NCOL >> 3) << 17), accum = plan.ops[q].fresh ? 0u : 1u;
    if (plan.ops[q].coll == 1) i8_mma<1>(dcol, adesc, bdesc, idesc, accum);
    else if (plan.ops[q].coll == 2) i8_mma<2>(dcol, adesc, bdesc, idesc, accum);
    else if (plan.ops[q].coll == 3) i8_mma<3>(dcol, adesc, bdesc, idesc, accum);
    else i8_mma<0>(dcol, adesc, bdesc, idesc, accum);
  }
}
// one K block = two k-steps; column block 1 (NCOL1 columns per anti-diagonal, TMEM columns [0, 7 NCOL1)) and
// the optional block 2 (NCOL2, TMEM columns [7 NCOL1, 7 (NCOL1 + NCOL2)), its own B region)
template <int NCOL1, int NCOL2>
__device__ __forceinline__ void i8_issue_block(bool first, uint32_t tmem, uint32_t sA, uint32_t sB1, uint32_t sB2,
                                               uint32_t a_bytes, uint32_t b1_bytes, uint32_t b2_bytes) {
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    const uint32_t o = 256u * ks;
    if (ks == 0 && first) {
      i8_issue_kstep<NCOL1, true>(tmem, sA + o, sB1 + o, a_bytes, b1_bytes);
      if (NCOL2 > 0) i8_issue_kstep<NCOL2 ? NCOL2 : 16, true>(tmem + I8_ND * NCOL1, sA + o, sB2 + o, a_bytes, b2_bytes);
    } else {
      i8_issue_kstep<NCOL1, false>(tmem, sA + o, sB1 + o, a_bytes, b1_bytes);
      if (NCOL2 > 0) i8_issue_kstep<NCOL2 ? NCOL2 : 16, false>(tmem + I8_ND * NCOL1, sA + o, sB2 + o, a_bytes, b2_bytes);
    }
  }
}

// ------------------------------------------------------------------------------ the window of the K-major schedule
// progress[cta] = (launch epoch << 32) | the first K block of the chunk the CTA's producer loads, or I8_DONE once it
// has loaded its last one.  The epoch is the CTA's own slot's epoch + 1 (every CTA publishes in every launch, the
// array is zeroed once at allocation), so a slot still holding the previous launch's value reads as "not started"
// and graph replays need no memset.  The window only keeps the CTAs' reads close enough for L2 to serve them:
// no data passes through it, so relaxed accesses suffice, and a CTA that has polled I8_POLL_CAP times stops
// waiting for the rest of the launch (CTAs need not be co-resident for the kernel to finish).
constexpr unsigned I8_DONE = 0x7fffffffu;
__device__ __forceinline__ void i8_progress_put(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// warp-collective: the smallest position of this launch over all CTAs (-1: a CTA that has not started)
__device__ __forceinline__ int i8_progress_min(const unsigned long long* progress, int nctas, unsigned epoch, int lane) {
  int m = 0x7fffffff;
  for (int i = lane; i < nctas; i += 32) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(progress + i) : "memory");
    m = min(m, (unsigned)(v >> 32) == epoch ? (int)(unsigned)v : -1);
  }
  return __reduce_min_sync(0xffffffffu, m);
}

// partial[cta][128][64] doubles: sum_d 2^-8(d+2) D_d  (row exponents are applied by k_i8_gather).
// window > 0: the K-major schedule's window in K blocks over progress[gridDim.x]; 0: no window.
__global__ void __launch_bounds__(I8_THREADS, 1)
k_i8_syrk(const __grid_constant__ I8Maps maps, const I8Work* __restrict__ work, double* __restrict__ partial, int* __restrict__ fail,
          unsigned long long* __restrict__ progress, int window,
          long long* __restrict__ stats /* null, or per CTA: MMA warp (waiting at FULL, total), producer (waiting for the window, total) cycles */) {
  extern __shared__ __align__(1024) uint8_t i8_smem[];
  __shared__ __align__(8) uint64_t s_bar[2 * I8_STAGES + 2];
  __shared__ uint32_t s_tmem;
  const I8Work W = work[blockIdx.x];
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const uint32_t a1_bytes = (uint32_t)W.m_nrg * I8_RG_BYTES, a_bytes = a1_bytes + (uint32_t)W.m2_nrg * I8_RG_BYTES;
  const uint32_t b_bytes = (uint32_t)W.n_nrg * I8_RG_BYTES;   // per slice
  const uint32_t b2_bytes = (uint32_t)W.n2_nrg * I8_RG_BYTES;
  const uint32_t B2_OFF = (uint32_t)I8_NS * b_bytes;          // block 2's B region follows block 1's
  constexpr uint32_t A_REGION = (uint32_t)I8_NS * 16 * I8_RG_BYTES;
  constexpr uint32_t STAGE_BYTES = (uint32_t)I8_NS * (16 + 8) * I8_RG_BYTES;
  const uint32_t smem0 = i8_smem_u32(i8_smem);
  const uint32_t bar_full = i8_smem_u32(&s_bar[0]), bar_empty = i8_smem_u32(&s_bar[I8_STAGES]);
  const uint32_t bar_tfull = i8_smem_u32(&s_bar[2 * I8_STAGES]), bar_tempty = i8_smem_u32(&s_bar[2 * I8_STAGES + 1]);
  const int ncol = W.n_nrg * 8, ncol2 = W.n2_nrg * 8;
  if (tid == 0) {
    for (int s = 0; s < I8_STAGES; ++s) { i8_mbar_init(bar_full + 8 * s, 1); i8_mbar_init(bar_empty + 8 * s, 1); }
    i8_mbar_init(bar_tfull, 1);
    i8_mbar_init(bar_tempty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (wid == 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(i8_smem_u32(&s_tmem)), "r"(512u) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = s_tmem;
  const int nkb = W.kb1 - W.kb0;

  if (wid == 4) {
    // ---- producer: TMA, one tensor copy per operand (all six digits of A / B1 / B2) issued by lane 0.  The whole
    // warp keeps the window.
    const long long t_begin = stats ? clock64() : 0;
    long long t_window = 0;
    unsigned epoch = 0;
    if (window > 0) epoch = __shfl_sync(0xffffffffu, lane == 0 ? (unsigned)(progress[blockIdx.x] >> 32) + 1u : 0u, 0);
    int lo = -1, polls = 0;                                   // lo: the slowest CTA's position as last seen
    for (int it = 0; it < nkb; ++it) {
      const int st = it % I8_STAGES;
      const int kb = W.kfirst + (it / W.kc) * W.kstride + it % W.kc;
      if (window > 0 && it % W.kc == 0) {
        if (lane == 0) i8_progress_put(progress + blockIdx.x, ((unsigned long long)epoch << 32) | (unsigned)kb);
        if (kb - window > lo && polls < I8_POLL_CAP) {
          const long long w0 = clock64();
          while (true) {
            lo = i8_progress_min(progress, gridDim.x, epoch, lane);
            if (kb - window <= lo || ++polls == I8_POLL_CAP) break;
            __nanosleep(256);
          }
          t_window += clock64() - w0;
        }
      }
      if (it >= I8_STAGES && lane == 0) i8_mbar_wait<false>(bar_empty + 8 * st, ((it / I8_STAGES) - 1) & 1, fail);
      if (lane == 0) i8_mbar_expect_tx(bar_full + 8 * st, (uint32_t)I8_NS * (a_bytes + b_bytes + b2_bytes));
      __syncwarp();
      if (lane == 0) {
        const uint32_t dstA = smem0 + st * STAGE_BYTES, dstB = dstA + A_REGION;
        if (W.m2_nrg > 0) i8_tma_5d(dstA, &maps.m[W.map_a], 0, W.m_rg0, 0, 0, kb, bar_full + 8 * st);
        else i8_tma_4d(dstA, &maps.m[W.map_a], 0, W.m_rg0, 0, kb, bar_full + 8 * st);
        i8_tma_4d(dstB, &maps.m[W.map_b1], 0, W.n_rg0, 0, kb, bar_full + 8 * st);
        if (W.n2_nrg > 0) i8_tma_4d(dstB + B2_OFF, &maps.m[W.map_b2], 0, W.n2_rg0, 0, kb, bar_full + 8 * st);
      }
    }
    if (window > 0 && lane == 0) i8_progress_put(progress + blockIdx.x, ((unsigned long long)epoch << 32) | I8_DONE);
    if (stats && lane == 0) { stats[4 * blockIdx.x + 2] = t_window; stats[4 * blockIdx.x + 3] = clock64() - t_begin; }
  } else if (wid == 5) {
    // ---- MMA issuer: the highest warp id of its scheduler; one elected lane
    if (i8_elect_one()) {
      int since_flush = 0, nflush = 0;
      long long t_wait = 0;
      const long long t_begin = stats ? clock64() : 0;
      for (int it = 0; it < nkb; ++it) {
        const int st = it % I8_STAGES;
        if (since_flush == 0 && nflush > 0) {                // the accumulators are with the epilogue
          i8_mbar_wait<false>(bar_tempty, (nflush - 1) & 1, fail);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        if (stats) {
          const long long w0 = clock64();
          i8_mbar_wait<false>(bar_full + 8 * st, (it / I8_STAGES) & 1, fail);
          t_wait += clock64() - w0;
        } else {
          i8_mbar_wait<false>(bar_full + 8 * st, (it / I8_STAGES) & 1, fail);
        }
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t sA = smem0 + st * STAGE_BYTES, sB = sA + A_REGION;
        const bool first = since_flush == 0;
        const uint32_t sB2 = sB + B2_OFF;
        if (ncol2 == 0) {
          if (ncol == 64) i8_issue_block<64, 0>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
          else if (ncol == 48) i8_issue_block<48, 0>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
          else if (ncol == 32) i8_issue_block<32, 0>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
          else i8_issue_block<16, 0>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
        } else if (ncol2 == 16) {
          if (ncol == 48) i8_issue_block<48, 16>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
          else if (ncol == 32) i8_issue_block<32, 16>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
          else i8_issue_block<16, 16>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
        } else {
          if (ncol == 32) i8_issue_block<32, 32>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
          else i8_issue_block<16, 32>(first, tmem, sA, sB, sB2, a_bytes, b_bytes, b2_bytes);
        }
        i8_commit(bar_empty + 8 * st);                       // frees the ring slot when these MMAs retire
        ++since_flush;
        if (since_flush == I8_FLUSH || it == nkb - 1) {
          i8_commit(bar_tfull);
          since_flush = 0;
          ++nflush;
        }
      }
      if (stats) { stats[4 * blockIdx.x] = t_wait; stats[4 * blockIdx.x + 1] = clock64() - t_begin; }
    }
  } else {
    // ---- epilogue: TMEM -> FP64 registers (thread = TMEM lane = tile row)
    const int q = wid & 3;
    const int row = q * 32 + lane;
    double acc[64];
#pragma unroll
    for (int c = 0; c < 64; ++c) acc[c] = 0.0;
    const int nfl = (nkb + I8_FLUSH - 1) / I8_FLUSH;
    for (int f = 0; f < nfl; ++f) {
      i8_mbar_wait<true>(bar_tfull, f & 1, fail);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
      for (int d = 0; d < I8_ND; ++d) {
        const double sc = ldexp(1.0, -8 * (d + 2));
        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(d * ncol);
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          if (16 * h < ncol) {                               // block 1: columns [0, ncol); warp-uniform
            uint32_t v[16];
            i8_tmem_ld16(taddr + 16 * h, v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[16 * h + c] = fma((double)(int)v[c], sc, acc[16 * h + c]);
          } else if (16 * h >= 64 - ncol2) {                 // block 2: the last ncol2 columns of the tile
            uint32_t v[16];
            i8_tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(I8_ND * ncol + d * ncol2 + 16 * h - (64 - ncol2)), v);
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
            for (int c = 0; c < 16; ++c) acc[16 * h + c] = fma((double)(int)v[c], sc, acc[16 * h + c]);
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      i8_mbar_arrive(bar_tempty);
    }
    double* out = partial + ((size_t)blockIdx.x * 128 + row) * 64;
#pragma unroll
    for (int c = 0; c < 64; ++c) out[c] = acc[c];
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (wid == 5) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// gridDim.x = tiles, gridDim.y splits a tile's entries: sum the partials of its CTAs (fixed order), apply the row
// exponents and write - Y Y^T into the pair-block layout of the slice partials (same convention as
// mma_consume: lower pair blocks 11 x 11, same-camera blocks with both triangles, the z row = reduced
// right-hand side).  Tile rows [0, 8 m_nrg) = range 1, the rest = range 2; tile columns [0, 8 n_nrg) = block 1,
// the last 8 n2_nrg columns = block 2.  An entry above the diagonal (rho < sig) stands for its transpose, except
// where that transpose is computed elsewhere: strip plan (cover = 0): the column is one of the tile's rows (the
// diagonal block's upper half; the rest of the row tile holds the transposes); cover plan: the entry lies in the
// square of the tile's rows and columns.  Every entry of the lower triangle is then taken exactly once.
__global__ void __launch_bounds__(256)
k_i8_gather(const double* __restrict__ partial, const I8Tile* __restrict__ tiles, int C, int cover,
            const int* __restrict__ e_row, int npairs, double* __restrict__ Sred) {
  const I8Tile T = tiles[blockIdx.x];
  const int n = NCP * C;
  const int nr1 = T.m_nrg * 8, nr = nr1 + T.m2_nrg * 8, nc1 = T.n_nrg * 8, nc2 = T.n2_nrg * 8, nc = nc1 + nc2;
  for (int idx = threadIdx.x + blockDim.x * blockIdx.y; idx < nr * nc; idx += blockDim.x * gridDim.y) {
    const int tr = idx / nc, tcl = idx - tr * nc;
    const bool second = tcl >= nc1;
    const int tc = second ? 64 - nc2 + (tcl - nc1) : tcl;               // column inside the 64-wide partial tile
    int rho = tr < nr1 ? T.m_rg0 * 8 + tr : T.m2_rg0 * 8 + (tr - nr1);
    int sig = second ? T.n2_rg0 * 8 + (tcl - nc1) : T.n_rg0 * 8 + tcl;
    if (rho < sig) {
      const int g = sig >> 3, gr = rho >> 3;
      const bool col_in_rows = (g >= T.m_rg0 && g < T.m_rg0 + T.m_nrg) || (g >= T.m2_rg0 && g < T.m2_rg0 + T.m2_nrg);
      if (col_in_rows && (!cover || (gr >= T.n_rg0 && gr < T.n_rg0 + T.n_nrg))) continue;
      const int x = rho; rho = sig; sig = x;
    }
    if (rho > n || sig >= n) continue;
    double s = 0.0;
    for (int w = 0; w < T.nw; ++w) s += partial[((size_t)(T.w0 + w) * 128 + tr) * 64 + tc];
    const double v = -ldexp(s, e_row[rho] + e_row[sig]);
    const int ck = sig / NCP, cb = sig % NCP;
    if (rho == n) { Sred[(size_t)npairs * 121 + ck * NCP + cb] = v; continue; }
    const int cj = rho / NCP, ra = rho % NCP;
    double* blk = Sred + (size_t)(cj * (cj + 1) / 2 + ck) * 121;
    blk[ra * NCP + cb] = v;
    if (cj == ck && ra != cb) blk[cb * NCP + ra] = v;
  }
}

// Resolution guard.  The digits hold every entry of row r to 48 bits of the row's maximum m_r, so the error of
// S_rc is ~ 2^-47 m_r m_c (measured 0.9 - 3.4 x that).  Where one point sets m_r far above the row's Schur
// diagonal (a heavily weighted point close to a camera: m_r^2 = 1.4e3 S_rr, Jacobi-scaled error 3.3e-11),
// that is coarser than FP64 needs.  One block: *gate = 1 when some camera row has m_r^2 > I8_RHO_MAX S_rr
// (S_rr = the diagonal of this shard's U - Y Y^T: a sum of per-point PSD terms, so never above the global
// one), then the DMMA kernel recomputes the slice partials and k_i8_fallback_finish replaces Sred.
// I8_RHO_MAX = 16 keeps 2^-47 * 3.4 * 16 = 4e-13 under a 1e-12 Jacobi-scaled error; ordinary rigs stay
// near 1e-3 (ring24, example18, ring64) and weights over six decades near 0.2.
constexpr double I8_RHO_MAX = 16.0;
__global__ void __launch_bounds__(256)
k_i8_check(const double* __restrict__ m_row, int C, const double* __restrict__ Sred, int* __restrict__ gate) {
  int bad = 0;
  for (int r = threadIdx.x; r < NCP * C; r += blockDim.x) {
    const double m = m_row[r];
    if (m > 0.0) {
      const int c = r / NCP, a = r % NCP;
      const double d = Sred[(size_t)(c * (c + 1) / 2 + c) * 121 + a * NCP + a];
      if (!(m * m <= I8_RHO_MAX * d)) bad = 1;
    }
  }
  bad = __syncthreads_or(bad);
  if (threadIdx.x == 0) *gate = bad;
}

// only when *gate: Sred = sum of the DMMA slice partials (fixed order) + U on the camera blocks
__global__ void __launch_bounds__(256)
k_i8_fallback_finish(const int* __restrict__ gate, const double* __restrict__ part, int nslices, size_t K,
                     const double* __restrict__ U, int C, double* __restrict__ Sred) {
  if (*gate == 0) return;
  for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < K; j += (size_t)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int b = 0; b < nslices; ++b) s += part[(size_t)b * K + j];
    const size_t blk = j / 121;
    if (j < (size_t)C * (C + 1) / 2 * 121) {
      // camera blocks are pair blocks cj * (cj + 1) / 2 + cj
      int c = (int)((sqrt(8.0 * (double)blk + 1.0) - 1.0) * 0.5);
      while (c * (c + 1) / 2 > (long long)blk) --c;
      while ((c + 1) * (c + 2) / 2 <= (long long)blk) ++c;
      if ((size_t)(c * (c + 1) / 2 + c) == blk) {
        const int e = (int)(j % 121), a = e / NCP, b2 = e % NCP;
        const int lo = a < b2 ? a : b2, hi = a < b2 ? b2 : a;
        s += U[c * CAMN_VALS + lo * NCP - lo * (lo - 1) / 2 + (hi - lo)];
      }
    }
    Sred[j] = s;
  }
}

}  // namespace lcba
