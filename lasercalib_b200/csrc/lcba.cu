// liblcba.so — C-ABI (include/lcba.h) over the sm_100a kernels.  Host side: handle,
// device memory, ingest, the trust-region driver loop (kernel sequencing only: all
// arithmetic, including step acceptance, runs on the device) and NCCL plumbing.
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <algorithm>
#include <map>
#include <string>
#include <thread>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "common.cuh"
#include "control.cuh"
#include "dense.cuh"
#include "eval.cuh"
#include "ingest.cuh"
#include "linearize.cuh"
#include "dense_passes.cuh"
#include "schur.cuh"
#include "schur_mma.cuh"
#include "schur_i8.cuh"
#include "peer_reduce.cuh"
#include "variants.cuh"
#include "bounds.cuh"
#include "covariance.cuh"

using namespace lcba;

// ------------------------------------------------------------------------------ NCCL (dlopen)
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;    // optional
  int (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
static const int NCCL_FLOAT64 = 8, NCCL_SUM = 0, NCCL_MAX = 2, NCCL_MIN = 3, NCCL_INT64 = 4;

static bool nccl_load(std::string& err) {
  if (g_nccl.lib) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) { err = std::string("dlopen libnccl.so.2 failed: ") + dlerror(); return false; }
#define LOADSYM(field, sym)                                                           \
  *(void**)(&g_nccl.field) = dlsym(g_nccl.lib, sym);                                  \
  if (!g_nccl.field) { err = std::string("missing NCCL symbol ") + sym; g_nccl.lib = nullptr; return false; }
  LOADSYM(GetUniqueId, "ncclGetUniqueId")
  LOADSYM(CommInitRank, "ncclCommInitRank")
  LOADSYM(AllReduce, "ncclAllReduce")
  LOADSYM(CommDestroy, "ncclCommDestroy")
  LOADSYM(GetErrorString, "ncclGetErrorString")
#undef LOADSYM
  *(void**)(&g_nccl.AllGather) = dlsym(g_nccl.lib, "ncclAllGather");
  return true;
}

// ------------------------------------------------------------------------------ handle
struct lcba_handle {
  int device = 0;
  int sm_count = SM_COUNT_B200;
  size_t smem_optin = 227 * 1024;
  cudaStream_t stream = nullptr;
  std::string err;
  std::vector<void*> allocs;

  // problem (this rank's shard)
  bool have_problem = false;
  int C = 0;
  long long P = 0, N = 0, P_total = 0;
  int kmax = 0, B = 0;
  long long nbins = 0;
  double *d_cams[2] = {nullptr, nullptr}, *d_pts[2] = {nullptr, nullptr}, *d_tab[2] = {nullptr, nullptr};
  int cur = 0;
  double2* d_uv = nullptr;
  double* d_w = nullptr;
  uint8_t* d_cam = nullptr;
  int32_t* d_pt = nullptr;
  int32_t* d_perm = nullptr;
  uint32_t* d_obs_start = nullptr;
  BinEntry* d_bins = nullptr;
  unsigned long long* d_mask = nullptr;
  // solver state
  double *d_Vg = nullptr, *d_scl_p = nullptr, *d_gt_p = nullptr, *d_Lz = nullptr, *d_gn_p = nullptr;
  double *d_camsum = nullptr, *d_scl_c = nullptr, *d_gt_c = nullptr, *d_g_c = nullptr, *d_pc = nullptr;
  double *d_campart = nullptr, *d_part = nullptr, *d_red = nullptr, *d_coef = nullptr;
  double *d_S = nullptr, *d_Lf = nullptr, *d_rhs = nullptr, *d_Sred = nullptr, *d_Spart = nullptr;
  int* d_fail = nullptr;
  long long* d_stats = nullptr;   // LCBA_SCHUR_STATS=1: per-CTA cycle counters of k_schur
  Ctl* d_ctl = nullptr;
  Ctl* h_ctl = nullptr;   // pinned
  int lin_grid = 0, obs_grid = 0, pt_grid = 0;
  SchurPlan plan;
  SchurKind* d_kinds = nullptr;
  SchurHw* d_hws = nullptr;
  MmaPlan mplan;                 // tensor-path plan (dense rigs)
  MmaKind* d_mkinds = nullptr;
  double *d_U = nullptr, *d_Upart = nullptr;
  int camn_grid = 0, camn_pb = 0;
  bool use_mma = false;
  // dense rigs: passes with a fixed camera per thread (dense_passes.cuh)
  bool use_dense = false;
  bool use_pt = false;           // point-parallel residual / jdot / backsub (no repeated pairs)
  int ptp_grid = 0;
  int dp_pb = 0, dp_grid_lin = 0;
  double *d_dpart = nullptr, *d_dred = nullptr;
  double* d_Yg = nullptr;        // Y of every (point, camera) in ring layout (k_make_Y), or null
  // int8 tensor-core Schur path (schur_i8.cuh)
  bool use_i8 = false;
  I8Maps i8maps;
  I8Plan i8plan;
  I8Work* d_i8work = nullptr;
  unsigned long long* d_i8progress = nullptr;   // k_i8_syrk's window: one slot per CTA (zeroed once)
  I8Tile* d_i8tiles = nullptr;
  unsigned char* d_i8planes = nullptr;
  double *d_i8partial = nullptr, *d_i8rmax = nullptr;
  int* d_i8erow = nullptr;
  int* d_i8gate = nullptr;        // 1: the last Schur pass fell back to DMMA (k_i8_check)
  double* d_i8mrow = nullptr;     // row maxima of Y (k_i8_rowexp -> k_i8_check)
  bool i8_guard = true;          // LCBA_I8_GUARD=0: no resolution check (tests of the int8 kernels alone)
  int i8_gx_max = 0, i8_gx_make = 0, i8_gx_make_ref = 0, i8_groups = 0;
  // outputs on demand
  double2* d_rout = nullptr;
  double *d_Jc = nullptr, *d_Jp = nullptr;
  // Schur-side view of the observations: one entry per distinct (point, camera) pair.  Equal to
  // (d_obs_start, d_w, N) unless the input repeats pairs; then repeated rows are merged into one
  // entry with the weight sqrt(sum w^2) (same Jacobian rows up to the weight: same U, W, Y).
  uint32_t* d_pair_start = nullptr;
  double* d_pair_w = nullptr;
  long long n_pairs = 0;
  // CUDA graphs of the two static launch sequences of an iteration (body: jdot .. trial; lin: commit +
  // linearise), one per parameter buffer; captured from the SECOND solve on a resident problem on
  // (a first solve never pays for capture + instantiation; LCBA_GRAPH=0 disables)
  struct GraphSlot { cudaGraphExec_t exec = nullptr; long long launches = 0; int key = -1; };
  GraphSlot g_body[2], g_lin[2];
  bool use_graphs = true;
  int solves_on_problem = 0;
  long long graph_replays = 0;
  // trace / profile
  lcba_iteration_cb iter_cb = nullptr;
  void* iter_cb_user = nullptr;
  std::vector<lcba_trace_row> trace;
  bool prof_on = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::map<std::string, std::pair<long long, double>> prof;
  long long launches = 0;
  // comm
  ncclComm_t comm = nullptr;
  int rank = 0, nranks = 1;
  int fix_cameras = 0, shared_intr = 0;
  // held parameters (lcba_set_fixed): C x 11 camera bytes and one byte per point of this shard, 1 = held.
  // Allocated with the problem and zero when nothing is held; their addresses never change, so the
  // captured graphs stay valid when the contents do.  masks_on = false: lcba_linearize, the unmasked tap.
  uint8_t *d_cam_fixed = nullptr, *d_pt_fixed = nullptr;
  long long n_cam_held = 0, n_pt_held = 0;
  double cam_fixed_sum = 0.0;      // checksum of the camera mask (the same on every rank of a sharded job)
  bool masks_on = true;
  std::vector<uint8_t> h_cam_fixed, h_pt_fixed;   // host copies of the masks (empty: nothing held)
  // box bounds (lcba_set_bounds): host copies over [cameras | points], -inf / +inf where a side is unbounded.  The
  // device buffers (effective box with held entries unbounded, then the bounded loop's per-entry vectors and
  // scalars) are allocated by the first bounded solve; `bounded`: the current solve or debug step runs that loop.
  std::vector<double> h_lb, h_ub;
  bool has_bounds = false, bounded = false;
  double *d_blb = nullptr, *d_bub = nullptr, *d_bsd = nullptr, *d_bdh = nullptr, *d_bp = nullptr, *d_br = nullptr;
  double* d_bred = nullptr;   // [0,6) linearise  [6,9) Gram diagonal  [9,11) step in box  [11,17) reflection  [17,19) J pass
  Bnd* d_bnd = nullptr;
  double *d_pred = nullptr, *d_scl_red = nullptr;   // shared-intrinsics mode: reduced step / scale
  double *d_sqpart = nullptr, *d_sqout = nullptr, *d_theta = nullptr;   // squared-residual variants
  // lcba_covariance, allocated by its first call (no captured graph references them): X = L_S^-1 (n_pad^2),
  // S^-1 (n^2), the per-point blocks (P x 6)
  double *d_cov_X = nullptr, *d_cov_Sinv = nullptr, *d_cov_pt = nullptr;
  int sq_grid = 0, sq_K = 0;
};

static std::string g_last_error;
// One NCCL communicator per process (one process per GPU): created by the first
// lcba_comm_init that carries a unique id, attached by later handles (id == NULL).
static ncclComm_t g_comm = nullptr;
static int g_comm_rank = -1, g_comm_nranks = 0, g_comm_device = -1;
// Peer-memory all-reduce of the process (peer_reduce.cuh): set up next to the communicator; ok == false -> NCCL
struct PeerState {
  bool ok = false;
  void* block = nullptr;                 // own block (cudaMalloc: exportable)
  void* opened[PEER_MAX_RANKS] = {};     // peers' blocks as mapped here
  PeerPtrs ptrs = {};
  unsigned epoch = 0;
  int* h_fail = nullptr;                 // mapped host word the kernel raises on a timed-out wait
  int* d_fail = nullptr;
};
static PeerState g_peer;
static bool g_peer_available = false;    // mapped on every rank (the route may still be switched off)
static void set_error(lcba_t* h, const std::string& s) {
  if (h) h->err = s;
  g_last_error = s;
}

template <typename T>
static int dev_alloc(lcba_t* h, T** p, size_t count) {
  *p = nullptr;
  if (count == 0) count = 1;
  void* q = nullptr;
  // stream-ordered pool allocation: repeated set_problem calls reuse the cached blocks
  cudaError_t e = cudaMallocAsync(&q, count * sizeof(T), h->stream);
  if (e != cudaSuccess) {
    set_error(h, std::string("cudaMallocAsync: ") + cudaGetErrorString(e));
    return LCBA_E_CUDA;
  }
  h->allocs.push_back(q);
  *p = (T*)q;
  return LCBA_OK;
}

static void drop_graphs(lcba_t* h) {
  lcba_handle::GraphSlot* slots[] = {&h->g_body[0], &h->g_body[1], &h->g_lin[0], &h->g_lin[1]};
  for (auto* sl : slots) {
    if (sl->exec) cudaGraphExecDestroy(sl->exec);
    sl->exec = nullptr;
    sl->key = -1;
  }
  h->solves_on_problem = 0;
}

static void dev_free_all(lcba_t* h) {
  drop_graphs(h);          // the graphs hold the device pointers
  for (void* p : h->allocs) cudaFreeAsync(p, h->stream);
  h->allocs.clear();
}

#define KL(h, name, ...)                                              \
  do {                                                                \
    if ((h)->prof_on) cudaEventRecord((h)->ev0, (h)->stream);         \
    __VA_ARGS__;                                                      \
    (h)->launches++;                                                  \
    if ((h)->prof_on) {                                               \
      cudaEventRecord((h)->ev1, (h)->stream);                         \
      cudaEventSynchronize((h)->ev1);                                 \
      float ms_ = 0;                                                  \
      cudaEventElapsedTime(&ms_, (h)->ev0, (h)->ev1);                 \
      auto& pr_ = (h)->prof[name];                                    \
      pr_.first++;                                                    \
      pr_.second += ms_;                                              \
    }                                                                 \
  } while (0)

// NVTX range per solver pass (visible in Nsight Systems / ncu --nvtx; free when no tool listens)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

static int check_launch(lcba_t* h, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error(h, std::string(what) + ": " + cudaGetErrorString(e));
    return LCBA_E_CUDA;
  }
  return LCBA_OK;
}

static int allreduce(lcba_t* h, double* p, size_t n, int op) {
  if (!h->comm) return LCBA_OK;
  if (g_peer.ok && n <= PEER_SLOT && op != NCCL_MIN) {
    // one kernel over NVLink peer memory (peer_reduce.cuh); same call order on every rank, like NCCL
    ++g_peer.epoch;
    k_peer_allreduce<<<peer_grid(n), PEER_THREADS, 0, h->stream>>>(g_peer.ptrs, h->rank, h->nranks, g_peer.epoch, p, n,
                                                                   op == NCCL_MAX ? PEER_OP_MAX : PEER_OP_SUM, g_peer.d_fail);
    h->launches++;
    return LCBA_OK;
  }
  int rc = g_nccl.AllReduce(p, p, n, NCCL_FLOAT64, op, h->comm, h->stream);
  if (rc != 0) {
    set_error(h, std::string("ncclAllReduce: ") + g_nccl.GetErrorString(rc));
    return LCBA_E_NCCL;
  }
  return LCBA_OK;
}

// ------------------------------------------------------------------------------ lifecycle
extern "C" int lcba_version(void) { return LCBA_VERSION; }

extern "C" const char* lcba_last_error(const lcba_t* h) {
  return h ? h->err.c_str() : g_last_error.c_str();
}

extern "C" void lcba_default_options(lcba_options* o) {
  if (!o) return;
  memset(o, 0, sizeof(*o));
  o->ftol = 1e-8;   // scipy default; PySBA.bundleAdjust passes 1e-4 (pySBA.py:132)
  o->xtol = 1e-8;
  o->gtol = 1e-8;
  o->max_nfev = 0;
  o->verbose = 0;
  o->profile = 0;
}

extern "C" int lcba_create(lcba_t** out, int device) {
  if (!out) { set_error(nullptr, "lcba_create: out is NULL"); return LCBA_E_ARG; }
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_error(nullptr, std::string("no CUDA device (the engine has no CPU fallback): ") +
                           (e != cudaSuccess ? cudaGetErrorString(e) : "device count 0"));
    return LCBA_E_CUDA;
  }
  lcba_t* h = new lcba_handle();
  if (device < 0) cudaGetDevice(&device);
  h->device = device;
  if ((e = cudaSetDevice(device)) != cudaSuccess) {
    set_error(nullptr, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
    delete h;
    return LCBA_E_CUDA;
  }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  h->sm_count = prop.multiProcessorCount;
  h->smem_optin = prop.sharedMemPerBlockOptin;
  cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  {
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long keep = ~0ull;       // keep freed blocks cached in the pool
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
  }
  cudaEventCreate(&h->ev0);
  cudaEventCreate(&h->ev1);
  cudaMallocHost((void**)&h->h_ctl, sizeof(Ctl));
  // opt in to large dynamic shared memory (limit = opt-in size minus the kernel's static part)
  {
    const void* big_smem_kernels[] = {(const void*)k_linearize, (const void*)k_backsub,
                                      (const void*)k_schur<true, 160>, (const void*)k_schur<false, 160>,
                                      (const void*)k_schur<true, 128>, (const void*)k_schur<false, 128>,
                                      (const void*)k_residual, (const void*)k_cam_normal, (const void*)k_make_Y,
                                      (const void*)k_schur_mma<1, false>, (const void*)k_schur_mma<2, false>,
                                      (const void*)k_schur_mma<3, false>, (const void*)k_schur_mma<4, false>,
                                      (const void*)k_schur_mma<5, false>, (const void*)k_schur_mma<6, false>,
                                      (const void*)k_schur_mma<1, true>, (const void*)k_schur_mma<2, true>,
                                      (const void*)k_schur_mma<3, true>, (const void*)k_schur_mma<4, true>,
                                      (const void*)k_schur_mma<5, true>, (const void*)k_schur_mma<6, true>,
                                      (const void*)k_sq_camonly<true>, (const void*)k_sq_camonly<false>,
                                      (const void*)k_linearize_dense,
                                      (const void*)k_residual_pt, (const void*)k_jdot_pt, (const void*)k_backsub_pt,
                                      (const void*)k_i8_syrk, (const void*)k_i8_make,
                                      (const void*)k_i8_make_ref,
                                      (const void*)k_jdot,      (const void*)k_jacobian_blocks,
                                      (const void*)k_point_cov<16>, (const void*)k_point_cov<8>};
    for (const void* f : big_smem_kernels) {
      cudaFuncAttributes fa;
      e = cudaFuncGetAttributes(&fa, f);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)(h->smem_optin - fa.sharedSizeBytes));
      if (e != cudaSuccess) {
        set_error(nullptr, std::string("lcba_create: shared-memory opt-in: ") + cudaGetErrorString(e));
        delete h;
        return LCBA_E_CUDA;
      }
    }
  }
  *out = h;
  return LCBA_OK;
}

extern "C" void lcba_destroy(lcba_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  h->comm = nullptr;   // the communicator belongs to the process (see g_comm)
  dev_free_all(h);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->h_ctl) cudaFreeHost(h->h_ctl);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

// ------------------------------------------------------------------------------ ingest
static inline unsigned nblk(long long n, int t) { return (unsigned)std::max<long long>(1, (n + t - 1) / t); }

extern "C" int lcba_set_problem(lcba_t* h, int32_t C, int64_t P, int64_t N, const double* cams,
                                const double* pts, const double* obs_uv, const int64_t* cam_idx,
                                const int64_t* pt_idx, const double* weights) {
  return lcba_set_problem_shard(h, C, P, N, cams, pts, obs_uv, cam_idx, pt_idx, weights, 0);
}

extern "C" int lcba_set_problem_shard(lcba_t* h, int32_t C, int64_t P, int64_t N, const double* cams,
                                      const double* pts, const double* obs_uv, const int64_t* cam_idx,
                                      const int64_t* pt_idx, const double* weights, int64_t pt_offset) {
  if (!h) return LCBA_E_ARG;
  if (C <= 0 || P <= 0 || N <= 0 || !cams || !pts || !obs_uv || !cam_idx || !pt_idx) {
    set_error(h, "lcba_set_problem: null pointer or non-positive size");
    return LCBA_E_ARG;
  }
  if (C > LCBA_MAX_CAMERAS) {
    set_error(h, "lcba_set_problem: more than 64 cameras is not supported");
    return LCBA_E_UNSUPPORTED;
  }
  if (N >= (1LL << 31) || P >= (1LL << 31) / 3) {
    set_error(h, "lcba_set_problem: shard too large for 32-bit indices; shard by point");
    return LCBA_E_UNSUPPORTED;
  }
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  dev_free_all(h);
  h->have_problem = false;
  h->d_rout = nullptr; h->d_Jc = nullptr; h->d_Jp = nullptr;
  h->d_sqpart = nullptr; h->d_sqout = nullptr; h->d_theta = nullptr; h->sq_grid = 0; h->sq_K = 0;
  h->d_cov_X = h->d_cov_Sinv = h->d_cov_pt = nullptr;
  h->C = C; h->P = P; h->N = N; h->P_total = P; h->cur = 0;
  cudaStream_t st = h->stream;

  for (int i = 0; i < 2; ++i) {
    LCBA_TRY(dev_alloc(h, &h->d_cams[i], (size_t)C * NCP));
    LCBA_TRY(dev_alloc(h, &h->d_pts[i], (size_t)P * 3));
    LCBA_TRY(dev_alloc(h, &h->d_tab[i], (size_t)C * CAMTAB));
  }
  LCBA_TRY(dev_alloc(h, &h->d_uv, (size_t)N));
  if (weights) LCBA_TRY(dev_alloc(h, &h->d_w, (size_t)N)); else h->d_w = nullptr;
  LCBA_TRY(dev_alloc(h, &h->d_cam, (size_t)N));
  LCBA_TRY(dev_alloc(h, &h->d_pt, (size_t)N));
  LCBA_TRY(dev_alloc(h, &h->d_obs_start, (size_t)P + 1));
  LCBA_TRY(dev_alloc(h, &h->d_mask, (size_t)P));
  LCBA_TRY(dev_alloc(h, &h->d_cam_fixed, (size_t)C * NCP));
  LCBA_TRY(dev_alloc(h, &h->d_pt_fixed, (size_t)P));
  LCBA_CUDA(h, cudaMemsetAsync(h->d_cam_fixed, 0, (size_t)C * NCP, h->stream));
  LCBA_CUDA(h, cudaMemsetAsync(h->d_pt_fixed, 0, (size_t)P, h->stream));
  h->n_cam_held = h->n_pt_held = 0;
  h->cam_fixed_sum = 0.0;
  h->h_cam_fixed.clear(); h->h_pt_fixed.clear();
  h->h_lb.clear(); h->h_ub.clear();
  h->has_bounds = h->bounded = false;
  h->d_blb = h->d_bub = h->d_bsd = h->d_bdh = h->d_bp = h->d_br = h->d_bred = nullptr;
  h->d_bnd = nullptr;

  // temporaries (freed at the end of ingest)
  long long *t_cam = nullptr, *t_pt = nullptr;
  unsigned long long *t_keys = nullptr, *t_keys2 = nullptr;
  double2* t_uv = nullptr;
  double* t_w = nullptr;
  int32_t *t_iota = nullptr, *t_perm = nullptr;
  int* d_flags = nullptr;
  void* t_cub = nullptr;
  auto cleanup = [&]() {
    void* tmp[] = {t_cam, t_pt, t_keys, t_keys2, t_uv, t_w, t_iota, t_cub, d_flags};
    for (void* q : tmp) if (q) cudaFreeAsync(q, st);
  };
#define ING(call)                                                                   \
  do {                                                                              \
    cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess) {                                                        \
      set_error(h, std::string(#call) + ": " + cudaGetErrorString(e_));             \
      cleanup();                                                                    \
      return LCBA_E_CUDA;                                                           \
    }                                                                               \
  } while (0)
  ING(cudaMallocAsync(&t_cam, N * 8, st));
  ING(cudaMallocAsync(&t_pt, N * 8, st));
  ING(cudaMallocAsync(&t_keys, N * 8, st));
  ING(cudaMallocAsync(&t_uv, N * 16, st));
  if (weights) ING(cudaMallocAsync(&t_w, N * 8, st));
  ING(cudaMallocAsync(&d_flags, 2 * sizeof(int), st));
  ING(cudaMemsetAsync(d_flags, 0, 2 * sizeof(int), st));
  ING(cudaMemcpyAsync(t_cam, cam_idx, N * 8, cudaMemcpyHostToDevice, st));
  ING(cudaMemcpyAsync(t_pt, pt_idx, N * 8, cudaMemcpyHostToDevice, st));
  ING(cudaMemcpyAsync(t_uv, obs_uv, N * 16, cudaMemcpyHostToDevice, st));
  if (weights) ING(cudaMemcpyAsync(t_w, weights, N * 8, cudaMemcpyHostToDevice, st));
  ING(cudaMemcpyAsync(h->d_cams[0], cams, (size_t)C * NCP * 8, cudaMemcpyHostToDevice, st));
  ING(cudaMemcpyAsync(h->d_pts[0], pts, (size_t)P * 3 * 8, cudaMemcpyHostToDevice, st));
  k_make_keys<<<nblk(N, 256), 256, 0, st>>>(t_cam, t_pt, N, C, P, pt_offset, t_keys, d_flags);
  h->launches++;
  int flags[2] = {0, 0};
  ING(cudaMemcpyAsync(flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, st));
  ING(cudaStreamSynchronize(st));
  if (flags[0] & 1) {
    set_error(h, "lcba_set_problem: camera or point index out of range");
    cleanup();
    return LCBA_E_ARG;
  }
  const unsigned long long* keys_sorted = t_keys;
  h->d_perm = nullptr;
  if (flags[0] & 2) {
    // unsorted input: radix sort by (point, camera), remember the permutation
    ING(cudaMallocAsync(&t_keys2, N * 8, st));
    ING(cudaMallocAsync(&t_iota, N * 4, st));
    LCBA_TRY(dev_alloc(h, &h->d_perm, (size_t)N));
    k_iota<<<nblk(N, 256), 256, 0, st>>>(t_iota, N);
    h->launches++;
    size_t cub_bytes = 0;
    int end_bit = 8;
    while ((1LL << (end_bit - 8)) < P && end_bit < 64) ++end_bit;
    cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, t_keys, t_keys2, t_iota, h->d_perm,
                                    (int)N, 0, end_bit, st);
    ING(cudaMallocAsync(&t_cub, cub_bytes, st));
    ING(cub::DeviceRadixSort::SortPairs(t_cub, cub_bytes, t_keys, t_keys2, t_iota, h->d_perm,
                                        (int)N, 0, end_bit, st));
    h->launches += 8;
    keys_sorted = t_keys2;
  }
  k_narrow_gather<<<nblk(N, 256), 256, 0, st>>>(keys_sorted, h->d_perm, t_uv, t_w, N, h->d_cam,
                                               h->d_pt, h->d_uv, h->d_w, d_flags);
  k_obs_start<<<nblk(N + 1, 256), 256, 0, st>>>(h->d_pt, N, P, h->d_obs_start);
  k_point_masks<<<nblk(P, 256), 256, 0, st>>>(h->d_cam, h->d_obs_start, P, h->d_mask, d_flags + 1);
  h->launches += 3;
  ING(cudaMemcpyAsync(flags, d_flags, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
  ING(cudaStreamSynchronize(st));
  ING(cudaGetLastError());
  h->d_pair_start = h->d_obs_start;
  h->d_pair_w = h->d_w;
  h->n_pairs = N;
  if (flags[0] & 4) {
    // repeated (camera, point) rows: distinct-pair view for the Schur-side passes
    int *t_first = nullptr, *t_rank = nullptr;
    void* t_scan = nullptr;
    auto drop = [&]() { void* q[] = {t_first, t_rank, t_scan}; for (void* x : q) if (x) cudaFreeAsync(x, st); };
    cudaError_t e = cudaMallocAsync(&t_first, N * sizeof(int), st);
    if (e == cudaSuccess) e = cudaMallocAsync(&t_rank, N * sizeof(int), st);
    size_t scan_bytes = 0;
    if (e == cudaSuccess) {
      k_pair_first<<<nblk(N, 256), 256, 0, st>>>(h->d_cam, h->d_pt, N, t_first);
      cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, t_first, t_rank, (int)N, st);
      e = cudaMallocAsync(&t_scan, scan_bytes, st);
    }
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(t_scan, scan_bytes, t_first, t_rank, (int)N, st);
    int last[2] = {0, 0};
    if (e == cudaSuccess) e = cudaMemcpyAsync(&last[0], t_rank + (N - 1), sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(&last[1], t_first + (N - 1), sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      set_error(h, std::string("lcba_set_problem: pair scan: ") + cudaGetErrorString(e));
      drop(); cleanup();
      return LCBA_E_CUDA;
    }
    h->n_pairs = (long long)last[0] + last[1];
    h->launches += 4;
    int rc = dev_alloc(h, &h->d_pair_w, (size_t)h->n_pairs);
    if (rc == LCBA_OK) rc = dev_alloc(h, &h->d_pair_start, (size_t)P + 1);
    if (rc != LCBA_OK) { drop(); cleanup(); return rc; }
    k_pair_weights<<<nblk(N, 256), 256, 0, st>>>(t_first, t_rank, h->d_w, N, h->d_pair_w);
    k_pair_start<<<nblk(P + 1, 256), 256, 0, st>>>(h->d_obs_start, t_rank, P, N, h->n_pairs, h->d_pair_start);
    h->launches += 2;
    drop();
  }
  cleanup();
#undef ING
  h->kmax = flags[1];
  h->B = LIN_THREADS - h->kmax;
  if (h->B < 32) { set_error(h, "lcba_set_problem: too many observations per point"); return LCBA_E_UNSUPPORTED; }
  h->nbins = N / h->B + 1;
  LCBA_TRY(dev_alloc(h, &h->d_bins, (size_t)h->nbins + 2));
  k_bin_table<<<nblk(h->nbins + 1, 256), 256, 0, st>>>(h->d_obs_start, P, h->nbins, h->B, h->d_bins);
  h->launches++;

  // solver buffers
  const int n = C * NCP;
  LCBA_TRY(dev_alloc(h, &h->d_Vg, (size_t)P * 9));
  LCBA_TRY(dev_alloc(h, &h->d_scl_p, (size_t)P * 3));
  LCBA_TRY(dev_alloc(h, &h->d_gt_p, (size_t)P * 3));
  LCBA_TRY(dev_alloc(h, &h->d_Lz, (size_t)P * 9));
  LCBA_TRY(dev_alloc(h, &h->d_gn_p, (size_t)P * 3));
  LCBA_TRY(dev_alloc(h, &h->d_camsum, (size_t)C * CAMSUM + 1 + PP_K));
  LCBA_TRY(dev_alloc(h, &h->d_scl_c, (size_t)n));
  LCBA_TRY(dev_alloc(h, &h->d_gt_c, (size_t)n));
  LCBA_TRY(dev_alloc(h, &h->d_g_c, (size_t)n));
  LCBA_TRY(dev_alloc(h, &h->d_pc, (size_t)n));
  LCBA_TRY(dev_alloc(h, &h->d_pred, (size_t)n));
  LCBA_TRY(dev_alloc(h, &h->d_scl_red, (size_t)n));
  LCBA_TRY(dev_alloc(h, &h->d_S, (size_t)n * n));
  LCBA_TRY(dev_alloc(h, &h->d_Lf, (size_t)(n + 1) * n));   // + rhs row (k_chol_fused)
  LCBA_TRY(dev_alloc(h, &h->d_rhs, (size_t)n));
  LCBA_TRY(dev_alloc(h, &h->d_red, 64));
  LCBA_TRY(dev_alloc(h, &h->d_coef, 2));
  LCBA_TRY(dev_alloc(h, &h->d_fail, 2));   // [0] failure bits, [1] grid-barrier counter
  LCBA_TRY(dev_alloc(h, &h->d_ctl, 1));
  // grids: persistent-style, a multiple of the SM count
  const size_t lin_smem = linearize_smem_doubles(C) * 8;
  const int lin_per_sm = std::max(1, (int)std::min<size_t>(4, h->smem_optin / (lin_smem + 1024)));
  h->lin_grid = (int)std::min<long long>(h->nbins, (long long)h->sm_count * lin_per_sm);
  h->obs_grid = (int)std::min<long long>(nblk(N, 256), (long long)h->sm_count * 8);
  h->pt_grid = (int)std::min<long long>(nblk(P, 256), (long long)h->sm_count * 8);
  const int max_grid = std::max(std::max(h->lin_grid, h->obs_grid), h->pt_grid);
  LCBA_TRY(dev_alloc(h, &h->d_campart, (size_t)h->lin_grid * C * CAMSUM));
  LCBA_TRY(dev_alloc(h, &h->d_part, (size_t)max_grid * 16));
  // Schur plan
  h->plan = make_schur_plan(C, h->sm_count, h->smem_optin - 2048);
  LCBA_TRY(dev_alloc(h, &h->d_kinds, h->plan.kinds.size()));
  LCBA_TRY(dev_alloc(h, &h->d_hws, h->plan.hws.size()));
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_kinds, h->plan.kinds.data(), h->plan.kinds.size() * sizeof(SchurKind),
                               cudaMemcpyHostToDevice, st));
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_hws, h->plan.hws.data(), h->plan.hws.size() * sizeof(SchurHw),
                               cudaMemcpyHostToDevice, st));
  LCBA_TRY(dev_alloc(h, &h->d_Sred, h->plan.part_stride));
  // tensor-path plan: dense rigs only (the DFMA kernel skips invisible blocks on sparse ones)
  h->use_mma = false;
  h->d_mkinds = nullptr; h->d_U = nullptr; h->d_Upart = nullptr; h->d_Yg = nullptr;
  int max_slices = h->plan.nslices;
  {
    // Density crossover, measured on ring24 x 1 M (profiles/r02_density_crossover.txt): the DMMA
    // SYRK costs ~P C^2 whatever the visibility, the DFMA kernel ~sum k_i^2; at 50 % visibility
    // the tensor path already wins 3.9 + 0.6 ms against 6.8 ms.  LCBA_MMA_DENSITY overrides.
    const char* de = getenv("LCBA_MMA_DENSITY");
    const double min_density = de ? atof(de) : 0.25;
    const bool dense = (double)h->n_pairs >= min_density * (double)P * C;
    const char* env = getenv("LCBA_SCHUR_MMA");
    const bool want = env ? atoi(env) != 0 : (dense && C >= 8);
    if (want && C <= MMA_MAX_CAMERAS) {
      // Y precomputed in HBM when it fits comfortably (288 B per (point, camera)); otherwise the
      // producers of k_schur_mma evaluate it in place (and need the camera tables in shared memory)
      // int8 tensor-core path (tcgen05, schur_i8.cuh): default for shards of >= 32768 points.  Its
      // quantisation errors are independent per entry, so its accuracy IMPROVES with the number of
      // points (2^-46 (rowmax/rms)^2 / sqrt(3 P): 2e-16 at 1 M points, FP64 rounding of the DMMA path
      // grows like sqrt(3 P)); below ~30 k points the DMMA path is the more accurate one and the
      // fixed costs of the 148-CTA pipeline do not pay.  LCBA_SCHUR_I8=0/1 overrides.
      {
        const char* ie = getenv("LCBA_SCHUR_I8");
        h->use_i8 = ie ? atoi(ie) != 0 : P >= 32768;
      }
      if (h->use_i8) {
        {
          // LCBA_I8_PLAN=strip|cover overrides the cost model's choice of tile plan; LCBA_I8_SCHED=range gives each
          // CTA one contiguous K range instead of the K-major schedule (A/B runs, tests)
          const char* pe = getenv("LCBA_I8_PLAN");
          const int which = !pe ? 0 : (strcmp(pe, "strip") == 0 ? 1 : (strcmp(pe, "cover") == 0 ? 2 : 0));
          const char* se = getenv("LCBA_I8_SCHED");
          h->i8plan = make_i8_best_plan(C, P, h->sm_count, which, !(se && strcmp(se, "range") == 0));
        }
        const I8Plan& ip = h->i8plan;
        h->i8_groups = (C + I8_GROUP_CAMS - 1) / I8_GROUP_CAMS;
        h->i8_gx_max = (int)std::max<long long>(1, std::min<long long>(ip.nkb, (long long)h->sm_count * 4 / h->i8_groups));   // one wave: 4 blocks per SM
        h->i8_gx_make = (int)std::max<long long>(1, std::min<long long>(ip.nkb, (long long)h->sm_count * 2 / h->i8_groups));   // one wave: 2 blocks per SM (87 KB of shared memory each)
        h->i8_gx_make_ref = (int)std::max<long long>(1, std::min<long long>(ip.nkb, (long long)h->sm_count * 3 / h->i8_groups));   // one wave: 3 blocks per SM
        LCBA_TRY(dev_alloc(h, &h->d_i8work, ip.work.size()));
        LCBA_TRY(dev_alloc(h, &h->d_i8tiles, ip.tiles.size()));
        LCBA_CUDA(h, cudaMemcpyAsync(h->d_i8work, ip.work.data(), ip.work.size() * sizeof(I8Work), cudaMemcpyHostToDevice, st));
        LCBA_CUDA(h, cudaMemcpyAsync(h->d_i8tiles, ip.tiles.data(), ip.tiles.size() * sizeof(I8Tile), cudaMemcpyHostToDevice, st));
        LCBA_TRY(dev_alloc(h, &h->d_i8progress, ip.work.size()));
        LCBA_CUDA(h, cudaMemsetAsync(h->d_i8progress, 0, ip.work.size() * sizeof(unsigned long long), st));
        LCBA_TRY(dev_alloc(h, &h->d_i8planes, ip.plane_bytes));
        if (!i8_encode_maps(ip, h->d_i8planes, &h->i8maps)) {
          set_error(h, "lcba_set_problem: tensor-map encode (cuTensorMapEncodeTiled) of the int8 Schur digit planes failed");
          return LCBA_E_CUDA;
        }
        LCBA_TRY(dev_alloc(h, &h->d_i8partial, ip.work.size() * 128 * 64));
        LCBA_TRY(dev_alloc(h, &h->d_i8rmax, (size_t)h->i8_gx_max * ip.NRG * 8));
        LCBA_TRY(dev_alloc(h, &h->d_i8erow, (size_t)ip.NRG * 8));
        LCBA_TRY(dev_alloc(h, &h->d_i8gate, 1));
        LCBA_TRY(dev_alloc(h, &h->d_i8mrow, (size_t)ip.NRG * 8));
        LCBA_CUDA(h, cudaMemsetAsync(h->d_i8gate, 0, sizeof(int), st));
        {
          const char* ge = getenv("LCBA_I8_GUARD");
          h->i8_guard = !(ge && atoi(ge) == 0);
        }
      }
      bool pre = false;
      if (!h->use_i8) {
        int rp = C * 12 + 2;
        while (rp % 16 != 4) ++rp;
        const size_t need = (size_t)(P + 1) * 3 * rp * 8;
        size_t fr = 0, tot = 0;
        const char* pe = getenv("LCBA_MMA_PRE");
        pre = cudaMemGetInfo(&fr, &tot) == cudaSuccess && need < fr / 3 && !(pe && atoi(pe) == 0);
        if (pre) LCBA_TRY(dev_alloc(h, &h->d_Yg, need / 8));
      }
      h->mplan = make_mma_plan(C, h->sm_count, h->smem_optin - 2048, !pre);
      LCBA_TRY(dev_alloc(h, &h->d_mkinds, h->mplan.kinds.size()));
      LCBA_CUDA(h, cudaMemcpyAsync(h->d_mkinds, h->mplan.kinds.data(), h->mplan.kinds.size() * sizeof(MmaKind),
                                   cudaMemcpyHostToDevice, st));
      h->camn_pb = std::max(1, 256 / C);
      h->camn_grid = (int)std::max<long long>(1, std::min<long long>((P + h->camn_pb - 1) / h->camn_pb,
                                                                    (long long)h->sm_count));
      LCBA_TRY(dev_alloc(h, &h->d_Upart, (size_t)h->camn_grid * C * CAMN_VALS));
      LCBA_TRY(dev_alloc(h, &h->d_U, (size_t)C * CAMN_VALS));
      max_slices = std::max(max_slices, h->mplan.nslices);
      h->use_mma = true;
    }
  }
  // dense linearisation (k_linearize_dense, U_c included): tensor-path rigs without repeated pairs
  h->use_dense = h->use_mma && h->n_pairs == N;
  if (h->use_dense) {
    h->dp_pb = DP_THREADS / C;
    const long long ntiles = (P + h->dp_pb - 1) / h->dp_pb;
    h->dp_grid_lin = (int)std::max<long long>(1, std::min<long long>(ntiles, (long long)h->sm_count));
    LCBA_TRY(dev_alloc(h, &h->d_dpart, (size_t)h->dp_grid_lin * C * DP_CAM_VALS));
    LCBA_TRY(dev_alloc(h, &h->d_dred, (size_t)C * DP_CAM_VALS));
  }
  {
    // LCBA_PT_PASSES=0 runs the observation-major kernels on rigs without repeated pairs (tests)
    const char* env = getenv("LCBA_PT_PASSES");
    h->use_pt = h->n_pairs == N && !(env && atoi(env) == 0);
    h->ptp_grid = (int)std::max<long long>(1, std::min<long long>(nblk(P, PT_THREADS), (long long)h->sm_count * 2));
  }
  LCBA_TRY(dev_alloc(h, &h->d_Spart, h->plan.part_stride * max_slices));
  h->d_stats = nullptr;
  if (getenv("LCBA_SCHUR_STATS"))
    LCBA_TRY(dev_alloc(h, &h->d_stats, (size_t)std::max(std::max(h->plan.nslices * h->plan.nkinds,
                                                                 h->use_mma ? h->mplan.nslices * h->mplan.nkinds : 0),
                                                        256) * 4));
  LCBA_CUDA(h, cudaStreamSynchronize(st));
  h->have_problem = true;
  return LCBA_OK;
}

extern "C" int lcba_set_params(lcba_t* h, const double* cams, const double* pts) {
  if (!h || !h->have_problem) { set_error(h, "lcba_set_params: no problem set"); return LCBA_E_STATE; }
  if (!cams || !pts) { set_error(h, "lcba_set_params: null pointer"); return LCBA_E_ARG; }
  cudaSetDevice(h->device);
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_cams[h->cur], cams, (size_t)h->C * NCP * 8, cudaMemcpyHostToDevice, h->stream));
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_pts[h->cur], pts, (size_t)h->P * 3 * 8, cudaMemcpyHostToDevice, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  return LCBA_OK;
}

extern "C" int lcba_set_fixed(lcba_t* h, const uint8_t* cam_fixed, const uint8_t* pt_fixed) {
  if (!h || !h->have_problem) { set_error(h, "lcba_set_fixed: no problem set"); return LCBA_E_STATE; }
  cudaSetDevice(h->device);
  const size_t nc = (size_t)h->C * NCP;
  long long nch = 0, nph = 0;
  uint32_t chk = 0;
  if (cam_fixed) {
    for (size_t i = 0; i < nc; ++i)
      if (cam_fixed[i]) { ++nch; chk = chk * 31u + (uint32_t)(i + 1); }
    LCBA_CUDA(h, cudaMemcpyAsync(h->d_cam_fixed, cam_fixed, nc, cudaMemcpyHostToDevice, h->stream));
  } else if (h->n_cam_held) {
    LCBA_CUDA(h, cudaMemsetAsync(h->d_cam_fixed, 0, nc, h->stream));
  }
  if (pt_fixed) {
    for (long long p = 0; p < h->P; ++p) nph += pt_fixed[p] != 0;
    LCBA_CUDA(h, cudaMemcpyAsync(h->d_pt_fixed, pt_fixed, (size_t)h->P, cudaMemcpyHostToDevice, h->stream));
  } else if (h->n_pt_held) {
    LCBA_CUDA(h, cudaMemsetAsync(h->d_pt_fixed, 0, (size_t)h->P, h->stream));
  }
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  if (cam_fixed) h->h_cam_fixed.assign(cam_fixed, cam_fixed + nc); else h->h_cam_fixed.clear();
  if (pt_fixed) h->h_pt_fixed.assign(pt_fixed, pt_fixed + h->P); else h->h_pt_fixed.clear();
  h->n_cam_held = nch;
  h->n_pt_held = nph;
  h->cam_fixed_sum = (double)chk;
  return LCBA_OK;
}

static const uint8_t* cam_mask(const lcba_t* h) { return h->masks_on ? h->d_cam_fixed : nullptr; }
static const uint8_t* pt_mask(const lcba_t* h) { return h->masks_on ? h->d_pt_fixed : nullptr; }

extern "C" int lcba_set_bounds(lcba_t* h, const double* cam_lb, const double* cam_ub, const double* pt_lb,
                               const double* pt_ub) {
  if (!h || !h->have_problem) { set_error(h, "lcba_set_bounds: no problem set"); return LCBA_E_STATE; }
  const size_t nc = (size_t)h->C * NCP, n = nc + (size_t)h->P * 3;
  if (!cam_lb && !cam_ub && !pt_lb && !pt_ub) {
    h->h_lb.clear(); h->h_ub.clear();
    h->has_bounds = false;
    return LCBA_OK;
  }
  std::vector<double> lb(n, -INFINITY), ub(n, INFINITY);
  if (cam_lb) std::copy(cam_lb, cam_lb + nc, lb.begin());
  if (cam_ub) std::copy(cam_ub, cam_ub + nc, ub.begin());
  if (pt_lb) std::copy(pt_lb, pt_lb + (n - nc), lb.begin() + nc);
  if (pt_ub) std::copy(pt_ub, pt_ub + (n - nc), ub.begin() + nc);
  for (size_t i = 0; i < n; ++i)
    if (std::isnan(lb[i]) || std::isnan(ub[i])) { set_error(h, "lcba_set_bounds: a bound is NaN"); return LCBA_E_ARG; }
  h->h_lb.swap(lb);
  h->h_ub.swap(ub);
  h->has_bounds = true;
  return LCBA_OK;
}

// find_active_constraints (scipy/optimize/_lsq/common.py:414-456) of one entry: -1 lower, 1 upper, 0 neither
static int active_of(double x, double lb, double ub, double rtol) {
  if (rtol == 0.0) return x >= ub ? 1 : (x <= lb ? -1 : 0);
  const double ld = x - lb, ud = ub - x;
  int a = 0;
  if (std::isfinite(lb) && ld <= std::min(ud, rtol * std::max(1.0, std::fabs(lb)))) a = -1;
  if (std::isfinite(ub) && ud <= std::min(ld, rtol * std::max(1.0, std::fabs(ub)))) a = 1;
  return a;
}

// the box the solver sees: held entries (and every camera entry under fix_cameras) unbounded
static void effective_bounds(const lcba_t* h, bool cams_held, std::vector<double>& lb, std::vector<double>& ub) {
  const size_t nc = (size_t)h->C * NCP, n = nc + (size_t)h->P * 3;
  lb = h->h_lb; ub = h->h_ub;
  for (size_t i = 0; i < n; ++i) {
    const bool held = i < nc ? (cams_held || (!h->h_cam_fixed.empty() && h->h_cam_fixed[i]))
                             : (!h->h_pt_fixed.empty() && h->h_pt_fixed[(i - nc) / 3]);
    if (held) { lb[i] = -INFINITY; ub[i] = INFINITY; }
  }
}

static int download_x(lcba_t* h, std::vector<double>& x) {
  const size_t nc = (size_t)h->C * NCP;
  x.resize(nc + (size_t)h->P * 3);
  LCBA_CUDA(h, cudaMemcpyAsync(x.data(), h->d_cams[h->cur], nc * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaMemcpyAsync(x.data() + nc, h->d_pts[h->cur], (size_t)h->P * 3 * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  return LCBA_OK;
}

// checksum of the camera part [0, nc) of a box: equal boxes give equal sums on every rank
static double cam_box_sum(const double* lb, const double* ub, size_t nc) {
  uint32_t chk = 2166136261u;
  for (size_t i = 0; i < nc; ++i) {
    uint64_t bits[2];
    memcpy(&bits[0], &lb[i], 8);
    memcpy(&bits[1], &ub[i], 8);
    for (int k = 0; k < 2; ++k) chk = (chk ^ (uint32_t)(bits[k] ^ (bits[k] >> 32))) * 16777619u;
  }
  return (double)chk;
}

// Local part of a bounded solve's set-up: the effective box and the current x.  flags: 1 = a finite bound on a free
// entry (the bounded loop runs), 2 = lb >= ub on such an entry, 4 = x outside the box there, 8 = x outside or on the
// boundary there.  cam_sum: checksum of the camera part of the box (must be the same on every rank of a sharded job;
// a handle without bounds has the all-infinite box, so its sum equals that of a rank with infinite camera bounds).
struct BoxSetup { std::vector<double> x, lb, ub; int flags = 0; double cam_sum = 0.0; };
static int box_setup(lcba_t* h, bool cams_held, BoxSetup& b) {
  const size_t nc = (size_t)h->C * NCP;
  b.flags = 0;
  b.x.clear();
  if (!h->has_bounds) {
    b.lb.clear(); b.ub.clear();
    const std::vector<double> lo(nc, -INFINITY), hi(nc, INFINITY);
    b.cam_sum = cam_box_sum(lo.data(), hi.data(), nc);
    return LCBA_OK;
  }
  effective_bounds(h, cams_held, b.lb, b.ub);
  LCBA_TRY(download_x(h, b.x));
  const size_t n = b.x.size();
  b.cam_sum = cam_box_sum(b.lb.data(), b.ub.data(), nc);
  for (size_t i = 0; i < n; ++i) {
    const double l = b.lb[i], u = b.ub[i];
    if (!std::isfinite(l) && !std::isfinite(u)) continue;
    b.flags |= 1;
    if (!(l < u)) b.flags |= 2;
    else if (!(b.x[i] >= l && b.x[i] <= u)) b.flags |= 4 | 8;
    else if (!(b.x[i] > l && b.x[i] < u)) b.flags |= 8;
  }
  return LCBA_OK;
}

// Device side of a bounded solve: buffers on first use, the box, and (move_x) x0 moved by
// make_strictly_feasible(x0, lb, ub, rstep=1e-10) as least_squares does before trf_bounds.
static int box_upload(lcba_t* h, BoxSetup& b, bool move_x) {
  const size_t nc = (size_t)h->C * NCP, n = nc + (size_t)h->P * 3;
  if (b.lb.empty()) {            // no bounds on this rank while another rank has some: the all-infinite box
    b.lb.assign(n, -INFINITY);
    b.ub.assign(n, INFINITY);
    move_x = false;
  }
  if (!h->d_blb) {
    LCBA_TRY(dev_alloc(h, &h->d_blb, n));
    LCBA_TRY(dev_alloc(h, &h->d_bub, n));
    LCBA_TRY(dev_alloc(h, &h->d_bsd, n));
    LCBA_TRY(dev_alloc(h, &h->d_bdh, n));
    LCBA_TRY(dev_alloc(h, &h->d_bp, n));
    LCBA_TRY(dev_alloc(h, &h->d_br, n));
    LCBA_TRY(dev_alloc(h, &h->d_bred, 32));
    LCBA_TRY(dev_alloc(h, &h->d_bnd, 1));
  }
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_blb, b.lb.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_bub, b.ub.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
  if (move_x) {
    const double rstep = 1e-10;
    bool moved = false;
    for (size_t i = 0; i < n; ++i) {
      const double l = b.lb[i], u = b.ub[i];
      const int a = active_of(b.x[i], l, u, rstep);
      double xn = b.x[i];
      if (a == -1) xn = l + rstep * std::max(1.0, std::fabs(l));
      else if (a == 1) xn = u - rstep * std::max(1.0, std::fabs(u));
      if (xn < l || xn > u) xn = 0.5 * (l + u);
      if (xn != b.x[i]) { b.x[i] = xn; moved = true; }
    }
    if (moved) {
      LCBA_CUDA(h, cudaMemcpyAsync(h->d_cams[h->cur], b.x.data(), nc * 8, cudaMemcpyHostToDevice, h->stream));
      LCBA_CUDA(h, cudaMemcpyAsync(h->d_pts[h->cur], b.x.data() + nc, (n - nc) * 8, cudaMemcpyHostToDevice, h->stream));
    }
  }
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  return LCBA_OK;
}

extern "C" int lcba_get_active_mask(lcba_t* h, double rtol, int8_t* out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_get_active_mask: no problem set"); return LCBA_E_STATE; }
  if (!out) { set_error(h, "lcba_get_active_mask: out is NULL"); return LCBA_E_ARG; }
  cudaSetDevice(h->device);
  const size_t n = (size_t)h->C * NCP + (size_t)h->P * 3;
  if (!h->has_bounds) { memset(out, 0, n); return LCBA_OK; }
  std::vector<double> x, lb, ub;
  effective_bounds(h, h->fix_cameras != 0, lb, ub);
  LCBA_TRY(download_x(h, x));
  for (size_t i = 0; i < n; ++i) out[i] = (int8_t)active_of(x[i], lb[i], ub[i], rtol);
  return LCBA_OK;
}

// per-entry vectors in the bounded loop: 1 / d and diag_h in place of the Jacobi scale and nothing
static const double* sd_c(const lcba_t* h) { return h->bounded ? h->d_bsd : h->d_scl_c; }
static const double* sd_p(const lcba_t* h) { return h->bounded ? h->d_bsd + (size_t)h->C * NCP : h->d_scl_p; }
static const double* dh_c(const lcba_t* h) { return h->bounded ? h->d_bdh : nullptr; }
static const double* dh_p(const lcba_t* h) { return h->bounded ? h->d_bdh + (size_t)h->C * NCP : nullptr; }

extern "C" int lcba_get_params(lcba_t* h, double* cams_out, double* pts_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_get_params: no problem set"); return LCBA_E_STATE; }
  cudaSetDevice(h->device);
  if (cams_out)
    LCBA_CUDA(h, cudaMemcpyAsync(cams_out, h->d_cams[h->cur], (size_t)h->C * NCP * 8, cudaMemcpyDeviceToHost, h->stream));
  if (pts_out)
    LCBA_CUDA(h, cudaMemcpyAsync(pts_out, h->d_pts[h->cur], (size_t)h->P * 3 * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  return LCBA_OK;
}

// ------------------------------------------------------------------------------ row-wise API
static int rows_call(lcba_t* h, int64_t M, const double* a, int acols, const double* b, int bcols,
                     double* out, int ocols, int which) {
  if (!h) return LCBA_E_ARG;
  if (M < 0 || (M > 0 && (!a || !b || !out))) { set_error(h, "null pointer or negative size"); return LCBA_E_ARG; }
  if (M == 0) return LCBA_OK;
  cudaSetDevice(h->device);
  double *da = nullptr, *db = nullptr, *dout = nullptr;
  cudaError_t e;
  auto fail = [&](const char* what) {
    set_error(h, std::string(what) + ": " + cudaGetErrorString(e));
    cudaFree(da); cudaFree(db); cudaFree(dout);
    return LCBA_E_CUDA;
  };
  if ((e = cudaMalloc(&da, (size_t)M * acols * 8)) != cudaSuccess) return fail("cudaMalloc");
  if ((e = cudaMalloc(&db, (size_t)M * bcols * 8)) != cudaSuccess) return fail("cudaMalloc");
  if ((e = cudaMalloc(&dout, (size_t)M * ocols * 8)) != cudaSuccess) return fail("cudaMalloc");
  cudaMemcpyAsync(da, a, (size_t)M * acols * 8, cudaMemcpyHostToDevice, h->stream);
  cudaMemcpyAsync(db, b, (size_t)M * bcols * 8, cudaMemcpyHostToDevice, h->stream);
  if (which == 0) k_rotate_rows<<<nblk(M, 256), 256, 0, h->stream>>>(da, db, dout, M);
  else k_project_rows<<<nblk(M, 256), 256, 0, h->stream>>>(da, db, dout, M);
  h->launches++;
  cudaMemcpyAsync(out, dout, (size_t)M * ocols * 8, cudaMemcpyDeviceToHost, h->stream);
  e = cudaStreamSynchronize(h->stream);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e != cudaSuccess) return fail("rows kernel");
  cudaFree(da); cudaFree(db); cudaFree(dout);
  return LCBA_OK;
}

extern "C" int lcba_rotate(lcba_t* h, int64_t M, const double* pts, const double* rot_vecs, double* out) {
  return rows_call(h, M, pts, 3, rot_vecs, 3, out, 3, 0);
}
extern "C" int lcba_project(lcba_t* h, int64_t M, const double* pts, const double* cams_rows, double* out_uv) {
  return rows_call(h, M, pts, 3, cams_rows, NCP, out_uv, 2, 1);
}

extern "C" int lcba_unproject(lcba_t* h, int64_t M, const double* uv, const double* Z, int64_t nZ,
                              const double* camera_matrix, const double* dist5, const double* rc_ext,
                              const double* tc_ext, double* out_xyz) {
  if (!h) return LCBA_E_ARG;
  if (M < 0 || (nZ != 1 && nZ != M) || !camera_matrix || !dist5 || !rc_ext || !tc_ext ||
      (M > 0 && (!uv || !Z || !out_xyz))) {
    set_error(h, "lcba_unproject: bad argument (Z must have 1 or M entries)");
    return LCBA_E_ARG;
  }
  if (M == 0) return LCBA_OK;
  cudaSetDevice(h->device);
  double par[26];
  memcpy(par, camera_matrix, 9 * 8);
  memcpy(par + 9, dist5, 5 * 8);
  memcpy(par + 14, rc_ext, 9 * 8);
  memcpy(par + 23, tc_ext, 3 * 8);
  double *d_uv = nullptr, *d_Z = nullptr, *d_par = nullptr, *d_out = nullptr;
  cudaError_t e = cudaMallocAsync(&d_uv, (size_t)M * 16, h->stream);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_Z, (size_t)nZ * 8, h->stream);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_par, sizeof(par), h->stream);
  if (e == cudaSuccess) e = cudaMallocAsync(&d_out, (size_t)M * 24, h->stream);
  if (e == cudaSuccess) {
    cudaMemcpyAsync(d_uv, uv, (size_t)M * 16, cudaMemcpyHostToDevice, h->stream);
    cudaMemcpyAsync(d_Z, Z, (size_t)nZ * 8, cudaMemcpyHostToDevice, h->stream);
    cudaMemcpyAsync(d_par, par, sizeof(par), cudaMemcpyHostToDevice, h->stream);
    k_unproject<<<nblk(M, 256), 256, 0, h->stream>>>((const double2*)d_uv, d_Z, (int)nZ, d_par, M, d_out);
    h->launches++;
    cudaMemcpyAsync(out_xyz, d_out, (size_t)M * 24, cudaMemcpyDeviceToHost, h->stream);
    e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
  }
  void* tmp[] = {d_uv, d_Z, d_par, d_out};
  for (void* q : tmp) if (q) cudaFreeAsync(q, h->stream);
  if (e != cudaSuccess) { set_error(h, std::string("lcba_unproject: ") + cudaGetErrorString(e)); return LCBA_E_CUDA; }
  return LCBA_OK;
}

extern "C" int lcba_sparsity_indices(lcba_t* h, int32_t C, int64_t P, int64_t N, const int64_t* cam_idx,
                                     const int64_t* pt_idx, int32_t* indices_out) {
  if (!h) return LCBA_E_ARG;
  if (C <= 0 || P <= 0 || N < 0 || (N > 0 && (!cam_idx || !pt_idx || !indices_out))) {
    set_error(h, "lcba_sparsity_indices: bad argument");
    return LCBA_E_ARG;
  }
  if ((long long)C * NCP + 3 * P >= (1LL << 31)) { set_error(h, "column index exceeds int32"); return LCBA_E_UNSUPPORTED; }
  if (N == 0) return LCBA_OK;
  cudaSetDevice(h->device);
  long long *dc = nullptr, *dp = nullptr;
  int32_t* dout = nullptr;
  cudaError_t e = cudaMalloc(&dc, N * 8);
  if (e == cudaSuccess) e = cudaMalloc(&dp, N * 8);
  if (e == cudaSuccess) e = cudaMalloc(&dout, (size_t)N * 28 * 4);
  if (e == cudaSuccess) {
    cudaMemcpyAsync(dc, cam_idx, N * 8, cudaMemcpyHostToDevice, h->stream);
    cudaMemcpyAsync(dp, pt_idx, N * 8, cudaMemcpyHostToDevice, h->stream);
    k_sparsity_indices<<<nblk(N * 28, 256), 256, 0, h->stream>>>(dc, dp, N, C, dout);
    h->launches++;
    cudaMemcpyAsync(indices_out, dout, (size_t)N * 28 * 4, cudaMemcpyDeviceToHost, h->stream);
    e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
  }
  cudaFree(dc); cudaFree(dp); cudaFree(dout);
  if (e != cudaSuccess) { set_error(h, std::string("lcba_sparsity_indices: ") + cudaGetErrorString(e)); return LCBA_E_CUDA; }
  return LCBA_OK;
}

// ------------------------------------------------------------------------------ evaluation
static int build_tables(lcba_t* h, int which) {
  KL(h, "cam_tables", k_cam_tables<<<1, 64, 0, h->stream>>>(h->d_cams[which], h->d_tab[which], h->C));
  return LCBA_OK;
}

// sum r^2 of buffer set `which` -> d_red[0] (all-reduced unless `local`); optional residual output
static int run_residual(lcba_t* h, int which, double2* r_out, bool local = false) {
  const size_t smem = (size_t)h->C * CAMTAB * 8;
  if (h->use_pt && !r_out) {
    KL(h, "residual", k_residual_pt<<<h->ptp_grid, PT_THREADS, smem, h->stream>>>(
          h->d_tab[which], h->d_pts[which], h->d_uv, h->d_w, h->d_obs_start, h->d_mask, h->P, h->C, h->d_part));
    KL(h, "reduce", k_reduce_scalars<<<1, 256, 0, h->stream>>>(h->d_part, h->ptp_grid, 1, h->d_red, 1));
    return local ? LCBA_OK : allreduce(h, h->d_red, 1, NCCL_SUM);
  }
  KL(h, "residual", k_residual<<<h->obs_grid, 256, smem, h->stream>>>(
        h->d_tab[which], h->d_pts[which], h->d_uv, h->d_cam, h->d_pt, h->d_w, h->d_perm, h->N, h->C,
        r_out, h->d_part));
  KL(h, "reduce", k_reduce_scalars<<<1, 256, 0, h->stream>>>(h->d_part, h->obs_grid, 1, h->d_red, 1));
  return local ? LCBA_OK : allreduce(h, h->d_red, 1, NCCL_SUM);
}

static int upload_x_to(lcba_t* h, const double* x, int which) {
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_cams[which], x, (size_t)h->C * NCP * 8, cudaMemcpyHostToDevice, h->stream));
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_pts[which], x + (size_t)h->C * NCP, (size_t)h->P * 3 * 8,
                               cudaMemcpyHostToDevice, h->stream));
  return LCBA_OK;
}

extern "C" int lcba_residuals(lcba_t* h, const double* x_or_null, double* r_out, double* cost_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_residuals: no problem set"); return LCBA_E_STATE; }
  cudaSetDevice(h->device);
  int which = h->cur;
  if (x_or_null) { which = 1 - h->cur; LCBA_TRY(upload_x_to(h, x_or_null, which)); }
  LCBA_TRY(build_tables(h, which));
  if (r_out && !h->d_rout) LCBA_TRY(dev_alloc(h, &h->d_rout, (size_t)h->N));
  LCBA_TRY(run_residual(h, which, r_out ? h->d_rout : nullptr, /*local=*/cost_out == nullptr));
  double ss = 0;
  LCBA_CUDA(h, cudaMemcpyAsync(&ss, h->d_red, 8, cudaMemcpyDeviceToHost, h->stream));
  if (r_out) LCBA_CUDA(h, cudaMemcpyAsync(r_out, h->d_rout, (size_t)h->N * 16, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  LCBA_TRY(check_launch(h, "lcba_residuals"));
  if (cost_out) *cost_out = 0.5 * ss;
  return LCBA_OK;
}

static int run_jacobian_blocks(lcba_t* h, int which) {
  const size_t smem = ((size_t)((h->C * CAMTAB + 1) & ~1) + (size_t)(JB_THREADS / 32) * JB_LD * JB_STAGE) * 8;
  const long long groups = (h->N + 31) / 32;
  const int grid = (int)std::min<long long>((groups + 7) / 8, (long long)h->sm_count * 4);
  KL(h, "jacobian_blocks", k_jacobian_blocks<<<grid, JB_THREADS, smem, h->stream>>>(
        h->d_tab[which], h->d_pts[which], h->d_uv, h->d_cam, h->d_pt, h->d_w, h->d_perm, h->N, h->C,
        h->d_rout, h->d_Jc, h->d_Jp));
  return LCBA_OK;
}

static int ensure_jac_buffers(lcba_t* h) {
  if (!h->d_rout) LCBA_TRY(dev_alloc(h, &h->d_rout, (size_t)h->N));
  if (!h->d_Jc) LCBA_TRY(dev_alloc(h, &h->d_Jc, (size_t)h->N * 22));
  if (!h->d_Jp) LCBA_TRY(dev_alloc(h, &h->d_Jp, (size_t)h->N * 6));
  return LCBA_OK;
}

extern "C" int lcba_jacobian_blocks(lcba_t* h, const double* x_or_null, double* Jc, double* Jp) {
  if (!h || !h->have_problem) { set_error(h, "lcba_jacobian_blocks: no problem set"); return LCBA_E_STATE; }
  cudaSetDevice(h->device);
  int which = h->cur;
  if (x_or_null) { which = 1 - h->cur; LCBA_TRY(upload_x_to(h, x_or_null, which)); }
  LCBA_TRY(build_tables(h, which));
  LCBA_TRY(ensure_jac_buffers(h));
  LCBA_TRY(run_jacobian_blocks(h, which));
  if (Jc) LCBA_CUDA(h, cudaMemcpyAsync(Jc, h->d_Jc, (size_t)h->N * 22 * 8, cudaMemcpyDeviceToHost, h->stream));
  if (Jp) LCBA_CUDA(h, cudaMemcpyAsync(Jp, h->d_Jp, (size_t)h->N * 6 * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  return check_launch(h, "lcba_jacobian_blocks");
}

// ------------------------------------------------------------------------------ solver passes
// Reduce the columns of a bounded pass's partials (k_reduce_ops) into out[0..K) and all-reduce them over the ranks.
static int reduce_ops(lcba_t* h, const double* part, int nblocks, int K, int nsum, int nmax, double* out) {
  KL(h, "reduce", k_reduce_ops<<<K, 256, 0, h->stream>>>(part, nblocks, K, nsum, nmax, out));
  if (nsum) LCBA_TRY(allreduce(h, out, nsum, NCCL_SUM));
  if (nmax) LCBA_TRY(allreduce(h, out + nsum, nmax, NCCL_MAX));
  if (K > nsum + nmax) LCBA_TRY(allreduce(h, out + nsum + nmax, K - nsum - nmax, NCCL_MIN));
  return LCBA_OK;
}

static int pass_linearize(lcba_t* h, int first) {
  NvtxRange nvtx_("lcba:linearize");
  const int C = h->C, w = h->cur;
  LCBA_TRY(build_tables(h, w));
  if (h->use_dense) {
    // one pass: V, g_p per point; g_c, diag(J^T J) AND the camera blocks U_c per camera; cost
    const size_t smem = dense_lin_smem_doubles(C) * 8;
    KL(h, "linearize", k_linearize_dense<<<h->dp_grid_lin, DP_THREADS, smem, h->stream>>>(
          h->d_tab[w], h->d_pts[w], h->d_uv, h->d_w, h->d_obs_start, h->d_mask, h->P, C, h->dp_pb,
          h->d_Vg, h->d_dpart, h->d_part));
    KL(h, "reduce", k_reduce_cols<<<nblk(C * DP_CAM_VALS, RC_COLS), RC_COLS * RC_ROWS, 0, h->stream>>>(
          h->d_dpart, h->dp_grid_lin, C * DP_CAM_VALS, h->d_dred));
    KL(h, "reduce", k_dense_cam_unpack<<<nblk(C * DP_CAM_VALS, 128), 128, 0, h->stream>>>(
          h->d_dred, C, h->d_camsum, h->d_U));
    KL(h, "reduce", k_reduce_scalars<<<1, 256, 0, h->stream>>>(h->d_part, h->dp_grid_lin, 1,
                                                               h->d_camsum + C * CAMSUM, 1));
  } else {
  const size_t smem = linearize_smem_doubles(C) * 8;
  KL(h, "linearize", k_linearize<<<h->lin_grid, LIN_THREADS, smem, h->stream>>>(
        h->d_tab[w], h->d_pts[w], h->d_uv, h->d_cam, h->d_pt, h->d_w, h->d_obs_start, h->d_bins,
        h->nbins, C, h->d_Vg, h->d_campart, h->d_part));
  KL(h, "reduce", k_reduce_cols<<<nblk(C * CAMSUM, RC_COLS), RC_COLS * RC_ROWS, 0, h->stream>>>(
        h->d_campart, h->lin_grid, C * CAMSUM, h->d_camsum));
  KL(h, "reduce", k_reduce_scalars<<<1, 256, 0, h->stream>>>(h->d_part, h->lin_grid, 1,
                                                             h->d_camsum + C * CAMSUM, 1));
  }
  if (h->bounded) {
    const size_t nc = (size_t)C * NCP;
    KL(h, "point_prep", k_bnd_point_prep<<<h->pt_grid, 256, 0, h->stream>>>(
          h->d_Vg, h->d_pts[w], h->d_scl_p, h->d_gt_p, h->P, first, pt_mask(h), h->d_blb + nc, h->d_bub + nc,
          h->d_bsd + nc, h->d_bdh + nc, h->d_part));
    LCBA_TRY(reduce_ops(h, h->d_part, h->pt_grid, BPP_K, 4, 1, h->d_bred));
    LCBA_TRY(allreduce(h, h->d_camsum, (size_t)C * CAMSUM + 1, NCCL_SUM));
    KL(h, "ctl", k_bnd_ctl_lin<<<1, 256, 0, h->stream>>>(h->d_camsum, h->d_cams[w], h->d_scl_c, h->d_gt_c, h->d_g_c, C,
                                                         cam_mask(h), h->d_blb, h->d_bub, h->d_bsd, h->d_bdh,
                                                         h->d_bred, h->d_ctl, h->d_bnd, first));
    return check_launch(h, "linearize pass");
  }
  // per-point scaling does not depend on the camera sums: run it first so that ONE sum
  // all-reduce carries [camera sums | cost | point sums] and one max all-reduce |g|_inf
  double* pp = h->d_camsum + C * CAMSUM + 1;
  KL(h, "point_prep", k_point_prep<<<h->pt_grid, 256, 0, h->stream>>>(
        h->d_Vg, h->d_pts[w], h->d_scl_p, h->d_gt_p, h->P, first, pt_mask(h), h->d_part));
  KL(h, "reduce", k_reduce_scalars<<<PP_K, 256, 0, h->stream>>>(h->d_part, h->pt_grid, PP_K, pp, 3));
  LCBA_TRY(allreduce(h, h->d_camsum, (size_t)C * CAMSUM + 1 + 3, NCCL_SUM));
  LCBA_TRY(allreduce(h, pp + 3, 1, NCCL_MAX));
  KL(h, "ctl", k_ctl_lin<<<1, 256, 0, h->stream>>>(h->d_camsum, h->d_cams[w], h->d_scl_c, h->d_gt_c,
                                                   h->d_g_c, C, h->d_ctl, first, h->fix_cameras, cam_mask(h),
                                                   h->shared_intr));
  KL(h, "ctl", k_ctl_lin2<<<1, 1, 0, h->stream>>>(pp, h->d_ctl, first));
  return check_launch(h, "linearize pass");
}

static int pass_jdot(lcba_t* h) {
  NvtxRange nvtx_("lcba:jdot");
  const int C = h->C, w = h->cur;
  const size_t smem = ((size_t)C * CAMTAB + (size_t)C * NCP) * 8;
  if (h->use_pt) {
    KL(h, "jdot", k_jdot_pt<<<h->ptp_grid, PT_THREADS, smem, h->stream>>>(
          h->d_tab[w], h->d_pts[w], h->d_w, h->d_obs_start, h->d_mask, h->d_gt_c, h->d_gt_p, h->P, C, h->d_part));
    KL(h, "reduce", k_reduce_scalars<<<1, 256, 0, h->stream>>>(h->d_part, h->ptp_grid, 1, h->d_red, 1));
  } else {
  KL(h, "jdot", k_jdot<<<h->obs_grid, 256, smem, h->stream>>>(
        h->d_tab[w], h->d_pts[w], h->d_cam, h->d_pt, h->d_w, h->d_gt_c, h->d_gt_p, h->N, C, h->d_part));
  KL(h, "reduce", k_reduce_scalars<<<1, 256, 0, h->stream>>>(h->d_part, h->obs_grid, 1, h->d_red, 1));
  }
  LCBA_TRY(allreduce(h, h->d_red, 1, NCCL_SUM));
  KL(h, "ctl", k_ctl_reg<<<1, 1, 0, h->stream>>>(h->d_red, h->d_ctl, h->bounded ? &h->d_bnd->dhg2 : nullptr));
  return check_launch(h, "jdot pass");
}

// int8 Schur path, the digit planes: row maxima and exponents of Y (after k_point_factor), then the planes
static void launch_i8_rowexp(lcba_t* h) {
  const int C = h->C, w = h->cur, RP = h->i8plan.NRG * 8;
  const size_t smem_rm = ((size_t)I8_GROUP_CAMS * CAMTAB + 192) * 4;
  KL(h, "i8_rowmax", k_i8_rowmax<<<dim3(h->i8_gx_max, h->i8_groups), 192, smem_rm, h->stream>>>(
        h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, C, RP, h->d_i8rmax));
  KL(h, "i8_rowmax", k_i8_rowexp<<<nblk(RP, 128), 128, 0, h->stream>>>(h->d_i8rmax, h->i8_gx_max, NCP * C + 1, RP,
                                                                 h->d_i8erow, h->d_i8mrow));
}
// ref: k_i8_make_ref, only from lcba_debug_i8_make
static void launch_i8_make(lcba_t* h, bool ref) {
  const int C = h->C, w = h->cur, NRG = h->i8plan.NRG;
  if (ref)
    KL(h, "make_Y", k_i8_make_ref<<<dim3(h->i8_gx_make_ref, h->i8_groups), 192, i8_make_ref_smem_bytes(), h->stream>>>(
          h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, C, NRG, h->d_i8erow,
          h->d_i8planes));
  else
    KL(h, "make_Y", k_i8_make<<<dim3(h->i8_gx_make, h->i8_groups), I8_MK_THREADS, i8_make_smem_bytes(), h->stream>>>(
          h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, C, NRG, h->d_i8erow,
          h->d_i8planes));
}

static int pass_schur(lcba_t* h, const double* lam_host_or_null) {
  NvtxRange nvtx_("lcba:schur");
  const int C = h->C, w = h->cur, n = C * NCP;
  const SchurPlan& pl = h->plan;
  const double lam_arg = lam_host_or_null ? *lam_host_or_null : 0.0;
  const Ctl* ctl_arg = lam_host_or_null ? nullptr : h->d_ctl;
  KL(h, "point_factor", k_point_factor<<<nblk(h->P, 256), 256, 0, h->stream>>>(
        h->d_Vg, sd_p(h), lam_arg, ctl_arg, h->P, pt_mask(h), dh_p(h), h->d_Lz));
  if (h->use_mma) {
    // dense rigs: SYRK on the FP64 tensor path + the camera blocks U from their own pass
    const MmaPlan& mp = h->mplan;
    if (!h->use_dense) {      // dense passes: U_c already came out of k_linearize_dense
    const size_t smem_u = ((size_t)((C * CAMTAB + 1) & ~1) + (size_t)h->camn_pb * C) * 8;
    KL(h, "cam_normal", k_cam_normal<<<h->camn_grid, 256, smem_u, h->stream>>>(
          h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->P, C, h->camn_pb, h->d_Upart));
    KL(h, "reduce", k_reduce_cols<<<nblk(C * CAMN_VALS, RC_COLS), RC_COLS * RC_ROWS, 0, h->stream>>>(
          h->d_Upart, h->camn_grid, C * CAMN_VALS, h->d_U));
    }
    const int nt = (NCP * C + 1 + 7) / 8, last = nt - 6 * ((nt + 5) / 6 - 1);
    if (h->use_i8) {
      // 5th-generation tensor cores: digit planes of Y, exact int8 x int8 -> int32 SYRK, FP64 recombination
      const I8Plan& ip = h->i8plan;
      launch_i8_rowexp(h);
      launch_i8_make(h, false);
      KL(h, "schur", k_i8_syrk<<<(unsigned)ip.work.size(), I8_THREADS, ip.smem_bytes, h->stream>>>(
            h->i8maps, h->d_i8work, h->d_i8partial, h->d_fail, h->d_i8progress, ip.window, h->d_stats));
      KL(h, "schur_reduce", k_i8_gather<<<dim3((unsigned)ip.tiles.size(), 16), 256, 0, h->stream>>>(
            h->d_i8partial, h->d_i8tiles, C, ip.cover ? 1 : 0, h->d_i8erow, pl.npairs, h->d_Sred));
      KL(h, "schur_reduce", k_add_cam_blocks<<<nblk(C * 121, 128), 128, 0, h->stream>>>(h->d_U, C, h->d_Sred));
      // rows whose maximum comes from one point far above their Schur diagonal: the DMMA kernel (Y evaluated in
      // place) redoes this pass; both launches return at once unless k_i8_check raised the gate
      if (h->i8_guard) {
        KL(h, "i8_check", k_i8_check<<<1, 256, 0, h->stream>>>(h->d_i8mrow, C, h->d_Sred, h->d_i8gate));
#define LCBA_MMA_GATED(L)                                                                            \
  KL(h, "i8_fallback", (k_schur_mma<L, false><<<dim3(mp.nslices, mp.nkinds), MMA_THREADS, mp.smem_bytes, h->stream>>>( \
          nullptr, h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, h->n_pairs, C, \
          h->d_mkinds, mp.nslices, pl.part_stride, pl.npairs, h->d_Spart, nullptr, h->d_i8gate)))
        switch (last) {
          case 1: LCBA_MMA_GATED(1); break;
          case 2: LCBA_MMA_GATED(2); break;
          case 3: LCBA_MMA_GATED(3); break;
          case 4: LCBA_MMA_GATED(4); break;
          case 5: LCBA_MMA_GATED(5); break;
          default: LCBA_MMA_GATED(6); break;
        }
#undef LCBA_MMA_GATED
        KL(h, "i8_fallback", k_i8_fallback_finish<<<h->sm_count, 256, 0, h->stream>>>(
              h->d_i8gate, h->d_Spart, mp.nslices, pl.part_stride, h->d_U, C, h->d_Sred));
      }
    } else {
    if (h->d_Yg) {
      const int pbk = MAKEY_THREADS / C, rpk = mp.kinds[0].rp;
      const size_t smem_y = ((size_t)((C * CAMTAB + 1) & ~1) + (size_t)3 * pbk * rpk) * 8;
      const int grid_y = (int)std::min<long long>((h->P + pbk - 1) / pbk, (long long)h->sm_count * 5);
      KL(h, "make_Y", k_make_Y<<<grid_y, MAKEY_THREADS, smem_y, h->stream>>>(
            h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, C, mp.kinds[0].rp,
            h->d_Yg));
    }
#define LCBA_MMA_LAUNCH(L)                                                                          \
  do {                                                                                              \
    if (h->d_Yg)                                                                                    \
      KL(h, "schur", (k_schur_mma<L, true><<<dim3(mp.nslices, mp.nkinds), MMA_THREADS, mp.smem_bytes, h->stream>>>( \
            h->d_Yg, h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, h->n_pairs, C, \
            h->d_mkinds, mp.nslices, pl.part_stride, pl.npairs, h->d_Spart, h->d_stats)));          \
    else                                                                                            \
      KL(h, "schur", (k_schur_mma<L, false><<<dim3(mp.nslices, mp.nkinds), MMA_THREADS, mp.smem_bytes, h->stream>>>( \
            nullptr, h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, h->n_pairs, C, \
            h->d_mkinds, mp.nslices, pl.part_stride, pl.npairs, h->d_Spart, h->d_stats)));          \
  } while (0)
    switch (last) {
      case 1: LCBA_MMA_LAUNCH(1); break;
      case 2: LCBA_MMA_LAUNCH(2); break;
      case 3: LCBA_MMA_LAUNCH(3); break;
      case 4: LCBA_MMA_LAUNCH(4); break;
      case 5: LCBA_MMA_LAUNCH(5); break;
      default: LCBA_MMA_LAUNCH(6); break;
    }
#undef LCBA_MMA_LAUNCH
    KL(h, "schur_reduce", k_reduce_cols<<<nblk((long long)pl.part_stride, RC_COLS), RC_COLS * RC_ROWS, 0, h->stream>>>(
          h->d_Spart, mp.nslices, (int)pl.part_stride, h->d_Sred));
    KL(h, "schur_reduce", k_add_cam_blocks<<<nblk(C * 121, 128), 128, 0, h->stream>>>(h->d_U, C, h->d_Sred));
    }
  } else {
  dim3 grid(pl.nslices, pl.nkinds);
  // sparse rigs skip duo blocks nobody sees; dense rigs run branch-free
  const bool skip = (double)h->n_pairs < 0.8 * (double)h->P * C;
#define LCBA_SCHUR_LAUNCH(SK, NR)                                                                   \
  KL(h, "schur", (k_schur<SK, NR><<<grid, pl.max_threads, pl.smem_bytes, h->stream>>>(              \
        h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, h->n_pairs, C, \
        h->d_kinds, h->d_hws, pl.nslices, pl.part_stride, pl.npairs, h->d_Spart, h->d_stats)))
  if (pl.cfg != 1) { if (skip) LCBA_SCHUR_LAUNCH(true, 160); else LCBA_SCHUR_LAUNCH(false, 160); }
  else             { if (skip) LCBA_SCHUR_LAUNCH(true, 128); else LCBA_SCHUR_LAUNCH(false, 128); }
#undef LCBA_SCHUR_LAUNCH
  KL(h, "schur_reduce", k_reduce_cols<<<nblk((long long)pl.part_stride, RC_COLS), RC_COLS * RC_ROWS, 0, h->stream>>>(
        h->d_Spart, pl.nslices, (int)pl.part_stride, h->d_Sred));
  }
  LCBA_TRY(allreduce(h, h->d_Sred, pl.part_stride, NCCL_SUM));
  if (h->shared_intr) {
    const int nr = 3 + 8 * C;
    KL(h, "assemble", k_assemble_S_shared<<<nblk((long long)nr * nr, 256), 256, 0, h->stream>>>(
          h->d_Sred, C, pl.npairs, h->d_camsum, h->d_scl_c, h->d_ctl,
          lam_host_or_null ? *lam_host_or_null : 0.0, lam_host_or_null ? 0 : 1, h->d_S, h->d_rhs,
          h->d_scl_red));
  } else {
    KL(h, "assemble", k_assemble_S<<<nblk((long long)n * n, 256), 256, 0, h->stream>>>(
          h->d_Sred, C, pl.npairs, h->d_camsum, sd_c(h), lam_arg, ctl_arg, cam_mask(h), dh_c(h), h->d_S, h->d_rhs));
  }
  return check_launch(h, "schur pass");
}

// grid of k_chol_fused = trailing tiles of the first panel (one tile per CTA), capped at
// LCBA_CHOL_GRID (read once per process, default 64) and the SM count; all CTAs co-resident
static int chol_grid(int n, int sm_count) {
  int tiles = 1;
  if (n > CH_NB) {
    const int ntr = (n + 1 - CH_NB + CH_NB - 1) / CH_NB, ntc = (n - CH_NB + CH_NB - 1) / CH_NB;
    tiles = 0;
    for (int ti = 0; ti < ntr; ++ti) tiles += std::min(ti + 1, ntc);
  }
  static const int cap = getenv("LCBA_CHOL_GRID") ? atoi(getenv("LCBA_CHOL_GRID")) : 64;
  return std::max(1, std::min(tiles, std::min(cap, sm_count)));
}

// Cholesky of S + mu*Dc^2, solve for the camera step
static int pass_camera_solve(lcba_t* h, double mu) {
  NvtxRange nvtx_("lcba:camera_solve");
  const int n = h->shared_intr ? 3 + 8 * h->C : h->C * NCP;
  LCBA_CUDA(h, cudaMemsetAsync(h->d_fail, 0, 2 * sizeof(int), h->stream));
  const double* scl = h->shared_intr ? h->d_scl_red : h->d_scl_c;
  double* out = h->shared_intr ? h->d_pred : h->d_pc;
  {
    KL(h, "chol_copy", k_copy_damped_rhs<<<nblk((long long)(n + 1) * n, 256), 256, 0, h->stream>>>(
          h->d_S, n, mu, scl, h->d_rhs, h->d_Lf));
    const int grid = chol_grid(n, h->sm_count);
    double* A = h->d_Lf;
    int nn = n;
    int* sync = h->d_fail;
    static long long* dbg = nullptr;
    static const bool want_dbg = getenv("LCBA_CHOL_DBG") != nullptr;
    if (want_dbg && !dbg) cudaMalloc(&dbg, 6 * sizeof(long long));
    void* args[] = {(void*)&A, (void*)&nn, (void*)&out, (void*)&sync, (void*)&dbg};
    KL(h, "chol_fused", {
      cudaError_t e = cudaLaunchCooperativeKernel((const void*)k_chol_fused, dim3(grid), dim3(256), args, 0, h->stream);
      if (e != cudaSuccess) {
        set_error(h, std::string("cudaLaunchCooperativeKernel(k_chol_fused): ") + cudaGetErrorString(e));
        return LCBA_E_CUDA;
      }
    });
    if (want_dbg) {
      long long tmh[6];
      cudaStreamSynchronize(h->stream);
      cudaMemcpy(tmh, dbg, sizeof(tmh), cudaMemcpyDeviceToHost);
      fprintf(stderr, "chol_fused n=%d grid=%d cycles: factor %lld trsm %lld bar1 %lld update %lld bar2 %lld backsub %lld\n",
              n, grid, tmh[0], tmh[1], tmh[2], tmh[3], tmh[4], tmh[5]);
    }
  }
  if (h->shared_intr)
    KL(h, "expand", k_expand_shared<<<nblk(h->C * NCP, 128), 128, 0, h->stream>>>(h->d_pred, h->C, h->d_pc));
  return check_launch(h, "camera solve");
}

static int pass_backsub(lcba_t* h) {
  NvtxRange nvtx_("lcba:backsub");
  const int C = h->C, w = h->cur;
  if (h->use_pt) {
    const size_t smem = ((size_t)C * CAMTAB + 2 * (size_t)C * NCP) * 8;
    KL(h, "backsub", k_backsub_pt<<<h->ptp_grid, PT_THREADS, smem, h->stream>>>(
          h->d_tab[w], h->d_pts[w], h->d_w, h->d_obs_start, h->d_mask, h->P, C, h->d_Vg, h->d_Lz, sd_p(h),
          h->d_gt_c, h->d_gt_p, h->d_pc, h->d_gn_p, h->d_part));
    KL(h, "reduce", k_reduce_scalars<<<BS_K, 256, 0, h->stream>>>(h->d_part, h->ptp_grid, BS_K, h->d_red, BS_K));
  } else {
  const size_t smem = ((size_t)C * CAMTAB + 2 * (size_t)C * NCP + 2 * LIN_THREADS * 3) * 8;
  KL(h, "backsub", k_backsub<<<h->lin_grid, LIN_THREADS, smem, h->stream>>>(
        h->d_tab[w], h->d_pts[w], h->d_cam, h->d_pt, h->d_w, h->d_obs_start, h->d_bins, h->nbins, C,
        h->d_Vg, h->d_Lz, sd_p(h), h->d_gt_c, h->d_gt_p, h->d_pc, h->d_gn_p, h->d_part));
  KL(h, "reduce", k_reduce_scalars<<<BS_K, 256, 0, h->stream>>>(h->d_part, h->lin_grid, BS_K, h->d_red, BS_K));
  }
  LCBA_TRY(allreduce(h, h->d_red, BS_K, NCCL_SUM));
  if (h->bounded) {   // B_S gains S^T diag_h S: added to the Gram totals JAA, JAB, JBB
    const int nc = C * NCP;
    KL(h, "bnd_gram", k_bnd_gram<<<h->pt_grid, 256, 0, h->stream>>>(
          h->d_g_c, h->d_pc, h->d_Vg, h->d_gn_p, h->d_bsd, h->d_bdh, nc, nc + h->P * 3, h->rank == 0, h->d_part));
    LCBA_TRY(reduce_ops(h, h->d_part, h->pt_grid, 3, 3, 0, h->d_bred + 6));
    KL(h, "ctl", k_bnd_gram_add<<<1, 1, 0, h->stream>>>(h->d_red, h->d_bred + 6));
  }
  KL(h, "ctl", k_ctl_sub<<<1, 256, 0, h->stream>>>(h->d_red, h->d_g_c, h->d_gt_c, h->d_pc, sd_c(h), C,
                                                   h->d_ctl, h->d_fail, h->d_coef, h->shared_intr));
  return check_launch(h, "backsub pass");
}

static int pass_trial(lcba_t* h) {
  NvtxRange nvtx_("lcba:trial");
  const int w = h->cur, t = 1 - h->cur;
  const long long nc = (long long)h->C * NCP, np = h->P * 3;
  if (h->bounded) {
    // select_step: the subspace step, its reflection off the first bound it crosses (the reflection's J pass only
    // does work when the step leaves the box) and the anti-gradient; then the strictly feasible trial point
    const int C = h->C;
    const long long n = nc + np;
    KL(h, "bnd_select", k_bnd_a<<<h->pt_grid, 256, 0, h->stream>>>(
          h->d_cams[w], h->d_pts[w], h->d_gt_c, h->d_gt_p, h->d_pc, h->d_gn_p, h->d_coef, h->d_blb, h->d_bub, (int)nc,
          n, h->d_bp, h->d_part));
    LCBA_TRY(reduce_ops(h, h->d_part, h->pt_grid, 2, 0, 1, h->d_bred + 9));
    KL(h, "ctl", k_bnd_ctl_a<<<1, 1, 0, h->stream>>>(h->d_bred + 9, h->d_bnd));
    KL(h, "bnd_select", k_bnd_b<<<h->pt_grid, 256, 0, h->stream>>>(
          h->d_cams[w], h->d_pts[w], h->d_g_c, h->d_Vg, h->d_bp, h->d_bsd, h->d_bdh, h->d_blb, h->d_bub, (int)nc, n,
          h->rank == 0, h->d_bnd, h->d_br, h->d_part));
    LCBA_TRY(reduce_ops(h, h->d_part, h->pt_grid, BB_K, 5, 0, h->d_bred + 11));
    const size_t smem = ((size_t)C * CAMTAB + 2 * (size_t)C * NCP) * 8;
    KL(h, "bnd_jdot", k_bnd_jdot<<<h->obs_grid, 256, smem, h->stream>>>(
          h->d_tab[w], h->d_pts[w], h->d_cam, h->d_pt, h->d_w, h->d_bp, h->d_br, h->N, C, h->d_bnd, h->d_part));
    LCBA_TRY(reduce_ops(h, h->d_part, h->obs_grid, 2, 2, 0, h->d_bred + 17));
    KL(h, "ctl", k_bnd_select<<<1, 1, 0, h->stream>>>(h->d_bred + 11, h->d_bred + 17, h->d_ctl, h->d_bnd));
    KL(h, "make_trial", k_bnd_trial<<<h->pt_grid, 256, 0, h->stream>>>(
          h->d_cams[w], h->d_pts[w], h->d_gt_c, h->d_gt_p, h->d_bp, h->d_blb, h->d_bub, (int)nc, n, h->d_bnd,
          h->d_cams[t], h->d_pts[t]));
  } else {
  KL(h, "make_trial", k_make_trial<<<1, 256, 0, h->stream>>>(h->d_cams[w], h->d_gt_c, h->d_pc, h->d_coef, nc,
                                                             h->d_cams[t]));
  KL(h, "make_trial", k_make_trial<<<h->pt_grid, 256, 0, h->stream>>>(h->d_pts[w], h->d_gt_p, h->d_gn_p,
                                                                      h->d_coef, np, h->d_pts[t]));
  }
  LCBA_TRY(build_tables(h, t));
  LCBA_TRY(run_residual(h, t, nullptr));
  KL(h, "ctl", k_ctl_trial<<<1, 1, 0, h->stream>>>(h->d_red, h->d_ctl, h->d_coef));
  return check_launch(h, "trial pass");
}

static int read_ctl(lcba_t* h) {
  LCBA_CUDA(h, cudaMemcpyAsync(h->h_ctl, h->d_ctl, sizeof(Ctl), cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  if (h->comm && g_peer.ok && *(volatile int*)g_peer.h_fail) {
    set_error(h, "peer all-reduce: a rank did not arrive within the time limit");
    return LCBA_E_NCCL;
  }
  return check_launch(h, "solver");
}

static void add_trace(lcba_t* h, long long it, long long nfev, double cost, double red, double step,
                      double opt, double delta, double reg) {
  if (h->trace.size() >= LCBA_MAX_TRACE) return;
  lcba_trace_row r;
  r.iteration = it; r.nfev = nfev; r.cost = cost; r.cost_reduction = red; r.step_norm = step;
  r.optimality = opt; r.delta = delta; r.reg_term = reg;
  h->trace.push_back(r);
  if (h->iter_cb) h->iter_cb(&h->trace.back(), h->iter_cb_user);
}

extern "C" int lcba_set_iteration_callback(lcba_t* h, lcba_iteration_cb cb, void* user) {
  if (!h) return LCBA_E_ARG;
  h->iter_cb = cb;
  h->iter_cb_user = user;
  return LCBA_OK;
}

// Run a static launch sequence through a CUDA graph (captured on first use, replayed afterwards):
// at 8 GPUs an iteration is ~35 launches of mostly microsecond kernels and the gaps between them are
// a tenth of the step.  Any failure to capture or instantiate (e.g. a driver that cannot capture the
// cooperative Cholesky launch) switches graphs off for the handle and enqueues directly.
template <class F>
static int run_graphed(lcba_t* h, lcba_handle::GraphSlot& slot, int key, bool allowed, F&& enqueue) {
  if (!allowed || !h->use_graphs || h->prof_on) return enqueue();
  if (slot.exec && slot.key != key) { cudaGraphExecDestroy(slot.exec); slot.exec = nullptr; }
  if (!slot.exec) {
    const long long l0 = h->launches;
    if (cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
      cudaGetLastError();
      h->use_graphs = false;
      return enqueue();
    }
    const int rc = enqueue();
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(h->stream, &g);
    if (rc == LCBA_OK && e == cudaSuccess && g) e = cudaGraphInstantiate(&slot.exec, g, 0);
    if (g) cudaGraphDestroy(g);
    if (rc != LCBA_OK || e != cudaSuccess || !slot.exec) {
      cudaGetLastError();
      slot.exec = nullptr;
      h->use_graphs = false;
      h->launches = l0;
      return enqueue();          // nothing was executed during the failed capture
    }
    slot.launches = h->launches - l0;
    slot.key = key;
    h->launches = l0;
  }
  if (cudaGraphLaunch(slot.exec, h->stream) != cudaSuccess) {
    cudaGetLastError();
    h->use_graphs = false;
    return enqueue();
  }
  h->launches += slot.launches;
  h->graph_replays++;
  return LCBA_OK;
}

extern "C" int lcba_solve(lcba_t* h, const lcba_options* opt_in, lcba_result* res) {
  if (!h || !h->have_problem) { set_error(h, "lcba_solve: no problem set"); return LCBA_E_STATE; }
  if (!res) { set_error(h, "lcba_solve: res is NULL"); return LCBA_E_ARG; }
  lcba_options opt;
  if (opt_in) opt = *opt_in; else lcba_default_options(&opt);
  cudaSetDevice(h->device);
  memset(res, 0, sizeof(*res));
  h->trace.clear();
  h->prof.clear();
  h->prof_on = opt.profile != 0;
  const long long launches0 = h->launches, replays0 = h->graph_replays;
  long long pt_held_total = h->n_pt_held;
  h->fix_cameras = opt.fix_cameras ? 1 : 0;
  h->shared_intr = (opt.shared_intrinsics && !h->fix_cameras) ? 1 : 0;
  h->masks_on = true;
  BoxSetup box;
  LCBA_TRY(box_setup(h, h->fix_cameras != 0, box));
  if (h->comm) {
    // total point and held-point counts over the ranks (max_nfev = 100 n_free); the camera mask and the camera
    // bounds must be the same on every rank: max of (count, checksum) and of their negatives, so that every rank
    // sees a mismatch; the box flags of box_setup: max over the ranks (every rank runs the same loop and fails alike)
    double v[10] = {(double)h->P, (double)h->n_pt_held, (double)h->n_cam_held, h->cam_fixed_sum,
                    -(double)h->n_cam_held, -h->cam_fixed_sum, (double)(box.flags & 1), (double)(box.flags & 6),
                    box.cam_sum, -box.cam_sum};
    LCBA_CUDA(h, cudaMemcpyAsync(h->d_red, v, sizeof(v), cudaMemcpyHostToDevice, h->stream));
    LCBA_TRY(allreduce(h, h->d_red, 2, NCCL_SUM));
    LCBA_TRY(allreduce(h, h->d_red + 2, 8, NCCL_MAX));
    LCBA_CUDA(h, cudaMemcpyAsync(v, h->d_red, sizeof(v), cudaMemcpyDeviceToHost, h->stream));
    LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
    h->P_total = (long long)(v[0] + 0.5);
    pt_held_total = (long long)(v[1] + 0.5);
    if (v[2] != -v[4] || v[3] != -v[5]) {
      set_error(h, "lcba_solve: the ranks hold different camera masks (lcba_set_fixed)");
      return LCBA_E_ARG;
    }
    box.flags = (v[6] != 0.0 ? 1 : 0) | (int)v[7];
    if (v[6] != 0.0 && v[8] != -v[9]) {
      set_error(h, "lcba_solve: the ranks hold different camera bounds (lcba_set_bounds)");
      return LCBA_E_ARG;
    }
  }
  h->bounded = false;
  if (box.flags & 1) {
    if (h->fix_cameras || h->shared_intr) {
      set_error(h, "lcba_solve: box bounds together with fix_cameras or shared_intrinsics are not supported");
      return LCBA_E_UNSUPPORTED;
    }
    if (box.flags & 2) {
      set_error(h, "lcba_solve: each lower bound must be strictly less than each upper bound (lcba_set_bounds)");
      return LCBA_E_ARG;
    }
    if (box.flags & 4) {
      set_error(h, "lcba_solve: the initial guess is outside of the bounds (lcba_set_bounds)");
      return LCBA_E_ARG;
    }
    LCBA_TRY(box_upload(h, box, true));
    h->bounded = true;
  }
  if (h->shared_intr && h->n_cam_held) {
    set_error(h, "lcba_solve: a camera mask together with shared_intrinsics is not supported");
    return LCBA_E_UNSUPPORTED;
  }
  {
    static const bool env_off = getenv("LCBA_GRAPH") && atoi(getenv("LCBA_GRAPH")) == 0;
    if (env_off) h->use_graphs = false;
  }
  // Replay from the second solve on a resident problem onwards, where launches matter: single GPU (with NCCL
  // all-reduces captured inside, a replay is SLOWER than direct launches: 4.48 vs 4.28 ms per iteration at 2 GPUs,
  // 2.12 vs 1.80 at 8) and fewer than 8 M observations (above, an iteration is several ms of long kernels: A/B on
  // one box, ring24 x 1 M: 8.06 / 8.36 vs 8.12 / 8.13 ms, and the capture + instantiation of the four graphs
  // would fall into the second solve)
  const bool graphs = h->solves_on_problem >= 1 && !h->comm && h->N < (8LL << 20) && !h->bounded;
  h->solves_on_problem++;
  const int gkey = h->fix_cameras * 2 + h->shared_intr;
  const long long n_cam = h->fix_cameras ? 0 : (h->shared_intr ? 3 + 8LL * h->C : (long long)h->C * NCP - h->n_cam_held);
  const long long n_total = n_cam + 3 * (h->P_total - pt_held_total);
  if (n_total <= 0) {
    set_error(h, "lcba_solve: every parameter is held (lcba_set_fixed): nothing to optimise");
    return LCBA_E_ARG;
  }
  const long long max_nfev = opt.max_nfev > 0 ? opt.max_nfev : 100 * n_total;

  struct EventPair {   // destroyed on every exit path
    cudaEvent_t a = nullptr, b = nullptr;
    EventPair() { cudaEventCreate(&a); cudaEventCreate(&b); }
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
  } ev;
  cudaEvent_t t0 = ev.a, t1 = ev.b;
  cudaEventRecord(t0, h->stream);

  Ctl init;
  memset(&init, 0, sizeof(init));
  init.ftol = opt.ftol;
  init.xtol = opt.xtol;
  init.term = -1;
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_ctl, &init, sizeof(Ctl), cudaMemcpyHostToDevice, h->stream));

  LCBA_TRY(pass_linearize(h, 1));
  LCBA_TRY(read_ctl(h));
  if (h->h_ctl->nonfinite) {
    set_error(h, "Residuals are not finite in the initial point.");
    return LCBA_E_NONFINITE;
  }
  long long nfev = 1, njev = 1, iteration = 0;
  int status = -1;
  res->initial_cost = h->h_ctl->cost;
  double cost = h->h_ctl->cost, g_norm = h->h_ctl->g_norm;
  double step_norm = NAN, actual = NAN;
  double last_reg = 0.0;
  // After an accepted step the re-linearisation is only enqueued; its scalars (cost, |g|_inf)
  // come back with the NEXT trial's status in one host sync per iteration.  If they say
  // "gtol reached", the speculatively evaluated trial is simply discarded.
  bool lin_pending = false;
  auto absorb_lin = [&]() {
    cost = h->h_ctl->cost;
    g_norm = h->h_ctl->g_norm;
    lin_pending = false;
  };
  while (true) {
    const bool limits = nfev >= max_nfev || (opt.max_iterations > 0 && iteration >= opt.max_iterations);
    if (lin_pending && (status >= 0 || limits)) {
      LCBA_TRY(read_ctl(h));
      absorb_lin();
    }
    if (!lin_pending) {
      if (g_norm < opt.gtol) status = LCBA_STATUS_GTOL;
      add_trace(h, iteration, nfev, cost, actual, step_norm, g_norm, h->h_ctl->Delta, last_reg);
      if (status >= 0 || limits) break;
    }

    auto enqueue_front = [&]() -> int {
      LCBA_TRY(pass_jdot(h));
      if (h->fix_cameras) {
        // points only: the normal equations are block diagonal, p_p = (V + lam Dp^2)^-1 g_p
        KL(h, "point_factor", k_point_factor<<<nblk(h->P, 256), 256, 0, h->stream>>>(
              h->d_Vg, h->d_scl_p, 0.0, h->d_ctl, h->P, pt_mask(h), nullptr, h->d_Lz));
        LCBA_CUDA(h, cudaMemsetAsync(h->d_pc, 0, (size_t)h->C * NCP * 8, h->stream));
        LCBA_CUDA(h, cudaMemsetAsync(h->d_fail, 0, 2 * sizeof(int), h->stream));
      } else {
        LCBA_TRY(pass_schur(h, nullptr));
      }
      return LCBA_OK;
    };
    auto enqueue_back = [&](double mu_) -> int {
      if (!h->fix_cameras) LCBA_TRY(pass_camera_solve(h, mu_));
      LCBA_TRY(pass_backsub(h));
      LCBA_TRY(pass_trial(h));
      return LCBA_OK;
    };
    // the whole static part of the iteration (mu = 0) as one graph; Cholesky retries enqueue directly
    LCBA_TRY(run_graphed(h, h->g_body[h->cur], gkey, graphs, [&]() -> int {
      LCBA_TRY(enqueue_front());
      return enqueue_back(0.0);
    }));
    bool body_done = true;
    double mu = 0.0;
    bool have_trial = false;
    double prev_actual = actual, prev_step = step_norm;
    actual = -1.0;
    int term = -1;
    bool gtol_hit = false;
    while (true) {   // Cholesky retry loop (extra camera damping on breakdown)
      if (!body_done) LCBA_TRY(enqueue_back(mu));
      body_done = false;
      LCBA_TRY(read_ctl(h));
      if (lin_pending) {
        absorb_lin();
        if (g_norm < opt.gtol) status = LCBA_STATUS_GTOL;
        add_trace(h, iteration, nfev, cost, prev_actual, prev_step, g_norm, h->h_ctl->Delta, last_reg);
        if (status >= 0) { gtol_hit = true; break; }
      }
      if (h->h_ctl->chol_fail & 2) {
        set_error(h, "k_chol_fused: grid barrier timed out");
        return LCBA_E_CUDA;
      }
      if (h->h_ctl->retry) {
        mu = std::max(std::max(10.0 * mu, 10.0 * h->h_ctl->reg_term), 1e-13);
        if (mu > 1e6) {
          set_error(h, "reduced camera system is not positive definite even with damping");
          return LCBA_E_NONFINITE;
        }
        continue;
      }
      have_trial = true;
      break;
    }
    if (gtol_hit) { actual = prev_actual; step_norm = prev_step; break; }
    last_reg = h->h_ctl->reg_term;
    // inner loop: trials until the cost decreases (trf.py:503-541); scipy would spin up to
    // max_nfev = 100 n when all tolerances are 0 and the step underflows — cap the rejections
    int rejected = 0;
    while (true) {
      if (have_trial) { nfev++; have_trial = false; }
      const Ctl& c = *h->h_ctl;
      const bool finite = (c.cost_new - c.cost_new == 0.0);
      if (finite) {
        actual = c.actual;
        step_norm = c.step_norm;
        term = c.term;
        if (term >= 0) break;
      }
      if (finite && actual > 0.0) break;
      if (nfev >= max_nfev || ++rejected > 64) break;
      LCBA_TRY(pass_trial(h));
      LCBA_TRY(read_ctl(h));
      have_trial = true;
    }
    if (term >= 0) status = term;
    if (actual > 0.0) {
      h->cur = 1 - h->cur;      // x <- x_new (buffers swap, tables included)
      LCBA_TRY(run_graphed(h, h->g_lin[h->cur], gkey, graphs, [&]() -> int {
        KL(h, "ctl", k_ctl_commit<<<1, 1, 0, h->stream>>>(h->d_ctl));
        return pass_linearize(h, 0);
      }));
      njev++;
      lin_pending = true;
    } else {
      step_norm = 0.0;
      actual = 0.0;
    }
    iteration++;
  }
  if (status < 0) status = LCBA_STATUS_MAX_NFEV;
  cudaEventRecord(t1, h->stream);
  cudaEventSynchronize(t1);
  float ms = 0;
  cudaEventElapsedTime(&ms, t0, t1);
  res->cost = cost;
  res->optimality = g_norm;
  res->nfev = nfev;
  res->njev = njev;
  res->iterations = iteration;
  res->status = status;
  res->n_trace = (int)h->trace.size();
  res->solve_ms = ms;
  res->gpu_launches = h->launches - launches0;
  res->reserved[0] = (double)(h->graph_replays - replays0);   // CUDA-graph replays inside this solve
  h->prof_on = false;
  return LCBA_OK;
}

extern "C" int lcba_get_trace(lcba_t* h, lcba_trace_row* rows, int32_t max_rows) {
  if (!h || !rows) return LCBA_E_ARG;
  const int n = std::min<int>(max_rows, (int)h->trace.size());
  for (int i = 0; i < n; ++i) rows[i] = h->trace[i];
  return n;
}

extern "C" int lcba_get_profile(lcba_t* h, lcba_kernel_stat* stats, int32_t max_stats, int32_t* n_out) {
  if (!h || !n_out) return LCBA_E_ARG;
  int i = 0;
  for (auto& kv : h->prof) {
    if (i >= max_stats) break;
    if (stats) {
      memset(&stats[i], 0, sizeof(stats[i]));
      strncpy(stats[i].name, kv.first.c_str(), sizeof(stats[i].name) - 1);
      stats[i].launches = kv.second.first;
      stats[i].total_ms = kv.second.second;
    }
    ++i;
  }
  *n_out = i;
  return LCBA_OK;
}

__global__ void k_extract_gp(const double* __restrict__ Vg, long long P, double* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P * 3) out[i] = Vg[(i / 3) * 9 + 6 + (i % 3)];
}

extern "C" int lcba_get_grad(lcba_t* h, double* g_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_get_grad: no problem set"); return LCBA_E_STATE; }
  if (!g_out) return LCBA_E_ARG;
  cudaSetDevice(h->device);
  const size_t nc = (size_t)h->C * NCP;
  KL(h, "extract", k_extract_gp<<<nblk(h->P * 3, 256), 256, 0, h->stream>>>(h->d_Vg, h->P, h->d_gn_p));
  LCBA_CUDA(h, cudaMemcpyAsync(g_out, h->d_g_c, nc * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaMemcpyAsync(g_out + nc, h->d_gn_p, (size_t)h->P * 3 * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  return check_launch(h, "lcba_get_grad");
}

__global__ void k_concat_scale(const double* __restrict__ scl_c, int nc, const double* __restrict__ scl_p,
                               long long np, double* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nc) out[i] = scl_c[i];
  else if (i < nc + np) out[i] = scl_p[i - nc];
}

extern "C" int lcba_linearize(lcba_t* h, double lam, double* S_out, double* rhs_out, double* grad_out,
                              double* scale_inv_out, double* cost_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_linearize: no problem set"); return LCBA_E_STATE; }
  cudaSetDevice(h->device);
  Ctl init;
  memset(&init, 0, sizeof(init));
  init.term = -1;
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_ctl, &init, sizeof(Ctl), cudaMemcpyHostToDevice, h->stream));
  h->fix_cameras = 0;
  h->shared_intr = 0;
  h->masks_on = false;
  h->bounded = false;
  LCBA_TRY(pass_linearize(h, 1));
  LCBA_TRY(pass_schur(h, &lam));
  const int n = h->C * NCP;
  if (S_out) LCBA_CUDA(h, cudaMemcpyAsync(S_out, h->d_S, (size_t)n * n * 8, cudaMemcpyDeviceToHost, h->stream));
  if (rhs_out) LCBA_CUDA(h, cudaMemcpyAsync(rhs_out, h->d_rhs, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_TRY(read_ctl(h));
  if (cost_out) *cost_out = h->h_ctl->cost;
  if (grad_out) LCBA_TRY(lcba_get_grad(h, grad_out));
  if (scale_inv_out) {
    LCBA_CUDA(h, cudaMemcpyAsync(scale_inv_out, h->d_scl_c, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    LCBA_CUDA(h, cudaMemcpyAsync(scale_inv_out + n, h->d_scl_p, (size_t)h->P * 3 * 8, cudaMemcpyDeviceToHost, h->stream));
    LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  }
  return check_launch(h, "lcba_linearize");
}

// Smallest Jacobi-relative pivot l_jj^2 / S_jj of the free camera rows below which S counts as singular.  At the
// gauge-fixed solutions of the golden rigs it is 5e-4 .. 9e-4; with the gauge free it is rounding noise of
// either sign, |.| <= 2e-10 (tests/test_covariance.py recomputes both).
static const double COV_PIVOT_TOL = 1e-7;

extern "C" int lcba_covariance(lcba_t* h, double* cam_cov_out, double* pt_cov_out, double* cost_out,
                               double* min_pivot_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_covariance: no problem set"); return LCBA_E_STATE; }
  cudaSetDevice(h->device);
  const int C = h->C, n = C * NCP, npad = cov_npad(n);
  cudaStream_t st = h->stream;
  // free-entry counts over the ranks; the camera mask must be the same on every rank (as in lcba_solve)
  long long pt_free = h->P - h->n_pt_held;
  if (h->comm) {
    double v[5] = {(double)pt_free, (double)h->n_cam_held, h->cam_fixed_sum, -(double)h->n_cam_held, -h->cam_fixed_sum};
    LCBA_CUDA(h, cudaMemcpyAsync(h->d_red, v, sizeof(v), cudaMemcpyHostToDevice, st));
    LCBA_TRY(allreduce(h, h->d_red, 1, NCCL_SUM));
    LCBA_TRY(allreduce(h, h->d_red + 1, 4, NCCL_MAX));
    LCBA_CUDA(h, cudaMemcpyAsync(v, h->d_red, sizeof(v), cudaMemcpyDeviceToHost, st));
    LCBA_CUDA(h, cudaStreamSynchronize(st));
    if (v[1] != -v[3] || v[2] != -v[4]) {
      set_error(h, "lcba_covariance: the ranks hold different camera masks (lcba_set_fixed)");
      return LCBA_E_ARG;
    }
    pt_free = (long long)(v[0] + 0.5);
  }
  const long long cam_free = n - h->n_cam_held;
  if (cam_free + 3 * pt_free <= 0) {
    set_error(h, "lcba_covariance: every parameter is held (lcba_set_fixed): nothing to estimate");
    return LCBA_E_ARG;
  }
  // LCBA_COV_PROFILE=1: CUDA-event time of every launch of this call (synchronising after each), for
  // lcba_get_profile (tools/cov_time.py); off again on every return
  struct ProfOff { lcba_t* h; ~ProfOff() { h->prof_on = false; } } prof_off{h};
  {
    const char* pe = getenv("LCBA_COV_PROFILE");
    h->prof_on = pe && atoi(pe) != 0;
    if (h->prof_on) h->prof.clear();
  }
  Ctl init;
  memset(&init, 0, sizeof(init));
  init.term = -1;
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_ctl, &init, sizeof(Ctl), cudaMemcpyHostToDevice, st));
  h->fix_cameras = 0;
  h->shared_intr = 0;
  h->masks_on = true;
  h->bounded = false;
  LCBA_TRY(pass_linearize(h, 1));
  // unheld points with fewer than two distinct cameras (k_point_factor would clamp their pivots)
  double* views = h->d_red + 40;
  KL(h, "cov_views", k_cov_views<<<h->pt_grid, 256, 0, st>>>(h->d_mask, h->d_pt_fixed, h->P, h->d_part));
  KL(h, "reduce", k_reduce_scalars<<<1, 256, 0, st>>>(h->d_part, h->pt_grid, 1, views, 1));
  LCBA_TRY(allreduce(h, views, 1, NCCL_SUM));
  // the exact undamped reduced camera system on the problem's Schur route, and its Cholesky factor
  const double lam = 0.0;
  LCBA_TRY(pass_schur(h, &lam));
  LCBA_TRY(pass_camera_solve(h, 0.0));
  double nviews = 0.0;
  int fail = 0;
  std::vector<double> dinv(n), sdiag(n);
  LCBA_CUDA(h, cudaMemcpyAsync(&nviews, views, 8, cudaMemcpyDeviceToHost, st));
  LCBA_CUDA(h, cudaMemcpyAsync(&fail, h->d_fail, sizeof(int), cudaMemcpyDeviceToHost, st));
  LCBA_CUDA(h, cudaMemcpy2DAsync(dinv.data(), 8, h->d_Lf, (size_t)(n + 1) * 8, 8, n, cudaMemcpyDeviceToHost, st));
  LCBA_CUDA(h, cudaMemcpy2DAsync(sdiag.data(), 8, h->d_S, (size_t)(n + 1) * 8, 8, n, cudaMemcpyDeviceToHost, st));
  LCBA_TRY(read_ctl(h));
  if (fail & 2) { set_error(h, "k_chol_fused: grid barrier timed out"); return LCBA_E_CUDA; }
  if (cost_out) *cost_out = h->h_ctl->cost;
  // Jacobi-relative pivots of the free rows (the diagonal of the factor stores 1 / l_jj); a non-positive pivot
  // (fail bit 0) reports 0
  double min_pivot = INFINITY;
  for (int j = 0; j < n; ++j)
    if (h->h_cam_fixed.empty() || !h->h_cam_fixed[j]) min_pivot = std::min(min_pivot, 1.0 / (dinv[j] * dinv[j] * sdiag[j]));
  if (fail & 1) min_pivot = 0.0;
  if (min_pivot_out) *min_pivot_out = min_pivot;
  if (nviews > 0.0) {
    set_error(h, "lcba_covariance: " + std::to_string((long long)(nviews + 0.5)) +
                     " unheld point(s) seen by fewer than two distinct cameras: their position is not determined; "
                     "hold them (fixed_points) or drop them");
    return LCBA_E_SINGULAR;
  }
  if (cam_free > 0 && !(min_pivot >= COV_PIVOT_TOL)) {
    char buf[96];
    snprintf(buf, sizeof(buf), "(smallest Jacobi-relative pivot %.3g < %.0e)", min_pivot, COV_PIVOT_TOL);
    set_error(h, std::string("lcba_covariance: the reduced camera system is singular ") + buf +
                     ": the gauge (rotation, translation, scale) is not fixed or a camera entry is unconstrained; "
                     "hold camera 0's extrinsics and three points or one scale coordinate (fixed_camera_params, "
                     "fixed_points), and every entry of a camera that sees no point");
    return LCBA_E_SINGULAR;
  }
  if (!h->d_cov_X) {
    LCBA_TRY(dev_alloc(h, &h->d_cov_X, (size_t)npad * npad));
    LCBA_TRY(dev_alloc(h, &h->d_cov_Sinv, (size_t)n * n));
    LCBA_TRY(dev_alloc(h, &h->d_cov_pt, (size_t)h->P * 6));
  }
  LCBA_CUDA(h, cudaMemsetAsync(h->d_cov_X, 0, (size_t)npad * npad * 8, st));
  KL(h, "chol_inverse", k_chol_inverse<<<n, 256, 0, st>>>(h->d_Lf, n, h->d_cam_fixed, npad, h->d_cov_X));
  const unsigned nt = (unsigned)((n + CH_NB - 1) / CH_NB);
  KL(h, "chol_inverse_gram", k_chol_inverse_gram<<<dim3(nt, nt), 256, 0, st>>>(h->d_cov_X, n, npad, h->d_cov_Sinv));
  if (pt_cov_out) {
    const int w = h->cur;
    const bool b16 = cov_smem_doubles(C, 16) * 8 + 2048 <= h->smem_optin;
    const size_t smem = cov_smem_doubles(C, b16 ? 16 : 8) * 8;
    const long long nbatch = (h->P + (b16 ? 16 : 8) - 1) / (b16 ? 16 : 8);
    const int per_sm = std::max(1, (int)(h->smem_optin / (smem + 1024)));
    const int grid = (int)std::max<long long>(1, std::min<long long>(nbatch, (long long)h->sm_count * per_sm));
    if (b16)
      KL(h, "point_cov", k_point_cov<16><<<grid, COV_THREADS, smem, st>>>(
            h->d_cov_X, h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, C,
            h->d_cov_pt));
    else
      KL(h, "point_cov", k_point_cov<8><<<grid, COV_THREADS, smem, st>>>(
            h->d_cov_X, h->d_tab[w], h->d_pts[w], h->d_pair_w, h->d_pair_start, h->d_mask, h->d_Lz, h->P, C,
            h->d_cov_pt));
    LCBA_CUDA(h, cudaMemcpyAsync(pt_cov_out, h->d_cov_pt, (size_t)h->P * 6 * 8, cudaMemcpyDeviceToHost, st));
  }
  if (cam_cov_out)
    LCBA_CUDA(h, cudaMemcpyAsync(cam_cov_out, h->d_cov_Sinv, (size_t)n * n * 8, cudaMemcpyDeviceToHost, st));
  LCBA_CUDA(h, cudaStreamSynchronize(st));
  return check_launch(h, "lcba_covariance");
}

extern "C" int lcba_time_device(lcba_t* h, int32_t what, int32_t reps, double* ms_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_time_device: no problem set"); return LCBA_E_STATE; }
  if (!ms_out || reps <= 0) return LCBA_E_ARG;
  cudaSetDevice(h->device);
  LCBA_TRY(build_tables(h, h->cur));
  if (what == 1) LCBA_TRY(ensure_jac_buffers(h));
  cudaEvent_t t0, t1;
  cudaEventCreate(&t0);
  cudaEventCreate(&t1);
  int rc = LCBA_OK;
  for (int r = -1; r < reps && rc == LCBA_OK; ++r) {   // r = -1: warm-up
    if (r == 0) cudaEventRecord(t0, h->stream);
    if (what == 0) rc = run_residual(h, h->cur, nullptr);
    else if (what == 1) rc = run_jacobian_blocks(h, h->cur);
    else { set_error(h, "lcba_time_device: unknown selector"); rc = LCBA_E_ARG; }
  }
  cudaEventRecord(t1, h->stream);
  cudaEventSynchronize(t1);
  float ms = 0;
  cudaEventElapsedTime(&ms, t0, t1);
  cudaEventDestroy(t0);
  cudaEventDestroy(t1);
  if (rc != LCBA_OK) return rc;
  *ms_out = (double)ms / reps;
  return check_launch(h, "lcba_time_device");
}

// ------------------------------------------------------------------------------ multi-GPU
extern "C" int lcba_nccl_unique_id(void* id_out128) {
  if (!id_out128) return LCBA_E_ARG;
  std::string err;
  if (!nccl_load(err)) { set_error(nullptr, err); return LCBA_E_NCCL; }
  ncclUniqueId id;
  int rc = g_nccl.GetUniqueId(&id);
  if (rc != 0) { set_error(nullptr, std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(rc)); return LCBA_E_NCCL; }
  memcpy(id_out128, &id, sizeof(id));
  return LCBA_OK;
}

// Map every rank's peer block (cudaIpc handles exchanged with ncclAllGather).  All ranks must agree on the
// outcome: the verdicts are summed with NCCL, anything short of "all ranks mapped all peers" disables the path
// everywhere.
static void peer_setup(lcba_t* h) {
  PeerState& ps = g_peer;
  const int n = h->nranks, rank = h->rank;
  for (int r = 0; r < PEER_MAX_RANKS; ++r)
    if (ps.opened[r]) { cudaIpcCloseMemHandle(ps.opened[r]); ps.opened[r] = nullptr; }
  if (ps.block) { cudaFree(ps.block); ps.block = nullptr; }
  ps.ok = false;
  ps.epoch = 0;
  // Opt-in: measured against ncclAllReduce inside one job (tools/peer_ab.py, 8 GPUs, 24 cameras x 1 M points) the
  // peer route is 0.7 % SLOWER per iteration (1.585 vs 1.574 ms): NCCL's small all-reduces are not what the fixed
  // cost of an iteration consists of.  LCBA_PEER_REDUCE=1: map and use; 2: map, keep NCCL until
  // lcba_debug_peer_reduce switches (A/B tool); unset / 0: NCCL only, nothing is mapped.
  const char* env = getenv("LCBA_PEER_REDUCE");
  const int mode = env ? atoi(env) : 0;
  if (mode <= 0) return;
  bool mine = n > 1 && n <= PEER_MAX_RANKS && g_nccl.AllGather != nullptr;
  cudaIpcMemHandle_t hdl;
  memset(&hdl, 0, sizeof(hdl));
  if (mine && !ps.h_fail)
    mine = cudaHostAlloc((void**)&ps.h_fail, sizeof(int), cudaHostAllocMapped) == cudaSuccess &&
           cudaHostGetDevicePointer((void**)&ps.d_fail, ps.h_fail, 0) == cudaSuccess;
  if (mine) {
    *ps.h_fail = 0;
    mine = cudaMalloc(&ps.block, peer_block_bytes()) == cudaSuccess &&
           cudaMemset(ps.block, 0, peer_block_bytes()) == cudaSuccess &&
           cudaIpcGetMemHandle(&hdl, ps.block) == cudaSuccess;
  }
  cudaGetLastError();
  // exchange the handles (every rank takes part, whatever its own verdict so far)
  std::vector<cudaIpcMemHandle_t> all(n);
  unsigned char* d_h = nullptr;
  bool xch = g_nccl.AllGather != nullptr && cudaMalloc((void**)&d_h, (size_t)n * sizeof(hdl)) == cudaSuccess;
  if (xch) {
    cudaMemcpyAsync(d_h + (size_t)rank * sizeof(hdl), &hdl, sizeof(hdl), cudaMemcpyHostToDevice, h->stream);
    xch = g_nccl.AllGather(d_h + (size_t)rank * sizeof(hdl), d_h, sizeof(hdl), /*ncclInt8*/ 0, h->comm, h->stream) == 0 &&
          cudaMemcpyAsync(all.data(), d_h, (size_t)n * sizeof(hdl), cudaMemcpyDeviceToHost, h->stream) == cudaSuccess &&
          cudaStreamSynchronize(h->stream) == cudaSuccess;
  }
  if (d_h) cudaFree(d_h);
  mine = mine && xch;
  if (mine) {
    for (int r = 0; r < n && mine; ++r) {
      void* q = ps.block;
      if (r != rank) {
        mine = cudaIpcOpenMemHandle(&q, all[r], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
        if (mine) ps.opened[r] = q;
      }
      if (mine) {
        ps.ptrs.sym[r] = (double*)q;
        ps.ptrs.flags[r] = (unsigned*)((char*)q + 2 * PEER_SLOT * sizeof(double));
      }
    }
  }
  cudaGetLastError();
  // agreement (also the barrier after which every block is zeroed and mapped): sum of the verdicts over NCCL
  double* d_v = nullptr;
  double v = mine ? 1.0 : 0.0, sum = 0.0;
  if (cudaMalloc((void**)&d_v, 8) == cudaSuccess &&
      cudaMemcpyAsync(d_v, &v, 8, cudaMemcpyHostToDevice, h->stream) == cudaSuccess &&
      g_nccl.AllReduce(d_v, d_v, 1, NCCL_FLOAT64, NCCL_SUM, h->comm, h->stream) == 0 &&
      cudaMemcpyAsync(&sum, d_v, 8, cudaMemcpyDeviceToHost, h->stream) == cudaSuccess &&
      cudaStreamSynchronize(h->stream) == cudaSuccess)
    ps.ok = mine && sum == (double)n;
  if (d_v) cudaFree(d_v);
  g_peer_available = ps.ok;
  if (mode == 2) ps.ok = false;
  cudaGetLastError();
  if (getenv("LCBA_PEER_VERBOSE"))
    fprintf(stderr, "[lcba] rank %d/%d: peer all-reduce %s\n", rank, n, ps.ok ? "on (NVLink peer memory)" : "off (NCCL)");
}

extern "C" int lcba_comm_init(lcba_t* h, int32_t rank, int32_t nranks, const void* id128) {
  if (!h || nranks < 1 || rank < 0 || rank >= nranks) { set_error(h, "lcba_comm_init: bad argument"); return LCBA_E_ARG; }
  std::string err;
  if (!nccl_load(err)) { set_error(h, err); return LCBA_E_NCCL; }
  cudaSetDevice(h->device);
  if (!id128) {
    // attach the communicator this process already created
    if (!g_comm || g_comm_rank != rank || g_comm_nranks != nranks || g_comm_device != h->device) {
      set_error(h, "lcba_comm_init: no matching process communicator to attach (pass a unique id first)");
      return LCBA_E_STATE;
    }
    h->comm = g_comm;
    h->rank = rank;
    h->nranks = nranks;
    return LCBA_OK;
  }
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  ncclComm_t comm = nullptr;
  int rc = g_nccl.CommInitRank(&comm, nranks, id, rank);
  if (rc != 0) { set_error(h, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(rc)); return LCBA_E_NCCL; }
  if (g_comm) g_nccl.CommDestroy(g_comm);
  g_comm = comm;
  g_comm_rank = rank;
  g_comm_nranks = nranks;
  g_comm_device = h->device;
  h->comm = comm;
  h->rank = rank;
  h->nranks = nranks;
  peer_setup(h);        // optional: any failure leaves the NCCL path in place
  return LCBA_OK;
}

// measurement switch: route the all-reduces through NVLink peer memory (1) or NCCL (0) from now on; every rank
// must call it at the same point of the program.  Returns 1 when the peer path is (now) active, 0 when it is off
// or was never set up (LCBA_PEER_REDUCE=0, mapping failed on some rank).
extern "C" int lcba_debug_peer_reduce(lcba_t* h, int enable) {
  if (!h || !h->comm) return 0;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  g_peer.ok = g_peer_available && enable != 0;
  return g_peer.ok ? 1 : 0;
}

// debug: per-CTA cycle counters of the last k_schur launch (LCBA_SCHUR_STATS=1)
extern "C" int lcba_debug_schur_stats(lcba_t* h, long long* out, int max_ctas, int* nkinds, int* nslices) {
  if (!h || !h->d_stats || !out) return LCBA_E_STATE;
  const int nk = h->use_i8 ? 1 : (h->use_mma ? h->mplan.nkinds : h->plan.nkinds);
  const int ns = h->use_i8 ? (int)h->i8plan.work.size() : (h->use_mma ? h->mplan.nslices : h->plan.nslices);
  const int n = std::min(max_ctas, ns * nk);
  cudaMemcpy(out, h->d_stats, (size_t)n * 4 * sizeof(long long), cudaMemcpyDeviceToHost);
  *nkinds = nk;
  *nslices = ns;
  return LCBA_OK;
}

// test hook: 1 when the last Schur pass of the int8 path handed the pass to DMMA (k_i8_check), 0 when the int8
// result stood, -1 when the handle does not use the int8 path
extern "C" int lcba_debug_i8_fallback(lcba_t* h) {
  if (!h || !h->have_problem || !h->use_i8 || !h->d_i8gate) return -1;
  cudaSetDevice(h->device);
  int v = 0;
  if (cudaStreamSynchronize(h->stream) != cudaSuccess ||
      cudaMemcpy(&v, h->d_i8gate, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return v;
}

// host-only test hook: the unit plan of the tensor-path Schur kernel for C cameras (no GPU needed).
// units_out: per kind MMA_CONS_WARPS rows of (tr0, tc0, nr, nc, tri); returns the number of kinds.
extern "C" int lcba_debug_mma_plan(int32_t C, int32_t sm_count, int32_t* units_out, int32_t max_kinds,
                                   int32_t* nslices_out, int32_t* ok_out) {
  if (C < 1 || C > LCBA_MAX_CAMERAS || !units_out) return LCBA_E_ARG;
  const MmaPlan pl = make_mma_plan(C, sm_count, 227 * 1024 - 2048);
  if (ok_out) *ok_out = (pl.nkinds > 0 && C <= MMA_MAX_CAMERAS) ? 1 : 0;
  if (nslices_out) *nslices_out = pl.nslices;
  for (int k = 0; k < pl.nkinds && k < max_kinds; ++k)
    for (int w = 0; w < MMA_CONS_WARPS; ++w) {
      const MmaUnit& u = pl.kinds[k].unit[w];
      int32_t* o = units_out + ((size_t)k * MMA_CONS_WARPS + w) * 5;
      o[0] = u.tr0; o[1] = u.tc0; o[2] = u.nr; o[3] = u.nc; o[4] = u.tri;
    }
  return pl.nkinds;
}

// host-only test hook: the strip plan of the int8 tensor-core Schur kernel (schur_i8.cuh make_i8_plan; the
// cover plan and the choice between the two: lcba_debug_i8_cover_plan).
// tiles_out: per tile 8 ints (m_rg0, m_nrg, n_rg0, n_nrg, n2_rg0, n2_nrg, first CTA, CTAs); work_out: per CTA
// 3 ints (tile, kb0, kb1).  Returns the number of tiles; *nwork_out CTAs, *nrg_out row groups, *nkb_out K blocks.
extern "C" int lcba_debug_i8_plan(int32_t C, int64_t P, int32_t sm_count, int32_t* tiles_out, int32_t max_tiles,
                                  int32_t* work_out, int32_t max_work, int32_t* nwork_out, int32_t* nrg_out,
                                  int64_t* nkb_out) {
  if (C < 1 || C > LCBA_MAX_CAMERAS || P < 1 || !tiles_out) return LCBA_E_ARG;
  const I8Plan pl = make_i8_plan(C, P, sm_count);
  for (size_t i = 0; i < pl.tiles.size() && (int)i < max_tiles; ++i) {
    const I8Tile& t = pl.tiles[i];
    int32_t* o = tiles_out + 8 * i;
    o[0] = t.m_rg0; o[1] = t.m_nrg; o[2] = t.n_rg0; o[3] = t.n_nrg; o[4] = t.n2_rg0; o[5] = t.n2_nrg; o[6] = t.w0; o[7] = t.nw;
  }
  if (work_out)
    for (size_t i = 0; i < pl.work.size() && (int)i < max_work; ++i) {
      work_out[3 * i] = (int32_t)i; work_out[3 * i + 1] = pl.work[i].kb0; work_out[3 * i + 2] = pl.work[i].kb1;
    }
  if (nwork_out) *nwork_out = (int32_t)pl.work.size();
  if (nrg_out) *nrg_out = pl.NRG;
  if (nkb_out) *nkb_out = pl.nkb;
  return (int)pl.tiles.size();
}

// host-only test hook: a tile plan of the int8 tensor-core Schur kernel with both row ranges of A.
// which: 0 = the plan k_i8_syrk runs (the cost model's choice), 1 = the strip plan, 2 = the cover plan.
// tiles_out: per tile 10 ints (m_rg0, m_nrg, m2_rg0, m2_nrg, n_rg0, n_nrg, n2_rg0, n2_nrg, first CTA, CTAs);
// work_out: per CTA 3 ints (tile, kb0, kb1); model_out: 4 doubles (executed int8 ops of one launch, the
// model's slowest-CTA cycles of this plan, of the strip plan, of the cover plan).  Returns the number of
// tiles; *nwork_out CTAs, *nrg_out row groups, *nkb_out K blocks, *cover_out 1 for a cover plan.
extern "C" int lcba_debug_i8_cover_plan(int32_t C, int64_t P, int32_t sm_count, int32_t which, int32_t* tiles_out,
                                        int32_t max_tiles, int32_t* work_out, int32_t max_work, int32_t* nwork_out,
                                        int32_t* nrg_out, int64_t* nkb_out, int32_t* cover_out, double* model_out) {
  if (C < 1 || C > LCBA_MAX_CAMERAS || P < 1 || sm_count < 1 || which < 0 || which > 2 || !tiles_out) return LCBA_E_ARG;
  const I8Plan pl = make_i8_best_plan(C, P, sm_count, which);
  for (size_t i = 0; i < pl.tiles.size() && (int)i < max_tiles; ++i) {
    const I8Tile& t = pl.tiles[i];
    int32_t* o = tiles_out + 10 * i;
    o[0] = t.m_rg0; o[1] = t.m_nrg; o[2] = t.m2_rg0; o[3] = t.m2_nrg; o[4] = t.n_rg0; o[5] = t.n_nrg;
    o[6] = t.n2_rg0; o[7] = t.n2_nrg; o[8] = t.w0; o[9] = t.nw;
  }
  if (work_out)
    for (size_t i = 0; i < pl.work.size() && (int)i < max_work; ++i) {
      const I8Work& w = pl.work[i];
      int ti = 0;
      while (ti + 1 < (int)pl.tiles.size() && pl.tiles[ti + 1].w0 <= (int)i) ++ti;
      work_out[3 * i] = ti; work_out[3 * i + 1] = w.kb0; work_out[3 * i + 2] = w.kb1;
    }
  if (nwork_out) *nwork_out = (int32_t)pl.work.size();
  if (nrg_out) *nrg_out = pl.NRG;
  if (nkb_out) *nkb_out = pl.nkb;
  if (cover_out) *cover_out = pl.cover ? 1 : 0;
  if (model_out) {
    model_out[0] = i8_executed_ops(pl);
    model_out[1] = pl.model_cycles;
    model_out[2] = make_i8_plan(C, P, sm_count).model_cycles;
    model_out[3] = make_i8_cover_plan(C, P, sm_count).model_cycles;
  }
  return (int)pl.tiles.size();
}

// host-only test hook: the K blocks of every CTA of a tile plan under a schedule (kmajor: 1 = K-major, the default;
// 0 = one contiguous range per CTA, LCBA_I8_SCHED=range).  work_out: per CTA 6 ints (tile, kb0, kb1, kfirst, kc,
// kstride): the K blocks kfirst + (i / kc) kstride + i % kc, i < kb1 - kb0.  *window_out: the window in K blocks.
// Returns the number of CTAs.
extern "C" int lcba_debug_i8_schedule(int32_t C, int64_t P, int32_t sm_count, int32_t which, int32_t kmajor,
                                      int32_t* work_out, int32_t max_work, int32_t* window_out) {
  if (C < 1 || C > LCBA_MAX_CAMERAS || P < 1 || sm_count < 1 || which < 0 || which > 2 || !work_out) return LCBA_E_ARG;
  const I8Plan pl = make_i8_best_plan(C, P, sm_count, which, kmajor != 0);
  for (size_t i = 0; i < pl.work.size() && (int)i < max_work; ++i) {
    const I8Work& w = pl.work[i];
    int ti = 0;
    while (ti + 1 < (int)pl.tiles.size() && pl.tiles[ti + 1].w0 <= (int)i) ++ti;
    int32_t* o = work_out + 6 * i;
    o[0] = ti; o[1] = w.kb0; o[2] = w.kb1; o[3] = w.kfirst; o[4] = w.kc; o[5] = w.kstride;
  }
  if (window_out) *window_out = pl.window;
  return (int)pl.work.size();
}

// ---- squared-residual variants (pySBA.py:151-206): cost, J^T f, J^T J in one pass ----------
extern "C" int lcba_sq_normal(lcba_t* h, int32_t mode, const double* theta, double* cost_out,
                              double* g_out, double* H_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_sq_normal: no problem set"); return LCBA_E_STATE; }
  if (!theta || (mode != LCBA_SQ_CAMONLY && mode != LCBA_SQ_TRANSFORM) || ((g_out == nullptr) != (H_out == nullptr))) {
    set_error(h, "lcba_sq_normal: bad mode, NULL theta, or only one of g / H given");
    return LCBA_E_ARG;
  }
  cudaSetDevice(h->device);
  const int C = h->C;
  const bool derivs = g_out != nullptr;
  const int K = (mode == LCBA_SQ_CAMONLY ? C * SQC_VALS : SQT_VALS) + 1;
  const int warps = sq_camonly_warps(C, h->smem_optin);
  const int threads = (mode == LCBA_SQ_CAMONLY) ? warps * 32 : SQ_THREADS;
  const int per_sm = (mode == LCBA_SQ_CAMONLY) ? 1 : 2;
  const int grid = (int)std::max<long long>(1, std::min<long long>((h->N + threads - 1) / threads,
                                                                   (long long)h->sm_count * per_sm));
  if (!h->d_sqpart || h->sq_grid < grid || h->sq_K < K) {
    LCBA_TRY(dev_alloc(h, &h->d_sqpart, (size_t)grid * K));
    LCBA_TRY(dev_alloc(h, &h->d_sqout, (size_t)K));
    if (!h->d_theta) LCBA_TRY(dev_alloc(h, &h->d_theta, 16));
    h->sq_grid = grid;
    h->sq_K = K;
  }
  const int cur = h->cur, scratch = 1 - h->cur;
  if (mode == LCBA_SQ_CAMONLY) {
    LCBA_CUDA(h, cudaMemcpyAsync(h->d_cams[scratch], theta, (size_t)C * NCP * 8, cudaMemcpyHostToDevice, h->stream));
    LCBA_TRY(build_tables(h, scratch));
    const size_t smem = ((size_t)((C * CAMTAB + 1) & ~1) + (derivs ? (size_t)warps * C * SQC_VALS : 0)) * 8;
    if (derivs)
      KL(h, "sq_camonly", k_sq_camonly<true><<<grid, threads, smem, h->stream>>>(
            h->d_tab[scratch], h->d_pts[cur], h->d_uv, h->d_cam, h->d_pt, h->d_w, h->N, C, h->d_sqpart));
    else
      KL(h, "sq_camonly_cost", k_sq_camonly<false><<<grid, threads, smem, h->stream>>>(
            h->d_tab[scratch], h->d_pts[cur], h->d_uv, h->d_cam, h->d_pt, h->d_w, h->N, C, h->d_sqpart));
  } else {
    LCBA_CUDA(h, cudaMemcpyAsync(h->d_theta, theta, 12 * 8, cudaMemcpyHostToDevice, h->stream));
    LCBA_TRY(build_tables(h, cur));
    const size_t smem = (size_t)((C * CAMTAB + 1) & ~1) * 8;
    if (derivs)
      KL(h, "sq_transform", k_sq_transform<true><<<grid, threads, smem, h->stream>>>(
            h->d_tab[cur], h->d_pts[cur], h->d_uv, h->d_cam, h->d_pt, h->d_w, h->N, C, h->d_theta, h->d_sqpart));
    else
      KL(h, "sq_transform_cost", k_sq_transform<false><<<grid, threads, smem, h->stream>>>(
            h->d_tab[cur], h->d_pts[cur], h->d_uv, h->d_cam, h->d_pt, h->d_w, h->N, C, h->d_theta, h->d_sqpart));
  }
  KL(h, "reduce", k_reduce_cols<<<nblk(K, RC_COLS), RC_COLS * RC_ROWS, 0, h->stream>>>(h->d_sqpart, grid, K, h->d_sqout));
  std::vector<double> v((size_t)K);
  LCBA_CUDA(h, cudaMemcpyAsync(v.data(), h->d_sqout, (size_t)K * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_CUDA(h, cudaStreamSynchronize(h->stream));
  LCBA_TRY(check_launch(h, "lcba_sq_normal"));
  if (cost_out) *cost_out = 0.5 * v[K - 1];
  if (!derivs) return LCBA_OK;
  if (mode == LCBA_SQ_CAMONLY) {
    for (int c = 0; c < C; ++c) {
      const double* s = v.data() + (size_t)c * SQC_VALS;
      double* Hc = H_out + (size_t)c * NCP * NCP;
      int idx = 0;
      for (int a = 0; a < NCP; ++a)
        for (int b = a; b < NCP; ++b, ++idx) Hc[a * NCP + b] = Hc[b * NCP + a] = s[idx];
      for (int a = 0; a < NCP; ++a) g_out[(size_t)c * NCP + a] = s[66 + a];
    }
  } else {
    // J^T J [(k,j),(l,i)] = sum M[k,l] Q[j,i]
    int mi[3][3], qi[4][4], n = 0;
    for (int k = 0; k < 3; ++k) for (int l = k; l < 3; ++l) mi[k][l] = mi[l][k] = n++;
    n = 0;
    for (int j = 0; j < 4; ++j) for (int i = j; i < 4; ++i) qi[j][i] = qi[i][j] = n++;
    for (int k = 0; k < 3; ++k)
      for (int j = 0; j < 4; ++j)
        for (int l = 0; l < 3; ++l)
          for (int i = 0; i < 4; ++i)
            H_out[(4 * k + j) * 12 + 4 * l + i] = v[(size_t)mi[k][l] * SQT_Q + qi[j][i]];
    for (int a = 0; a < 12; ++a) g_out[a] = v[60 + a];
  }
  return LCBA_OK;
}

// test hook: the 2-D trust-region solver used by the device control kernel
extern "C" int lcba_debug_tr2d(double B00, double B01, double B11, double g0, double g1, double Delta,
                               double* p_out, int* newton_out) {
  if (!p_out) return LCBA_E_ARG;
  const TR2 t = solve_tr2d(B00, B01, B11, g0, g1, Delta);
  p_out[0] = t.p0;
  p_out[1] = t.p1;
  if (newton_out) *newton_out = t.newton;
  return LCBA_OK;
}

// test hook: k_copy_damped_rhs + k_chol_fused on a host matrix with an explicit cooperative grid
extern "C" int lcba_debug_chol(lcba_t* h, int32_t n, const double* A, const double* rhs, double mu, const double* d,
                               int32_t grid, double* x_out, double* factor_out, int32_t* fail_out) {
  if (!h) return LCBA_E_ARG;
  if (n < 1 || n > CH_MAXN || !A || !rhs || !x_out || (mu != 0.0 && !d)) {
    set_error(h, "lcba_debug_chol: n outside 1..704, or a NULL array");
    return LCBA_E_ARG;
  }
  cudaSetDevice(h->device);
  int per_sm = 0;
  LCBA_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)k_chol_fused, 256, 0));
  if (grid == 0) grid = chol_grid(n, h->sm_count);
  if (grid < 1 || grid > per_sm * h->sm_count) {
    set_error(h, "lcba_debug_chol: grid outside 1.." + std::to_string(per_sm * h->sm_count) + " (co-resident CTAs)");
    return LCBA_E_ARG;
  }
  cudaStream_t st = h->stream;
  double *dA = nullptr, *drhs = nullptr, *dd = nullptr, *dL = nullptr, *dx = nullptr;
  int* dsync = nullptr;
  cudaError_t e = cudaMallocAsync(&dA, (size_t)n * n * 8, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&drhs, (size_t)n * 8, st);
  if (e == cudaSuccess && d) e = cudaMallocAsync(&dd, (size_t)n * 8, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&dL, (size_t)(n + 1) * n * 8, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&dx, (size_t)n * 8, st);
  if (e == cudaSuccess) e = cudaMallocAsync(&dsync, 2 * sizeof(int), st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(dA, A, (size_t)n * n * 8, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(drhs, rhs, (size_t)n * 8, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess && d) e = cudaMemcpyAsync(dd, d, (size_t)n * 8, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(dsync, 0, 2 * sizeof(int), st);
  if (e == cudaSuccess) {
    k_copy_damped_rhs<<<nblk((long long)(n + 1) * n, 256), 256, 0, st>>>(dA, n, mu, dd, drhs, dL);
    long long* dbg = nullptr;
    int nn = n;
    void* args[] = {(void*)&dL, (void*)&nn, (void*)&dx, (void*)&dsync, (void*)&dbg};
    e = cudaLaunchCooperativeKernel((const void*)k_chol_fused, dim3(grid), dim3(256), args, 0, st);
    h->launches += 2;
  }
  int fail = 0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(x_out, dx, (size_t)n * 8, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && factor_out) e = cudaMemcpyAsync(factor_out, dL, (size_t)(n + 1) * n * 8, cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaMemcpyAsync(&fail, dsync, sizeof(int), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  void* tmp[] = {dA, drhs, dd, dL, dx, dsync};
  for (void* q : tmp) if (q) cudaFreeAsync(q, st);
  if (e != cudaSuccess) { set_error(h, std::string("lcba_debug_chol: ") + cudaGetErrorString(e)); return LCBA_E_CUDA; }
  if (fail_out) *fail_out = fail;
  return LCBA_OK;
}

// test hook: one Gauss-Newton step of the solver's passes on the resident problem, damped with the host's lam
extern "C" int lcba_debug_step(lcba_t* h, double lam, double mu, int32_t mode, double* pc_out, double* pp_out,
                               double* scalars_out) {
  if (!h || !h->have_problem) { set_error(h, "lcba_debug_step: no problem set"); return LCBA_E_STATE; }
  if (mode < 0 || mode > 2) { set_error(h, "lcba_debug_step: mode must be 0, 1 or 2"); return LCBA_E_ARG; }
  cudaSetDevice(h->device);
  Ctl init;
  memset(&init, 0, sizeof(init));
  init.term = -1;
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_ctl, &init, sizeof(Ctl), cudaMemcpyHostToDevice, h->stream));
  h->fix_cameras = mode == 1 ? 1 : 0;
  h->shared_intr = mode == 2 ? 1 : 0;
  h->masks_on = true;
  if (h->shared_intr && h->n_cam_held) {
    set_error(h, "lcba_debug_step: a camera mask together with shared intrinsics is not supported");
    return LCBA_E_UNSUPPORTED;
  }
  if ((h->fix_cameras ? 0 : (h->shared_intr ? 3 + 8LL * h->C : (long long)h->C * NCP - h->n_cam_held)) +
          3 * (h->P - h->n_pt_held) <= 0) {
    set_error(h, "lcba_debug_step: every parameter is held (lcba_set_fixed)");
    return LCBA_E_ARG;
  }
  // the bounded loop's damping and Gram diagonal at the current x (which must lie inside the box)
  BoxSetup box;
  LCBA_TRY(box_setup(h, h->fix_cameras != 0, box));
  h->bounded = false;
  if (box.flags & 1) {
    if (mode != 0) {
      set_error(h, "lcba_debug_step: box bounds are supported in mode 0 only");
      return LCBA_E_UNSUPPORTED;
    }
    if (box.flags & (2 | 8)) {    // on a bound, v = 0 and d = 0: the tap needs x strictly inside
      set_error(h, "lcba_debug_step: an empty box, or x not strictly inside the bounds (lcba_set_bounds)");
      return LCBA_E_ARG;
    }
    LCBA_TRY(box_upload(h, box, false));
    h->bounded = true;
  }
  LCBA_TRY(pass_linearize(h, 1));
  LCBA_TRY(pass_jdot(h));
  if (h->fix_cameras) {
    KL(h, "point_factor", k_point_factor<<<nblk(h->P, 256), 256, 0, h->stream>>>(
          h->d_Vg, h->d_scl_p, lam, nullptr, h->P, pt_mask(h), nullptr, h->d_Lz));
    LCBA_CUDA(h, cudaMemsetAsync(h->d_pc, 0, (size_t)h->C * NCP * 8, h->stream));
    LCBA_CUDA(h, cudaMemsetAsync(h->d_fail, 0, 2 * sizeof(int), h->stream));
  } else {
    LCBA_TRY(pass_schur(h, &lam));
    LCBA_TRY(pass_camera_solve(h, mu));
  }
  LCBA_TRY(pass_backsub(h));
  if (pc_out) LCBA_CUDA(h, cudaMemcpyAsync(pc_out, h->d_pc, (size_t)h->C * NCP * 8, cudaMemcpyDeviceToHost, h->stream));
  if (pp_out) LCBA_CUDA(h, cudaMemcpyAsync(pp_out, h->d_gn_p, (size_t)h->P * 3 * 8, cudaMemcpyDeviceToHost, h->stream));
  LCBA_TRY(read_ctl(h));
  if (scalars_out) {
    const Ctl& c = *h->h_ctl;
    const double v[LCBA_STEP_SCALARS] = {c.reg_term, c.Delta, c.Jg2, c.aa, c.ab, c.bb, c.JAA, c.JAB, c.JBB,
                                         c.gtgt, c.gtp, c.pp, c.c0, c.c1, c.predicted, c.step_h_norm,
                                         c.step_norm, (double)c.chol_fail};
    memcpy(scalars_out, v, sizeof(v));
  }
  return LCBA_OK;
}

// test hook: the digit planes of the int8 Schur path at the current x, damped with the host's lam, from
// k_i8_make (ref = 0) or k_i8_make_ref (ref = 1), which runs `reps` times on a plane buffer first filled with the
// byte `poison` (>= 0), so that a byte the kernel does not write shows
extern "C" int lcba_debug_i8_make(lcba_t* h, double lam, int32_t ref, int32_t reps, int32_t poison, double* ms_out,
                                  void* planes_out, int64_t planes_bytes) {
  if (!h || !h->have_problem) { set_error(h, "lcba_debug_i8_make: no problem set"); return LCBA_E_STATE; }
  if (!h->use_i8) { set_error(h, "lcba_debug_i8_make: the problem does not take the int8 path (LCBA_SCHUR_I8)"); return LCBA_E_STATE; }
  if (ref < 0 || ref > 1 || reps < 1 || poison < -1 || poison > 255 ||
      (planes_out && planes_bytes != (int64_t)h->i8plan.plane_bytes)) {
    set_error(h, "lcba_debug_i8_make: ref must be 0 or 1, reps >= 1, poison -1..255, planes_bytes = " +
                     std::to_string(h->i8plan.plane_bytes));
    return LCBA_E_ARG;
  }
  cudaSetDevice(h->device);
  Ctl init;
  memset(&init, 0, sizeof(init));
  init.term = -1;
  LCBA_CUDA(h, cudaMemcpyAsync(h->d_ctl, &init, sizeof(Ctl), cudaMemcpyHostToDevice, h->stream));
  h->masks_on = true;
  h->bounded = false;
  LCBA_TRY(pass_linearize(h, 1));
  KL(h, "point_factor", k_point_factor<<<nblk(h->P, 256), 256, 0, h->stream>>>(
        h->d_Vg, h->d_scl_p, lam, nullptr, h->P, pt_mask(h), nullptr, h->d_Lz));
  launch_i8_rowexp(h);
  if (poison >= 0) LCBA_CUDA(h, cudaMemsetAsync(h->d_i8planes, poison, h->i8plan.plane_bytes, h->stream));
  cudaEvent_t e0, e1;
  LCBA_CUDA(h, cudaEventCreate(&e0));
  if (cudaEventCreate(&e1) != cudaSuccess) { cudaEventDestroy(e0); set_error(h, "lcba_debug_i8_make: cudaEventCreate"); return LCBA_E_CUDA; }
  cudaError_t e = cudaEventRecord(e0, h->stream);
  for (int r = 0; r < reps && e == cudaSuccess; ++r) launch_i8_make(h, ref != 0);
  if (e == cudaSuccess) e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaEventRecord(e1, h->stream);
  if (e == cudaSuccess && planes_out)
    e = cudaMemcpyAsync(planes_out, h->d_i8planes, h->i8plan.plane_bytes, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  float ms = 0.0f;
  if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (e != cudaSuccess) { set_error(h, std::string("lcba_debug_i8_make: ") + cudaGetErrorString(e)); return LCBA_E_CUDA; }
  if (ms_out) *ms_out = (double)ms / reps;
  return LCBA_OK;
}

// host-only: is v[0..n) non-decreasing?  (dist.py: may the observation arrays be cut into contiguous ranges?)
extern "C" int lcba_host_is_nondecreasing_i64(const int64_t* v, int64_t n, int32_t threads) {
  if (!v || n < 2) return 1;
  const int nt = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(threads, 16), n / (1 << 20)));
  std::vector<int> ok(nt, 1);
  auto piece = [&](int i) {
    const int64_t a = n * i / nt, b = std::min<int64_t>(n, n * (i + 1) / nt + 1);      // one element of overlap
    int64_t bad = 0;
    for (int64_t k = a + 1; k < b; ++k) bad |= (int64_t)(v[k] < v[k - 1]);
    ok[i] = bad ? 0 : 1;
  };
  if (nt == 1) { piece(0); return ok[0]; }
  std::vector<std::thread> th;
  int started = 1;                                  // pieces [started, nt) fall back to this thread
  try {
    for (int i = 1; i < nt; ++i) { th.emplace_back(piece, i); started = i + 1; }
  } catch (...) {                                   // no more threads: nothing may cross the C boundary
  }
  piece(0);
  for (int i = started; i < nt; ++i) piece(i);
  for (auto& t : th) t.join();
  for (int i = 0; i < nt; ++i) if (!ok[i]) return 0;
  return 1;
}
