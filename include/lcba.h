/*
 * lcba.h — C-ABI of the B200-native bundle-adjustment engine (liblcba.so).
 *
 * Drop-in boundary for the bundle-adjustment step of JohnsonLabJanelia/laserCalib:
 * every entry point below replaces one member of the reference's `PySBA` class
 * (reference file lasercalib/pySBA.py) or the scipy call it makes.  The reference is
 * pure Python, so "the FFI it would bind" is a ctypes binding; INTEGRATION.md shows
 * the stub.  Plain C types only: host pointers to contiguous FP64 / int64 arrays exactly
 * as the reference's numpy arrays hand them over; no torch / CUDA types in signatures
 * (device pointers and streams cross the boundary as void* / uintptr).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (LCBA_E_*); the message is
 *     available from lcba_last_error(h) (h may be NULL for lcba_create failures);
 *   - one handle = one GPU = one host thread at a time (one process per GPU; ranks are
 *     joined with lcba_comm_init);
 *   - the library copies inputs to the device and owns all device memory;
 *   - camera vector layout [rotvec(3), t(3), f, k1, k2, cx, cy]  (pySBA.py:31-35);
 *   - residual layout [u0, v0, u1, v1, ...] in the CALLER's observation order
 *     (pySBA.py:100-101), also when the library re-sorts observations internally.
 *   - there is NO CPU fallback: without a CUDA device every compute call fails with
 *     LCBA_E_CUDA.
 */
#ifndef LCBA_H
#define LCBA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LCBA_VERSION 100          /* 0.1.0 */
#define LCBA_CAM_PARAMS 11
#define LCBA_MAX_CAMERAS 64       /* per-point visibility is a 64-bit mask */
#define LCBA_MAX_TRACE 512

enum {
  LCBA_OK = 0,
  LCBA_E_ARG = -1,        /* bad argument (null pointer, negative size, index out of range) */
  LCBA_E_CUDA = -2,       /* CUDA runtime error / no device */
  LCBA_E_STATE = -3,      /* call order (e.g. solve before set_problem) */
  LCBA_E_UNSUPPORTED = -4,/* >64 cameras, duplicate (camera, point) observation, ... */
  LCBA_E_NONFINITE = -5,  /* residuals not finite at the initial point
                             (scipy raises ValueError: _lsq/least_squares.py:945-946) */
  LCBA_E_NCCL = -6
};

/* scipy termination codes (scipy/optimize/_lsq/least_squares.py:23-31) */
enum {
  LCBA_STATUS_MAX_NFEV = 0,
  LCBA_STATUS_GTOL = 1,
  LCBA_STATUS_FTOL = 2,
  LCBA_STATUS_XTOL = 3,
  LCBA_STATUS_FTOL_XTOL = 4
};

typedef struct lcba_handle lcba_t;

/* Options of one bundleAdjust call.  Defaults (lcba_default_options) reproduce the
 * reference call `least_squares(fun, x0, jac_sparsity=A, x_scale='jac', ftol=ftol,
 * method='trf', jac='3-point')` (pySBA.py:141-142): xtol = gtol = 1e-8,
 * max_nfev = 100 * n. */
typedef struct lcba_options {
  double ftol;
  double xtol;
  double gtol;
  int64_t max_nfev;   /* <=0: 100 * (11 C + 3 P) */
  int32_t verbose;    /* 2: keep a per-iteration trace (the host prints scipy's table) */
  int32_t profile;    /* 1: bracket every kernel launch with CUDA events (lcba_get_profile) */
  int32_t max_iterations; /* >0: stop after this many outer iterations (bench: time exactly K) */
  int32_t fix_cameras;    /* 1: optimise the 3-D points only (PySBA.bundleAdjust_nocam,
                             pySBA.py:237-250): x = points, cameras stay at their values */
  int32_t shared_intrinsics; /* 1: one (f, k1, k2) for all cameras (PySBA.bundleAdjust_sharedcam,
                                pySBA.py:252-325); the caller passes cameras whose columns 6..8
                                are identical */
  int32_t reserved[3];
} lcba_options;

/* One row of scipy's verbose=2 table (_lsq/common.py:545-563). */
typedef struct lcba_trace_row {
  int64_t iteration;
  int64_t nfev;
  double cost;
  double cost_reduction;  /* NaN on row 0 */
  double step_norm;       /* NaN on row 0 */
  double optimality;
  double delta;           /* trust radius when the row was emitted */
  double reg_term;        /* damping of the iteration that produced this row */
} lcba_trace_row;

typedef struct lcba_result {
  double cost;            /* 0.5 * |f|^2 at the returned x */
  double optimality;      /* |J^T f|_inf */
  double initial_cost;
  int64_t nfev;
  int64_t njev;
  int64_t iterations;     /* outer iterations completed */
  int32_t status;         /* LCBA_STATUS_* */
  int32_t n_trace;        /* rows valid in lcba_get_trace */
  double solve_ms;        /* device time of the whole loop (CUDA events) */
  int64_t gpu_launches;   /* kernels launched by this call */
  double reserved[6];     /* [0] = CUDA-graph replays inside this solve (0 on the first solve of a problem) */
} lcba_result;

/* Per-kernel device time (profile=1), accumulated over a solve. */
typedef struct lcba_kernel_stat {
  char name[32];
  int64_t launches;
  double total_ms;
} lcba_kernel_stat;

/* ---- lifecycle ------------------------------------------------------------------ */
int lcba_version(void);
/* device < 0: use the current CUDA device. */
int lcba_create(lcba_t** out, int device);
void lcba_destroy(lcba_t* h);
const char* lcba_last_error(const lcba_t* h);
void lcba_default_options(lcba_options* o);

/* ---- PySBA.__init__ (pySBA.py:28-59) ----------------------------------------------
 * cams C x 11, pts P x 3, obs_uv N x 2 (row-major FP64); cam_idx / pt_idx N int64;
 * weights N FP64 or NULL (the reference's default is integer ones).  Observations in any
 * order; the library validates indices, sorts point-major / camera-ascending on the
 * device when needed and remembers the permutation.  A (camera, point) pair observed more
 * than once is accepted like the reference accepts it (one more residual pair each; the
 * reference's own dataset concatenation produces such rows for 3 or more laser datasets,
 * calibrate_camera.py:41-44). */
int lcba_set_problem(lcba_t* h, int32_t C, int64_t P, int64_t N, const double* cams,
                     const double* pts, const double* obs_uv, const int64_t* cam_idx,
                     const int64_t* pt_idx, const double* weights_or_null);
/* Same for one shard of a point-sharded job: pts holds the shard's P points, pt_idx may keep the
 * caller's GLOBAL point indices, pt_offset = global index of the shard's first point. */
int lcba_set_problem_shard(lcba_t* h, int32_t C, int64_t P, int64_t N, const double* cams,
                           const double* pts, const double* obs_uv, const int64_t* cam_idx,
                           const int64_t* pt_idx, const double* weights_or_null, int64_t pt_offset);
/* Replace the current parameter vector x = [cams.ravel(), pts.ravel()]. */
int lcba_set_params(lcba_t* h, const double* cams, const double* pts);
/* Hold parameters at their current values: cam_fixed C x 11 bytes (row-major like cams), pt_fixed one byte
 * per point of THIS handle's P points (its shard on a point-sharded job); nonzero = held, NULL clears that
 * mask.  A masked lcba_solve is scipy's trf_no_bounds on the free sub-vector with the same residuals: the
 * Jacobi scaling, the initial Delta, reg_term, the 2-D subspace, |x| (xtol) and |g|_inf (gtol, optimality)
 * run over free entries only, max_nfev defaults to 100 * n_free, and held entries of x come back
 * bit-identical.  The masks apply to lcba_solve and lcba_debug_step (and lcba_debug_i8_make); lcba_get_grad
 * after them returns 0 at held entries.  lcba_linearize stays the unmasked tap.  lcba_set_problem /
 * lcba_set_problem_shard clear both masks, lcba_set_params keeps them.  The point mask combines with
 * fix_cameras and shared_intrinsics; a camera mask with shared_intrinsics makes lcba_solve return
 * LCBA_E_UNSUPPORTED, nothing free LCBA_E_ARG.  Sharded jobs: the camera mask must be the same on every
 * rank (lcba_solve compares its count and checksum over the ranks and fails on every rank otherwise). */
int lcba_set_fixed(lcba_t* h, const uint8_t* cam_fixed, const uint8_t* pt_fixed);
/* PySBA.optimizedParams (pySBA.py:121-129): copy x back, split. */
int lcba_get_params(lcba_t* h, double* cams_out, double* pts_out);

/* ---- PySBA.rotate / PySBA.project (pySBA.py:61-89) --------------------------------
 * Row-wise on already-gathered arrays, per-row rotation vector / camera vector. */
int lcba_rotate(lcba_t* h, int64_t M, const double* pts, const double* rot_vecs, double* out);
int lcba_project(lcba_t* h, int64_t M, const double* pts, const double* cams_rows,
                 double* out_uv);

/* ---- 3-D initialisation: Unproject (lasercalib/rigid_body.py:205-243) -----------------
 * Pixels of the reference camera -> world points on the plane(s) z = Z: OpenCV's iterative
 * undistortPoints (5 iterations) + ray/plane intersection.  camera_matrix 3x3 row-major,
 * dist 5 (k1 k2 p1 p2 k3), rc_ext 3x3 row-major, tc_ext 3; Z has nZ = 1 or M entries. */
int lcba_unproject(lcba_t* h, int64_t M, const double* uv, const double* Z, int64_t nZ,
                   const double* camera_matrix, const double* dist5, const double* rc_ext,
                   const double* tc_ext, double* out_xyz);

/* ---- squared-residual variants: fun_camonly (pySBA.py:151-156, driver :160-173) and
 * fun_transform_points_3d (pySBA.py:176-188, driver :191-206) --------------------------
 * f = w (proj - obs)^2 per pixel coordinate; the reference hands these to a DENSE scipy
 * least_squares.  One pass over the resident observations returns cost = 0.5 sum f^2,
 * g = J^T f and J^T J (analytic J = 2 w e dproj/dtheta); the n x n trust-region arithmetic
 * stays with the caller (lasercalib_b200/_trf_dense.py).
 *   LCBA_SQ_CAMONLY  : theta = (C,11) cameras, the handle's points fixed;
 *                      g (11C), H (C,11,11) = the diagonal blocks (cameras do not couple)
 *   LCBA_SQ_TRANSFORM: theta = 12 = rows of [A|t] applied to the handle's points, the
 *                      handle's cameras fixed; g (12), H (12,12)
 * g and H both NULL = cost only.  Sums run over this handle's observations only (no
 * collective: under torchrun the variants run as replicas). */
#define LCBA_SQ_CAMONLY 0
#define LCBA_SQ_TRANSFORM 1
int lcba_sq_normal(lcba_t* h, int32_t mode, const double* theta, double* cost_out, double* g_out,
                   double* H_out);

/* ---- PySBA.fun (pySBA.py:92-101) --------------------------------------------------
 * x_or_null: 11C + 3P parameters (NULL = the handle's current x). r_out: 2N or NULL.
 * cost_out != NULL: 0.5 |f|^2 over ALL ranks (collective on a point-sharded job: every rank
 * must call); cost_out == NULL: this handle's residuals only, no collective. */
int lcba_residuals(lcba_t* h, const double* x_or_null, double* r_out, double* cost_out);

/* ---- the Jacobian scipy differentiates numerically (scipy/optimize/_numdiff.py:770) --
 * Analytic blocks in the caller's observation order: Jc N x 2 x 11, Jp N x 2 x 3. */
int lcba_jacobian_blocks(lcba_t* h, const double* x_or_null, double* Jc, double* Jp);

/* ---- PySBA.bundle_adjustment_sparsity (pySBA.py:103-118) --------------------------
 * Column indices of the (2N, 11C+3P) 0/1 pattern in CSR order, 28 per observation,
 * each row sorted ascending: indices_out has 2*N*14 int32 entries (indptr = 14*i). */
int lcba_sparsity_indices(lcba_t* h, int32_t C, int64_t P, int64_t N, const int64_t* cam_idx,
                          const int64_t* pt_idx, int32_t* indices_out);

/* ---- PySBA.bundleAdjust (pySBA.py:132-147) ----------------------------------------
 * Trust-region-reflective loop of scipy (trf_no_bounds, _lsq/trf.py:415-587) with an
 * analytic Jacobian and the exact Schur-complement solution of the regularised normal
 * equations in place of LSMR.  Updates the handle's x in place. */
int lcba_solve(lcba_t* h, const lcba_options* opt, lcba_result* res);
int lcba_get_trace(lcba_t* h, lcba_trace_row* rows, int32_t max_rows);
/* Called by lcba_solve, on the calling thread, as soon as a row of scipy's verbose=2 table is
 * known: scipy prints the table live (least_squares(verbose=2), pySBA.py:141;
 * _lsq/common.py:551-563), so the host prints from here.  cb == NULL clears it. */
typedef void (*lcba_iteration_cb)(const lcba_trace_row* row, void* user);
int lcba_set_iteration_callback(lcba_t* h, lcba_iteration_cb cb, void* user);
int lcba_get_grad(lcba_t* h, double* g_out /* 11C + 3P, at the current x */);
int lcba_get_profile(lcba_t* h, lcba_kernel_stat* stats, int32_t max_stats, int32_t* n_out);

/* ---- debug / parity taps -----------------------------------------------------------
 * Linearise at the current x and form the damped reduced camera system
 *   S = U + lam*Dc^2 - sum_p W (V + lam*Dp^2)^-1 W^T,  rhs = gc - sum_p W (V+lam*Dp^2)^-1 gp
 * with D = column norms of J (first-call Jacobi scaling).  Any output may be NULL.
 * Ignores the masks of lcba_set_fixed (every parameter free): the unmasked debug tap.
 * S_out (11C)^2 full symmetric, rhs_out 11C, grad_out 11C+3P, scale_inv_out 11C+3P. */
int lcba_linearize(lcba_t* h, double lam, double* S_out, double* rhs_out, double* grad_out,
                   double* scale_inv_out, double* cost_out);

/* ---- device-resident timing (bench) ------------------------------------------------
 * what: 0 = residual only (fun), 1 = residual + Jacobian blocks written to HBM (M1),
 *       2 = linearise + Schur + solve + back-substitution (one Gauss-Newton system).
 * Runs `reps` times on resident data; ms_out = mean device time per repetition. */
int lcba_time_device(lcba_t* h, int32_t what, int32_t reps, double* ms_out);

/* ---- multi-GPU: one process per GPU, points sharded by the host -------------------
 * Each rank calls lcba_set_problem with ITS shard (local point indices, all cameras).
 * Camera-block sums, the reduced camera system and the scalar sums are all-reduced with
 * NCCL inside lcba_solve / lcba_linearize.  The unique id is created on rank 0 and
 * distributed by the host (torch.distributed broadcast). */
int lcba_nccl_unique_id(void* id_out128);
/* id128 != NULL: create the process-wide communicator (collective over all ranks);
 * id128 == NULL: attach the communicator this process created earlier to another handle. */
int lcba_comm_init(lcba_t* h, int32_t rank, int32_t nranks, const void* id128);
/* total point count over all ranks is needed for max_nfev = 100*n and is all-reduced, together with
 * the held point count and the camera mask's count and checksum (lcba_set_fixed). */

/* ---- test hook -----------------------------------------------------------------------
 * The 2-D trust-region sub-problem solver the device control kernel uses
 * (scipy/optimize/_lsq/common.py:171-219), callable on the host for unit tests. */
int lcba_debug_tr2d(double B00, double B01, double B11, double g0, double g1, double Delta,
                    double* p_out2, int* newton_out);

/* The dense camera solve of the solver (csrc/dense.cuh: k_copy_damped_rhs + k_chol_fused) on a host
 * system: Cholesky of A + mu*diag(d^2) (A n x n row-major, lower triangle read; 1 <= n <= 704) and
 * x = (A + mu*diag(d^2))^-1 rhs, with `grid` cooperative CTAs (0: the solver's own choice; above the
 * co-resident limit: LCBA_E_ARG).  d may be NULL when mu == 0.  x_out n; factor_out (n+1) x n or NULL:
 * the work buffer as the kernel leaves it (strict lower triangle L, 1 / l_jj on the diagonal, row n =
 * z = L^-1 rhs, upper triangle untouched); fail_out: bit 0 = non-positive or NaN pivot, bit 1 = grid
 * barrier timed out. */
int lcba_debug_chol(lcba_t* h, int32_t n, const double* A, const double* rhs, double mu, const double* d,
                    int32_t grid, double* x_out, double* factor_out, int32_t* fail_out);

/* One Gauss-Newton step of the solver on the resident problem at its current x, through the same
 * kernels lcba_solve launches: linearise (first-call scaling, Delta = |x * scale_inv|), the Cauchy
 * reg_term, point factors and the reduced camera system damped with `lam` (it overrides reg_term,
 * like lcba_linearize), the dense camera solve with extra damping mu * Dc^2, back-substitution and the
 * 2-D subspace scalars.  mode 0: all parameters; 1: cameras fixed (fix_cameras); 2: shared
 * intrinsics; the masks of lcba_set_fixed apply (held entries of the step are 0).  pc_out 11C (the camera step, expanded in mode 2; zeros in mode 1), pp_out 3P (the
 * point step); scalars_out LCBA_STEP_SCALARS doubles:
 *   [0] reg_term  [1] Delta  [2] Jg2 = |J D^-2 g|^2
 *   [3] aa  [4] ab  [5] bb      (a = g_h = g / s, b = gn_h = p * s, scaled space)
 *   [6] JAA [7] JAB [8] JBB     (|J D^-2 g|^2, (J D^-2 g).(J p), |J p|^2)
 *   [9] gtgt [10] gtp [11] pp   (g~ = D^-2 g and p, unscaled)
 *   [12] c0 [13] c1 [14] predicted [15] step_h_norm [16] step_norm  (step = c0 g~ + c1 p)
 *   [17] fail word of the camera solve (as in lcba_debug_chol). */
#define LCBA_STEP_SCALARS 18
int lcba_debug_step(lcba_t* h, double lam, double mu, int32_t mode, double* pc_out, double* pp_out,
                    double* scalars_out);

/* The digit planes of the int8 tensor-core Schur path on the resident problem at its current x: linearise,
 * point factors damped with `lam`, row maxima and exponents, then `reps` launches of the plane kernel,
 * k_i8_make (ref = 0) or the reference k_i8_make_ref (ref = 1).  poison 0..255: the plane buffer is filled
 * with that byte before the launches (outside the timed window), so that bytes the kernel leaves unwritten
 * show; -1: it is left as it is.  ms_out: CUDA-event time per launch of the plane kernel.  planes_out (may be
 * NULL): the planes after the last launch, planes_bytes bytes, which must equal the plane buffer's size
 * (K blocks x 6 digits x row groups x 512).  LCBA_E_STATE when the problem does not take the int8 path.  Synchronises the handle's stream; not part of lcba_solve. */
int lcba_debug_i8_make(lcba_t* h, double lam, int32_t ref, int32_t reps, int32_t poison, double* ms_out,
                       void* planes_out, int64_t planes_bytes);

/* ---- profiling hook --------------------------------------------------------------------
 * Per-CTA cycle counters of the last Schur launch (4 int64 per CTA, [kind][slice]); only
 * filled when the process runs with LCBA_SCHUR_STATS=1 (tools/schur_stats.py). */
int lcba_debug_schur_stats(lcba_t* h, long long* out, int max_ctas, int* nkinds, int* nslices);

/* Host-only: the unit plan of the tensor-path Schur kernel (schur_mma.cuh) for C cameras; per
 * kind 8 rows of (first tile row, first tile column, tile rows, tile columns, triangular), a
 * row of zeros = idle warp.  Returns the number of kinds (needs no GPU). */
int lcba_debug_mma_plan(int32_t C, int32_t sm_count, int32_t* units_out, int32_t max_kinds,
                        int32_t* nslices_out, int32_t* ok_out);

/* Host-only: the strip plan of the int8 tensor-core Schur kernel (schur_i8.cuh) for C cameras and P
 * points (the plan the kernel runs may be the cover plan instead: lcba_debug_i8_cover_plan).  tiles_out: per tile 8 ints (first row group of the rows, row groups; column block 1: first row
 * group, row groups; column block 2 (the folded left-over rows, transposed): first row group, row groups;
 * first CTA, CTAs); work_out: per CTA (index, first K block, end K block).
 * Returns the number of tiles (needs no GPU). */
int lcba_debug_i8_plan(int32_t C, int64_t P, int32_t sm_count, int32_t* tiles_out, int32_t max_tiles,
                       int32_t* work_out, int32_t max_work, int32_t* nwork_out, int32_t* nrg_out,
                       int64_t* nkb_out);

/* Host-only: a tile / CTA plan of the int8 tensor-core Schur kernel with both row ranges of its A operand.
 * which: 0 = the plan the kernel runs (the cost model's choice, without LCBA_I8_PLAN), 1 = the strip plan,
 * 2 = the cover plan.  tiles_out: per tile 10 ints (rows: range 1 first row group, row groups, range 2 first
 * row group, row groups; column block 1 and 2: first row group, row groups each; first CTA, CTAs); work_out:
 * per CTA (tile, first K block, end K block); model_out: 4 doubles (executed int8 ops of one launch, slowest
 * CTA of the cost model in cycles of the MMA warp for this plan, the strip plan and the cover plan).
 * *cover_out: 1 when the plan is the cover plan.  Returns the number of tiles (needs no GPU). */
int lcba_debug_i8_cover_plan(int32_t C, int64_t P, int32_t sm_count, int32_t which, int32_t* tiles_out,
                             int32_t max_tiles, int32_t* work_out, int32_t max_work, int32_t* nwork_out,
                             int32_t* nrg_out, int64_t* nkb_out, int32_t* cover_out, double* model_out);

/* Host-only: the K blocks every CTA of a tile plan (which as above) reads, under the K-major schedule (kmajor = 1, the
 * default) or one contiguous K range per CTA (kmajor = 0, LCBA_I8_SCHED=range).  work_out: per CTA 6 ints (tile,
 * kb0, kb1, kfirst, kc, kstride): the K blocks kfirst + (i / kc) kstride + i % kc for i < kb1 - kb0.  *window_out:
 * how many K blocks a CTA may run ahead of the slowest one (0: no window).  Returns the number of CTAs. */
int lcba_debug_i8_schedule(int32_t C, int64_t P, int32_t sm_count, int32_t which, int32_t kmajor, int32_t* work_out,
                           int32_t max_work, int32_t* window_out);

/* 1 when the last Schur pass of the int8 tensor-core path found a camera row whose largest |Y| entry is more
 * than 4x the square root of its Schur diagonal (finer than the 48-bit digits resolve) and recomputed the
 * pass with the FP64 DMMA kernel; 0 when the int8 result stood; -1 when the handle does not use the int8
 * path.  Synchronises the handle's stream. */
int lcba_debug_i8_fallback(lcba_t* h);

/* Measurement switch (tools/peer_ab.py): all-reduce through NVLink peer memory (csrc/peer_reduce.cuh; needs LCBA_PEER_REDUCE=1 or 2 at
 * lcba_comm_init so that every rank has mapped every peer's block) or through ncclAllReduce, from the next call on.  Collective in the
 * sense that every rank must switch at the same point.  Returns 1 if the peer path is active afterwards. */
int lcba_debug_peer_reduce(lcba_t* h, int enable);

/* Host-only helper of the sharding layer (lasercalib_b200/dist.py): 1 when v[0..n) is non-decreasing.  The
 * reference keeps its observations point-major (scripts/get_points3d.py:74-86); the host mirror must verify
 * that before it may cut contiguous observation ranges, on every call (the arrays are the caller's).  One
 * streaming read on up to `threads` threads (numpy needs two reads and a temporary: 60 ms for 24 M indices). */
int lcba_host_is_nondecreasing_i64(const int64_t* v, int64_t n, int32_t threads);

#ifdef __cplusplus
}
#endif
#endif /* LCBA_H */
