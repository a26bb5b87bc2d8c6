"""ctypes binding of liblcba.so (include/lcba.h).  No CPU fallback: if the shared library
is missing or cannot be loaded the import of the engine fails loudly."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "liblcba.so")

LCBA_MAX_TRACE = 512
E_NAMES = {-1: "LCBA_E_ARG", -2: "LCBA_E_CUDA", -3: "LCBA_E_STATE", -4: "LCBA_E_UNSUPPORTED",
           -5: "LCBA_E_NONFINITE", -6: "LCBA_E_NCCL", -7: "LCBA_E_SINGULAR"}
E_SINGULAR = -7

# every symbol include/lcba.h declares (tests/test_cabi.py checks the export list)
SYMBOLS = ["lcba_version", "lcba_create", "lcba_destroy", "lcba_last_error", "lcba_default_options",
           "lcba_set_problem", "lcba_set_problem_shard", "lcba_set_params", "lcba_get_params", "lcba_rotate", "lcba_project",
           "lcba_unproject", "lcba_residuals", "lcba_jacobian_blocks", "lcba_sparsity_indices", "lcba_solve",
           "lcba_get_trace", "lcba_get_grad", "lcba_get_profile", "lcba_linearize",
           "lcba_time_device", "lcba_nccl_unique_id", "lcba_comm_init", "lcba_debug_tr2d",
           "lcba_sq_normal", "lcba_debug_schur_stats", "lcba_debug_mma_plan",
           "lcba_set_iteration_callback", "lcba_debug_i8_plan", "lcba_host_is_nondecreasing_i64", "lcba_debug_peer_reduce",
           "lcba_debug_i8_fallback", "lcba_debug_chol", "lcba_debug_step", "lcba_debug_i8_cover_plan",
           "lcba_debug_i8_make", "lcba_set_fixed", "lcba_debug_i8_schedule", "lcba_set_bounds",
           "lcba_get_active_mask", "lcba_covariance"]

# scalars_out of lcba_debug_step, in order (include/lcba.h)
STEP_SCALARS = ["reg_term", "Delta", "Jg2", "aa", "ab", "bb", "JAA", "JAB", "JBB", "gtgt", "gtp", "pp",
                "c0", "c1", "predicted", "step_h_norm", "step_norm", "chol_fail"]


class Options(C.Structure):
    _fields_ = [("ftol", C.c_double), ("xtol", C.c_double), ("gtol", C.c_double),
                ("max_nfev", C.c_int64), ("verbose", C.c_int32), ("profile", C.c_int32),
                ("max_iterations", C.c_int32), ("fix_cameras", C.c_int32), ("shared_intrinsics", C.c_int32), ("reserved", C.c_int32 * 3)]


class TraceRow(C.Structure):
    _fields_ = [("iteration", C.c_int64), ("nfev", C.c_int64), ("cost", C.c_double),
                ("cost_reduction", C.c_double), ("step_norm", C.c_double),
                ("optimality", C.c_double), ("delta", C.c_double), ("reg_term", C.c_double)]


class Result(C.Structure):
    _fields_ = [("cost", C.c_double), ("optimality", C.c_double), ("initial_cost", C.c_double),
                ("nfev", C.c_int64), ("njev", C.c_int64), ("iterations", C.c_int64),
                ("status", C.c_int32), ("n_trace", C.c_int32), ("solve_ms", C.c_double),
                ("gpu_launches", C.c_int64), ("reserved", C.c_double * 6)]


class KernelStat(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("launches", C.c_int64), ("total_ms", C.c_double)]


ITERATION_CB = C.CFUNCTYPE(None, C.POINTER(TraceRow), C.c_void_p)


def _row_dict(r):
    return dict(iteration=r.iteration, nfev=r.nfev, cost=r.cost, cost_reduction=r.cost_reduction,
                step_norm=r.step_norm, optimality=r.optimality, delta=r.delta, reg_term=r.reg_term)


class LcbaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s (%d): %s" % (E_NAMES.get(code, "LCBA_E_?"), code, msg))
        self.code = code


_lib = None


def load():
    """dlopen liblcba.so and declare prototypes.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "lasercalib_b200: %s is missing — build it with `python -m lasercalib_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    pd = C.POINTER(C.c_double)
    lib.lcba_version.restype = C.c_int
    lib.lcba_create.argtypes = [C.POINTER(vp), C.c_int]
    lib.lcba_destroy.argtypes = [vp]
    lib.lcba_destroy.restype = None
    lib.lcba_last_error.argtypes = [vp]
    lib.lcba_last_error.restype = C.c_char_p
    lib.lcba_default_options.argtypes = [C.POINTER(Options)]
    lib.lcba_default_options.restype = None
    lib.lcba_set_problem.argtypes = [vp, i32, i64, i64, vp, vp, vp, vp, vp, vp]
    lib.lcba_set_problem_shard.argtypes = [vp, i32, i64, i64, vp, vp, vp, vp, vp, vp, i64]
    lib.lcba_set_params.argtypes = [vp, vp, vp]
    lib.lcba_get_params.argtypes = [vp, vp, vp]
    lib.lcba_set_fixed.argtypes = [vp, vp, vp]
    lib.lcba_set_bounds.argtypes = [vp, vp, vp, vp, vp]
    lib.lcba_get_active_mask.argtypes = [vp, dbl, vp]
    lib.lcba_covariance.argtypes = [vp, vp, vp, pd, pd]
    lib.lcba_rotate.argtypes = [vp, i64, vp, vp, vp]
    lib.lcba_project.argtypes = [vp, i64, vp, vp, vp]
    lib.lcba_unproject.argtypes = [vp, i64, vp, vp, i64, vp, vp, vp, vp, vp]
    lib.lcba_residuals.argtypes = [vp, vp, vp, pd]
    lib.lcba_jacobian_blocks.argtypes = [vp, vp, vp, vp]
    lib.lcba_sparsity_indices.argtypes = [vp, i32, i64, i64, vp, vp, vp]
    lib.lcba_solve.argtypes = [vp, C.POINTER(Options), C.POINTER(Result)]
    lib.lcba_get_trace.argtypes = [vp, C.POINTER(TraceRow), i32]
    lib.lcba_set_iteration_callback.argtypes = [vp, ITERATION_CB, vp]
    lib.lcba_get_grad.argtypes = [vp, vp]
    lib.lcba_get_profile.argtypes = [vp, C.POINTER(KernelStat), i32, C.POINTER(i32)]
    lib.lcba_linearize.argtypes = [vp, dbl, vp, vp, vp, vp, pd]
    lib.lcba_time_device.argtypes = [vp, i32, i32, pd]
    lib.lcba_nccl_unique_id.argtypes = [vp]
    lib.lcba_comm_init.argtypes = [vp, i32, i32, vp]
    lib.lcba_sq_normal.argtypes = [vp, i32, vp, pd, vp, vp]
    lib.lcba_debug_mma_plan.argtypes = [i32, i32, vp, i32, C.POINTER(i32), C.POINTER(i32)]
    lib.lcba_debug_schur_stats.argtypes = [vp, vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.lcba_debug_i8_plan.argtypes = [i32, i64, i32, vp, i32, vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)]
    lib.lcba_debug_i8_cover_plan.argtypes = [i32, i64, i32, i32, vp, i32, vp, i32, C.POINTER(i32), C.POINTER(i32),
                                             C.POINTER(i64), C.POINTER(i32), vp]
    lib.lcba_debug_i8_schedule.argtypes = [i32, i64, i32, i32, i32, vp, i32, C.POINTER(i32)]
    lib.lcba_host_is_nondecreasing_i64.argtypes = [vp, i64, i32]
    lib.lcba_debug_peer_reduce.argtypes = [vp, i32]
    lib.lcba_debug_i8_fallback.argtypes = [vp]
    lib.lcba_debug_tr2d.argtypes = [dbl, dbl, dbl, dbl, dbl, dbl, pd, C.POINTER(C.c_int)]
    lib.lcba_debug_chol.argtypes = [vp, i32, vp, vp, dbl, vp, i32, vp, vp, C.POINTER(i32)]
    lib.lcba_debug_step.argtypes = [vp, dbl, dbl, i32, vp, vp, vp]
    lib.lcba_debug_i8_make.argtypes = [vp, dbl, i32, i32, i32, pd, vp, i64]
    _lib = lib
    return lib


def i8_plane_bytes(n_cams, n_points):
    """Bytes of the int8 path's digit planes (schur_i8.cuh): K blocks of 21 points x 6 digits x row groups of 8
    of the 11 C + 1 rows, rounded up to an even count, x 512."""
    nrg = (11 * n_cams + 1 + 7) // 8
    nrg += nrg & 1
    return -(-n_points // 21) * 6 * nrg * 512


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


class Engine:
    """One GPU handle (lcba_t*).  Thin, explicit mirror of the C-ABI."""

    def __init__(self, device=-1):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.lcba_create(C.byref(h), int(device))
        if rc != 0:
            raise LcbaError(rc, self.lib.lcba_last_error(None).decode())
        self.h = h
        self.C = self.P = self.N = 0
        self.has_fixed = False     # a mask of set_fixed is in place (set_problem clears it)
        self.has_bounds = False    # bounds of set_bounds are in place (set_problem clears them)
        # bumped by every call that changes what the handle holds (observation set or x): lazy
        # readers (res.fun / res.grad / res.jac) compare it with the value they were created at
        self.generation = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.lcba_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise LcbaError(rc, self.lib.lcba_last_error(self.h).decode())

    # ---- problem ----
    def set_problem(self, cams, pts, points_2d, camera_ind, point_ind, weights=None, pt_offset=0):
        cams, pts = _f64(cams), _f64(pts)
        p2 = _f64(points_2d)
        ci, pi = _i64(camera_ind).ravel(), _i64(point_ind).ravel()
        w = None if weights is None else _f64(weights).ravel()
        if cams.ndim != 2 or cams.shape[1] != 11:
            raise ValueError("cameraArray must have shape (n_cameras, 11)")
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError("points3D must have shape (n_points, 3)")
        N = ci.size
        if pi.size != N or p2.shape != (N, 2) or (w is not None and w.size != N):
            raise ValueError("observation arrays must share their first dimension")
        self._check(self.lib.lcba_set_problem_shard(self.h, cams.shape[0], pts.shape[0], N,
                                                    _ptr(cams), _ptr(pts), _ptr(p2), _ptr(ci),
                                                    _ptr(pi), _ptr(w), int(pt_offset)))
        self.C, self.P, self.N = cams.shape[0], pts.shape[0], N
        self.has_fixed = False
        self.has_bounds = False
        self.generation += 1

    def set_params(self, cams, pts):
        self.generation += 1
        cams, pts = _f64(cams, (self.C, 11)), _f64(pts, (self.P, 3))
        self._check(self.lib.lcba_set_params(self.h, _ptr(cams), _ptr(pts)))

    def set_fixed(self, cam_fixed=None, pt_fixed=None):
        """Hold parameters at their current values in solve() and debug_step() (lcba_set_fixed):
        cam_fixed bool (C, 11), pt_fixed bool (P,) over this handle's points; None clears that mask."""
        cm = None if cam_fixed is None else np.ascontiguousarray(cam_fixed, dtype=np.uint8)
        pm = None if pt_fixed is None else np.ascontiguousarray(pt_fixed, dtype=np.uint8)
        if cm is not None and cm.shape != (self.C, 11):
            raise ValueError("cam_fixed must have shape (%d, 11)" % self.C)
        if pm is not None and pm.shape != (self.P,):
            raise ValueError("pt_fixed must have shape (%d,)" % self.P)
        self._check(self.lib.lcba_set_fixed(self.h, _ptr(cm), _ptr(pm)))
        self.has_fixed = cm is not None or pm is not None

    def set_bounds(self, cam_lb=None, cam_ub=None, pt_lb=None, pt_ub=None):
        """Box bounds for solve() and debug_step() (lcba_set_bounds): (C, 11) camera and (P, 3) point arrays over
        this handle's points, +-inf allowed; None leaves that side unbounded, four None clear the bounds."""
        arrs = [None if a is None else _f64(a, shape) for a, shape in
                ((cam_lb, (self.C, 11)), (cam_ub, (self.C, 11)), (pt_lb, (self.P, 3)), (pt_ub, (self.P, 3)))]
        self._check(self.lib.lcba_set_bounds(self.h, *[_ptr(a) for a in arrs]))
        self.has_bounds = any(a is not None for a in arrs)

    def active_mask(self, rtol):
        """find_active_constraints(x, lb, ub, rtol) at the current x (lcba_get_active_mask), int8 (11 C + 3 P,)."""
        out = np.empty(11 * self.C + 3 * self.P, dtype=np.int8)
        self._check(self.lib.lcba_get_active_mask(self.h, float(rtol), _ptr(out)))
        return out

    def get_params(self, x_out=None):
        """(cams, pts) of the current iterate; with `x_out` (11 C + 3 P doubles, contiguous) the
        two arrays are views into it, i.e. x_out becomes the reference's parameter vector."""
        if x_out is None:
            cams = np.empty((self.C, 11))
            pts = np.empty((self.P, 3))
        else:
            cams = x_out[: 11 * self.C].reshape(self.C, 11)
            pts = x_out[11 * self.C:].reshape(self.P, 3)
        self._check(self.lib.lcba_get_params(self.h, _ptr(cams), _ptr(pts)))
        return cams, pts

    # ---- model ----
    def rotate(self, points, rot_vecs):
        points, rot_vecs = _f64(points), _f64(rot_vecs)
        out = np.empty_like(points)
        self._check(self.lib.lcba_rotate(self.h, points.shape[0], _ptr(points), _ptr(rot_vecs),
                                         _ptr(out)))
        return out

    def project(self, points, cam_rows):
        points, cam_rows = _f64(points), _f64(cam_rows)
        if points.shape[0] != cam_rows.shape[0]:
            raise ValueError("operands could not be broadcast together with shapes %s %s"
                             % (points.shape, cam_rows.shape))
        out = np.empty((points.shape[0], 2))
        self._check(self.lib.lcba_project(self.h, points.shape[0], _ptr(points), _ptr(cam_rows),
                                          _ptr(out)))
        return out

    def unproject(self, points, Z, intrinsic, distortion, rotation_matrix, tvec):
        points = _f64(points)
        Zv = _f64(np.atleast_1d(Z)).ravel()
        K, R = _f64(intrinsic, (3, 3)), _f64(rotation_matrix, (3, 3))
        d = np.zeros(5)
        dv = _f64(distortion).ravel()
        d[: min(5, dv.size)] = dv[:5]
        t = _f64(tvec).ravel()[:3].copy()
        out = np.empty((points.shape[0], 3))
        self._check(self.lib.lcba_unproject(self.h, points.shape[0], _ptr(points), _ptr(Zv), Zv.size,
                                            _ptr(K), _ptr(d), _ptr(R), _ptr(t), _ptr(out)))
        return out

    def residuals(self, x=None, want_r=True, want_cost=True):
        """(r, cost).  want_cost=False: this handle's residuals only and NO collective, so one
        rank of a point-sharded job may call it alone (cost is returned as None)."""
        x = None if x is None else _f64(x).ravel()
        if x is not None and x.size != 11 * self.C + 3 * self.P:
            raise ValueError("params has the wrong size")
        r = np.empty(2 * self.N) if want_r else None
        cost = C.c_double()
        self._check(self.lib.lcba_residuals(self.h, _ptr(x), _ptr(r),
                                            C.byref(cost) if want_cost else None))
        return r, (cost.value if want_cost else None)

    SQ_CAMONLY, SQ_TRANSFORM = 0, 1

    def sq_normal(self, mode, theta, derivs=True):
        """(cost, g, H) of the squared-residual variants at theta (lcba_sq_normal): camera-only
        mode returns H as the (C,11,11) diagonal blocks, transform mode as (12,12)."""
        theta = _f64(theta).ravel()
        n = 11 * self.C if mode == self.SQ_CAMONLY else 12
        if theta.size != n:
            raise ValueError("theta has the wrong size")
        cost = C.c_double()
        g = H = None
        if derivs:
            g = np.empty(n)
            H = np.empty((self.C, 11, 11)) if mode == self.SQ_CAMONLY else np.empty((12, 12))
        self._check(self.lib.lcba_sq_normal(self.h, int(mode), _ptr(theta), C.byref(cost), _ptr(g), _ptr(H)))
        return cost.value, g, H

    def jacobian_blocks(self, x=None):
        x = None if x is None else _f64(x).ravel()
        Jc = np.empty((self.N, 2, 11))
        Jp = np.empty((self.N, 2, 3))
        self._check(self.lib.lcba_jacobian_blocks(self.h, _ptr(x), _ptr(Jc), _ptr(Jp)))
        return Jc, Jp

    def sparsity_indices(self, n_cameras, n_points, camera_ind, point_ind):
        ci, pi = _i64(camera_ind).ravel(), _i64(point_ind).ravel()
        out = np.empty(ci.size * 28, dtype=np.int32)
        self._check(self.lib.lcba_sparsity_indices(self.h, int(n_cameras), int(n_points), ci.size,
                                                   _ptr(ci), _ptr(pi), _ptr(out)))
        return out

    # ---- solver ----
    def solve(self, ftol=1e-8, xtol=1e-8, gtol=1e-8, max_nfev=0, verbose=0, profile=False,
              max_iterations=0, fix_cameras=False, shared_intrinsics=False, on_iteration=None):
        """on_iteration(row_dict): called from inside lcba_solve as each row of scipy's
        verbose=2 table becomes known (live printing)."""
        self.generation += 1
        opt = Options()
        self.lib.lcba_default_options(C.byref(opt))
        opt.ftol, opt.xtol, opt.gtol = ftol, xtol, gtol
        opt.max_nfev = int(max_nfev or 0)
        opt.verbose = int(verbose)
        opt.profile = 1 if profile else 0
        opt.max_iterations = int(max_iterations or 0)
        opt.fix_cameras = 1 if fix_cameras else 0
        opt.shared_intrinsics = 1 if shared_intrinsics else 0
        res = Result()
        cb = None
        if on_iteration is not None:
            cb = ITERATION_CB(lambda row, _user: on_iteration(_row_dict(row.contents)))
            self.lib.lcba_set_iteration_callback(self.h, cb, None)
        try:
            self._check(self.lib.lcba_solve(self.h, C.byref(opt), C.byref(res)))
        finally:
            if cb is not None:
                self.lib.lcba_set_iteration_callback(self.h, ITERATION_CB(), None)
        rows = (TraceRow * LCBA_MAX_TRACE)()
        n = self.lib.lcba_get_trace(self.h, rows, LCBA_MAX_TRACE)
        trace = [_row_dict(r) for r in rows[:max(n, 0)]]
        return res, trace

    def grad(self):
        g = np.empty(11 * self.C + 3 * self.P)
        self._check(self.lib.lcba_get_grad(self.h, _ptr(g)))
        return g

    def profile(self):
        stats = (KernelStat * 64)()
        n = C.c_int32()
        self._check(self.lib.lcba_get_profile(self.h, stats, 64, C.byref(n)))
        return {s.name.decode(): dict(launches=s.launches, total_ms=s.total_ms)
                for s in stats[:n.value]}

    def linearize(self, lam):
        n = 11 * self.C
        S = np.empty((n, n))
        rhs = np.empty(n)
        g = np.empty(n + 3 * self.P)
        sc = np.empty(n + 3 * self.P)
        cost = C.c_double()
        self._check(self.lib.lcba_linearize(self.h, float(lam), _ptr(S), _ptr(rhs), _ptr(g),
                                            _ptr(sc), C.byref(cost)))
        return dict(S=S, rhs=rhs, grad=g, scale_inv=sc, cost=cost.value)

    def covariance(self, points=True):
        """Unscaled covariance (J_f^T J_f)^-1 at the current x over the entries lcba_set_fixed leaves free
        (lcba_covariance; bounds ignored): (camera block (11 C, 11 C), this handle's point blocks (P, 6) as
        00 01 02 11 12 22 or None, cost, min_pivot).  Held entries are 0.  Raises LcbaError with code E_SINGULAR
        when the free parameters are not determined.  Collective on a point-sharded job."""
        n = 11 * self.C
        cam = np.empty((n, n))
        pt = np.empty((self.P, 6)) if points else None
        cost, piv = C.c_double(), C.c_double()
        self._check(self.lib.lcba_covariance(self.h, _ptr(cam), _ptr(pt), C.byref(cost), C.byref(piv)))
        return cam, pt, cost.value, piv.value

    def i8_fell_back(self):
        """1: the last Schur pass of the int8 path was recomputed on DMMA (rows finer than its digits resolve),
        0: the int8 result stood, -1: this handle does not use the int8 path."""
        return self.lib.lcba_debug_i8_fallback(self.h)

    I8_PLAN_CHOSEN, I8_PLAN_STRIP, I8_PLAN_COVER = 0, 1, 2

    @staticmethod
    def i8_plan(n_cams, P, sm_count, which=0):
        """A tile plan of the int8 tensor-core Schur kernel (lcba_debug_i8_cover_plan, host only): dict of
        tiles (n, 10) int32 [range 1 first row group, row groups, range 2 first row group, row groups, column
        block 1 first row group, row groups, block 2 first row group, row groups, first CTA, CTAs], work
        (CTAs, 3) [tile, kb0, kb1], nrg, nkb, cover (bool), executed_ops (int8 ops of one launch) and the
        cost model's slowest CTA in MMA-warp cycles: cycles (this plan), strip_cycles, cover_cycles."""
        lib = load()
        tiles = np.zeros((512, 10), dtype=np.int32)
        work = np.zeros((1024, 3), dtype=np.int32)
        nwork, nrg, nkb, cover = C.c_int32(), C.c_int32(), C.c_int64(), C.c_int32()
        model = np.zeros(4)
        nt = lib.lcba_debug_i8_cover_plan(int(n_cams), int(P), int(sm_count), int(which), _ptr(tiles), tiles.shape[0],
                                          _ptr(work), work.shape[0], C.byref(nwork), C.byref(nrg), C.byref(nkb),
                                          C.byref(cover), _ptr(model))
        if nt < 0:
            raise LcbaError(nt, "lcba_debug_i8_cover_plan: bad arguments")
        return dict(tiles=tiles[:nt].copy(), work=work[:nwork.value].copy(), nrg=nrg.value, nkb=nkb.value,
                    cover=bool(cover.value), executed_ops=model[0], cycles=model[1], strip_cycles=model[2],
                    cover_cycles=model[3])

    @staticmethod
    def i8_schedule(n_cams, P, sm_count, which=0, kmajor=True):
        """The K blocks every CTA of a tile plan of the int8 Schur kernel reads (lcba_debug_i8_schedule, host
        only): dict of work (CTAs, 6) int32 [tile, kb0, kb1, kfirst, kc, kstride] -- the K blocks
        kfirst + (i // kc) kstride + i % kc for i < kb1 - kb0 -- and window (K blocks a CTA may run ahead of
        the slowest one; 0 without a window).  kmajor=False: one contiguous range per CTA (LCBA_I8_SCHED=range)."""
        lib = load()
        work = np.zeros((1024, 6), dtype=np.int32)
        window = C.c_int32()
        n = lib.lcba_debug_i8_schedule(int(n_cams), int(P), int(sm_count), int(which), int(bool(kmajor)), _ptr(work),
                                       work.shape[0], C.byref(window))
        if n < 0:
            raise LcbaError(n, "lcba_debug_i8_schedule: bad arguments")
        return dict(work=work[:n].copy(), window=window.value)

    def debug_chol(self, A, rhs, mu=0.0, d=None, grid=0):
        """The solver's dense camera solve on a host system (lcba_debug_chol): returns (x, factor, fail)
        with factor the (n+1, n) work buffer (strict lower L, 1 / l_jj on the diagonal, row n = L^-1 rhs)."""
        A = _f64(A)
        n = A.shape[0]
        if A.shape != (n, n):
            raise ValueError("A must be square")
        rhs = _f64(rhs).ravel()
        d = None if d is None else _f64(d).ravel()
        if rhs.size != n or (d is not None and d.size != n):
            raise ValueError("rhs and d must have n entries")
        x = np.empty(n)
        factor = np.empty((n + 1, n))
        fail = C.c_int32()
        self._check(self.lib.lcba_debug_chol(self.h, n, _ptr(A), _ptr(rhs), float(mu), _ptr(d), int(grid),
                                             _ptr(x), _ptr(factor), C.byref(fail)))
        return x, factor, fail.value

    STEP_FULL, STEP_FIX_CAMERAS, STEP_SHARED_INTRINSICS = 0, 1, 2

    def debug_step(self, lam, mu=0.0, mode=0):
        """One Gauss-Newton step of the solver's passes at the current x (lcba_debug_step), damped with
        lam: (camera step 11 C, point step 3 P, dict of the STEP_SCALARS)."""
        pc = np.empty(11 * self.C)
        pp = np.empty(3 * self.P)
        sc = np.empty(len(STEP_SCALARS))
        self._check(self.lib.lcba_debug_step(self.h, float(lam), float(mu), int(mode), _ptr(pc), _ptr(pp), _ptr(sc)))
        return pc, pp, dict(zip(STEP_SCALARS, sc.tolist()))

    def debug_i8_make(self, lam, ref=False, reps=1, planes=True, poison=0xA5):
        """The digit planes of the int8 Schur path at the current x, damped with lam (lcba_debug_i8_make):
        (ms per launch of k_i8_make, or of the reference k_i8_make_ref with ref=True, planes as a uint8 array or
        None).  The plane buffer is filled with the byte `poison` first (None: left as it is).  The problem must
        take the int8 path (LCBA_SCHUR_I8=1 when it is set, below 32 768 points)."""
        ms = C.c_double()
        buf, nbytes = None, 0
        if planes:
            nbytes = i8_plane_bytes(self.C, self.P)
            buf = np.empty(nbytes, dtype=np.uint8)
        self._check(self.lib.lcba_debug_i8_make(self.h, float(lam), int(bool(ref)), int(reps),
                                                -1 if poison is None else int(poison), C.byref(ms), _ptr(buf), nbytes))
        return ms.value, buf

    def time_device(self, what, reps=10):
        ms = C.c_double()
        self._check(self.lib.lcba_time_device(self.h, int(what), int(reps), C.byref(ms)))
        return ms.value

    # ---- multi-GPU ----
    @staticmethod
    def nccl_unique_id():
        lib = load()
        buf = C.create_string_buffer(128)
        rc = lib.lcba_nccl_unique_id(buf)
        if rc != 0:
            raise LcbaError(rc, lib.lcba_last_error(None).decode())
        return buf.raw

    def comm_init(self, rank, nranks, unique_id=None):
        """unique_id bytes: create the process-wide communicator; None: attach the existing one."""
        buf = None if unique_id is None else C.create_string_buffer(bytes(unique_id), 128)
        self._check(self.lib.lcba_comm_init(self.h, int(rank), int(nranks), buf))


def debug_tr2d(B00, B01, B11, g0, g1, Delta):
    lib = load()
    p = (C.c_double * 2)()
    newton = C.c_int()
    lib.lcba_debug_tr2d(B00, B01, B11, g0, g1, Delta, p, C.byref(newton))
    return np.array([p[0], p[1]]), bool(newton.value)
