"""Drop-in ``PySBA`` for the bundle-adjustment step of laserCalib, running on a B200.

Mirrors the surface of the reference ``lasercalib/pySBA.py`` (class ``PySBA``: constructor
``:28``, ``rotate`` ``:61``, ``project`` ``:76``, ``fun`` ``:92``,
``bundle_adjustment_sparsity`` ``:103``, ``optimizedParams`` ``:121``, ``bundleAdjust``
``:132``) with the same names, argument meaning and error behaviour, so that
``scripts/calibrate_camera.py:62,71`` and ``lasercalib/sba_print.py:13-17`` work unchanged
after ``from lasercalib_b200.pySBA import PySBA``.

Every numerical method calls the C-ABI of ``liblcba.so`` (include/lcba.h) through ctypes;
there is no numpy/scipy compute path here and no CPU fallback: without the CUDA library or
a GPU the calls raise.
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import OptimizeResult
from scipy.sparse import csr_matrix

from . import _cabi
from . import dist as _dist

N_CAM_PARAMS = 11

# scipy/optimize/_lsq/least_squares.py:23-31
TERMINATION_MESSAGES = {
    -1: "Improper input parameters status returned from `leastsq`",
    0: "The maximum number of function evaluations is exceeded.",
    1: "`gtol` termination condition is satisfied.",
    2: "`ftol` termination condition is satisfied.",
    3: "`xtol` termination condition is satisfied.",
    4: "Both `ftol` and `xtol` termination conditions are satisfied.",
}


_ENGINES = {}      # device -> shared _cabi.Engine


class BAResult(OptimizeResult):
    """OptimizeResult whose large members (``fun``, ``jac``) are produced on first access
    (the reference materialises a 2N x n CSR Jacobian: ~4 KB per observation)."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        object.__setattr__(self, "_lazy", {})

    def set_lazy(self, key, fn):
        self._lazy[key] = fn

    def __contains__(self, key):
        return dict.__contains__(self, key) or key in object.__getattribute__(self, "_lazy")

    def keys(self):
        return list(dict.keys(self)) + [k for k in self._lazy if not dict.__contains__(self, k)]

    def __dir__(self):
        return self.keys()

    def __missing__(self, key):
        lazy = object.__getattribute__(self, "_lazy")
        if key in lazy:
            self[key] = lazy.pop(key)()
            return dict.__getitem__(self, key)
        raise KeyError(key)

    def __getattr__(self, name):
        try:
            return self[name]
        except KeyError as e:
            raise AttributeError(name) from e

    def __reduce__(self):
        for k in list(self._lazy):
            self[k]
        return (OptimizeResult, (dict(self),))


def normalize_fixed(fixed_camera_params, fixed_points, n_cameras, n_points):
    """The masks of ``bundleAdjust(fixed_camera_params=..., fixed_points=...)`` as (C, 11) and (P,)
    bool arrays, or None where nothing is held.

    fixed_camera_params: bool array of shape (11,) (the same entries of every camera) or (C, 11).
    fixed_points: bool array of shape (P,) or an integer array of point indices in [0, P).
    Raises ValueError on any other shape, dtype or index."""
    cam = pt = None
    if fixed_camera_params is not None:
        m = np.asarray(fixed_camera_params)
        if m.dtype != np.bool_:
            raise ValueError("fixed_camera_params must be a bool array, got dtype %s" % m.dtype)
        if m.shape == (N_CAM_PARAMS,):
            m = np.broadcast_to(m, (n_cameras, N_CAM_PARAMS))
        elif m.shape != (n_cameras, N_CAM_PARAMS):
            raise ValueError("fixed_camera_params must have shape (11,) or (%d, 11), got %s"
                             % (n_cameras, m.shape))
        if m.any():
            cam = np.ascontiguousarray(m)
    if fixed_points is not None:
        m = np.asarray(fixed_points)
        if m.dtype == np.bool_:
            if m.shape != (n_points,):
                raise ValueError("a bool fixed_points must have shape (%d,), got %s" % (n_points, m.shape))
        elif m.dtype.kind in "iu":
            if m.ndim != 1:
                raise ValueError("fixed_points indices must be a 1-D array, got shape %s" % (m.shape,))
            if m.size and (m.min() < 0 or m.max() >= n_points):
                raise ValueError("fixed_points indices must lie in [0, %d)" % n_points)
            idx = m
            m = np.zeros(n_points, dtype=bool)
            m[idx] = True
        else:
            raise ValueError("fixed_points must be a bool mask or an integer index array, got dtype %s" % m.dtype)
        if m.any():
            pt = np.ascontiguousarray(m)
    return cam, pt


def normalize_bounds(bounds, x0, held=None):
    """``bounds`` of ``bundleAdjust`` as ``least_squares`` takes it (a 2-tuple of scalars or arrays, or
    ``scipy.optimize.Bounds``) -> (lb, ub) float arrays of x0's shape, or None when every bound of a free entry is
    infinite (the unbounded loop runs, as scipy dispatches to trf_no_bounds).  ``held``: bool mask of the held
    entries of x0, which are not checked.  Raises ValueError with least_squares' messages
    (scipy/optimize/_lsq/least_squares.py:883-901)."""
    from scipy.optimize import Bounds
    from scipy.optimize._lsq.least_squares import prepare_bounds
    if bounds is None:
        return None
    if isinstance(bounds, Bounds):
        lb, ub = prepare_bounds((bounds.lb, bounds.ub), x0.shape[0])
    elif len(bounds) == 2:
        lb, ub = prepare_bounds(bounds, x0.shape[0])
    else:
        raise ValueError("`bounds` must contain 2 elements.")
    if lb.shape != x0.shape or ub.shape != x0.shape:
        raise ValueError("Inconsistent shapes between bounds and `x0`.")
    free = np.ones(x0.shape, dtype=bool) if held is None else ~held
    lf, uf, xf = lb[free], ub[free], x0[free]
    if np.any(lf >= uf):
        raise ValueError("Each lower bound must be strictly less than each upper bound.")
    if not np.all((xf >= lf) & (xf <= uf)):
        raise ValueError("Initial guess is outside of provided bounds")
    if np.all(np.isneginf(lf)) and np.all(np.isposinf(uf)):
        return None
    return lb, ub


def covariance_result(cam_cov, pt6, cost, min_pivot, m, cam_fixed=None, pt_fixed=None, absolute_sigma=False):
    """``PySBA.covariance``'s result from lcba_covariance's unscaled blocks: cam_cov (11 C, 11 C), pt6 (P, 6) as
    00 01 02 11 12 22, cost = 0.5 |f|^2, m residuals, the held masks of ``normalize_fixed`` (or None).  Applies
    curve_fit's ``s^2 = 2 cost / (m - n_free)`` unless ``absolute_sigma``; ``dof <= 0`` fills the free entries with
    inf and warns (scipy/optimize/_minpack_py.py, curve_fit)."""
    n_cam = cam_cov.shape[0]
    P = pt6.shape[0]
    cam_free = np.ones(n_cam, dtype=bool) if cam_fixed is None else ~np.asarray(cam_fixed).ravel()
    pt_free = np.ones(P, dtype=bool) if pt_fixed is None else ~np.asarray(pt_fixed)
    n_free = int(cam_free.sum()) + 3 * int(pt_free.sum())
    dof = int(m) - n_free
    iu = np.array([[0, 1, 2], [1, 3, 4], [2, 4, 5]])
    point_cov = np.asarray(pt6)[:, iu]
    camera_cov = np.array(cam_cov, dtype=np.float64)
    sigma2 = 1.0
    if not absolute_sigma:
        if dof > 0:
            sigma2 = 2.0 * cost / dof
            camera_cov *= sigma2
            point_cov *= sigma2
        else:
            import warnings
            from scipy.optimize import OptimizeWarning
            sigma2 = np.inf
            camera_cov[np.ix_(cam_free, cam_free)] = np.inf
            point_cov[pt_free] = np.inf
            warnings.warn("Covariance of the parameters could not be estimated", category=OptimizeWarning,
                          stacklevel=3)
    return OptimizeResult(camera_cov=camera_cov,
                          camera_std=np.sqrt(np.diag(camera_cov)).reshape(-1, N_CAM_PARAMS),
                          point_cov=point_cov, point_std=np.sqrt(np.einsum("paa->pa", point_cov)),
                          sigma2=sigma2, dof=dof, cost=cost, min_pivot=min_pivot)


def _print_header():
    # scipy/optimize/_lsq/common.py:545-548
    print("{:^15}{:^15}{:^15}{:^15}{:^15}{:^15}".format(
        "Iteration", "Total nfev", "Cost", "Cost reduction", "Step norm", "Optimality"))


def _print_row(r):
    # scipy/optimize/_lsq/common.py:551-563
    cr = " " * 15 if np.isnan(r["cost_reduction"]) else f"{r['cost_reduction']:^15.2e}"
    sn = " " * 15 if np.isnan(r["step_norm"]) else f"{r['step_norm']:^15.2e}"
    print(f"{r['iteration']:^15}{r['nfev']:^15}{r['cost']:^15.4e}{cr}{sn}{r['optimality']:^15.2e}")


class PySBA:
    """Python class for Simple Bundle Adjustment (B200 engine behind the reference API)."""

    def __init__(self, cameraArray, points3D, points2D, cameraIndices, point2DIndices,
                 points3Dfixed=None, pointWeights=None):
        # attributes and defaults exactly as the reference keeps them (pySBA.py:50-59)
        self.cameraArray = cameraArray
        self.points3D = points3D
        self.points2D = points2D
        self.cameraIndices = cameraIndices
        self.point2DIndices = point2DIndices
        self.points3Dfixed = points3Dfixed
        # The reference materialises np.full_like(point2DIndices, 1).reshape(-1, 1) here
        # (pySBA.py:56-58); the same array appears on first access of `.pointWeights`, but the
        # solver path never pays for 8 bytes per observation of ones.
        self._default_weights = pointWeights is None
        self._pointWeights = None if pointWeights is None else pointWeights.reshape((-1, 1))
        self.points3Dfixed_labeled = None
        self._engine = None
        self._problem_key = None
        self._owner_token = None
        self._fresh_problem = True
        self.last_trace = None
        self.last_timing = None
        # engine knob (not in the reference): True = the observation arrays are promised not to
        # change, so their device copy is reused between calls; default = re-read every call
        self.observations_static = False

    @property
    def pointWeights(self):
        if self._pointWeights is None:
            self._pointWeights = np.full_like(self.point2DIndices, 1).reshape((-1, 1))
        return self._pointWeights

    @pointWeights.setter
    def pointWeights(self, value):
        self._default_weights = False
        self._pointWeights = value

    # ---- pickling: device handles never enter the pickle (calibrate_camera.py:86-88) ----
    def __getstate__(self):
        d = dict(self.__dict__)
        d["_engine"] = None
        d["_problem_key"] = None
        d["_owner_token"] = None
        d.pop("_keep", None)
        d.pop("_shard", None)
        return d

    def __setstate__(self, d):
        self.__dict__.update(d)

    # ---- engine plumbing ----
    def _get_engine(self):
        """One engine (GPU handle, stream, NCCL attachment) per device and process, shared by
        all PySBA objects; `_owner` tells whose observation set is resident."""
        if self._engine is None:
            rank, ws, local = _dist.world()
            dev = local if ws > 1 else -1
            eng = _ENGINES.get(dev)
            if eng is None or eng.h is None:
                eng = _cabi.Engine(dev)
                eng._comm_ready = False
                eng._owner = None
                eng._owner_token = None
                _ENGINES[dev] = eng
            self._engine = eng
        return self._engine

    def _weights_arg(self, pointWeights):
        if pointWeights is None or (self._default_weights and pointWeights is self._pointWeights):
            return None
        w = np.asarray(pointWeights).reshape(-1)
        if w.dtype.kind in "iu" and np.all(w == 1):
            return None
        return np.ascontiguousarray(w, dtype=np.float64)

    def invalidate(self):
        """Forget the device-resident copy of the observation arrays (only meaningful with
        ``observations_static = True``): the next call uploads them again."""
        self._problem_key = None

    def _ensure_problem(self, cams, pts, camera_indices, point_indices, points_2d, pointWeights):
        """Load the observation set on the device.

        Like the reference, every call reads the caller's arrays again (an in-place edit of
        ``points2D`` / ``pointWeights`` / the index arrays between two calls is honoured).
        Set ``sba.observations_static = True`` to promise that those arrays do not change
        while this object lives: the device copy is then reused as long as the same array
        objects are passed (`invalidate()` drops it)."""
        eng = self._get_engine()
        w = self._weights_arg(pointWeights)
        ci = np.asarray(camera_indices)
        pi = np.asarray(point_indices)
        p2 = np.asarray(points_2d)
        key = (cams.shape[0], pts.shape[0], ci.ctypes.data, ci.size, pi.ctypes.data,
               p2.ctypes.data, None if w is None else (w.ctypes.data, w.size))
        reuse = (self.observations_static and key == self._problem_key and eng._owner is self
                 and eng._owner_token == self._owner_token)
        self._fresh_problem = not reuse
        if self._fresh_problem:
            eng.set_problem(cams, pts, p2, ci, pi, w)
            eng._owner = self
            self._owner_token = eng._owner_token = object()
            self._problem_key = key
            self._keep = (ci, pi, p2, w, pointWeights)   # keep the keyed buffers alive
        return eng

    def _ensure_shard(self, cams0, pts0, rank, ws):
        """Point-sharded counterpart of _ensure_problem (collective): one process per GPU, this rank keeps a
        contiguous range of points and their observations; cameras are replicated; the library all-reduces with
        NCCL.  x is (cams0, this rank's rows of pts0).  Returns (engine, shard)."""
        w = self._weights_arg(self._pointWeights)
        eng = self._get_engine()
        key = ("shard", ws, cams0.shape[0], pts0.shape[0], id(self.points2D),
               id(self.cameraIndices), id(self.point2DIndices), None if w is None else id(self._pointWeights))
        reuse = (self.observations_static and key == self._problem_key and eng._owner is self
                 and eng._owner_token == self._owner_token)
        if reuse:
            shard = self._shard
            eng.set_params(cams0, shard["pts0_of"](pts0))
        else:
            shard = _dist.shard_problem(pts0, self.points2D, self.cameraIndices,
                                        self.point2DIndices, w, rank, ws, collective=True)
            lo, hi = shard["lo"], shard["hi"]
            shard["pts0_of"] = lambda p, lo=lo, hi=hi: np.ascontiguousarray(p[lo:hi])
            eng.set_problem(cams0, shard["pts"], shard["points_2d"], shard["camera_ind"],
                            shard["point_ind"], shard["weights"], pt_offset=shard["pt_offset"])
            self._problem_key = key
            self._shard = shard
            eng._owner = self
            self._owner_token = eng._owner_token = object()
        if not eng._comm_ready:
            _dist.connect_engine(eng)
            eng._comm_ready = True
        return eng, shard

    # ---- model (pySBA.py:61-89) ----
    def rotate(self, points, rot_vecs):
        """Rotate points by given rotation vectors (Rodrigues), row by row."""
        return self._get_engine().rotate(np.asarray(points, dtype=np.float64),
                                         np.asarray(rot_vecs, dtype=np.float64))

    def project(self, points, cameraArray):
        """Convert 3-D points to 2-D by projecting onto images (per-row camera vector)."""
        return self._get_engine().project(np.asarray(points, dtype=np.float64),
                                          np.asarray(cameraArray, dtype=np.float64))

    def fun(self, params, n_cameras, n_points, camera_indices, point_indices, points_2d,
            pointWeights):
        """Compute residuals; ``params`` = camera parameters then 3-D coordinates
        (pySBA.py:92-101).  Interleaved [u0, v0, u1, v1, ...] in the caller's order."""
        params = np.ascontiguousarray(params, dtype=np.float64)
        nc = n_cameras * N_CAM_PARAMS
        cams = params[:nc].reshape((n_cameras, N_CAM_PARAMS))
        pts = params[nc:].reshape((n_points, 3))
        eng = self._ensure_problem(cams, pts, camera_indices, point_indices, points_2d,
                                   pointWeights)
        r, _ = eng.residuals(params)
        return r

    def bundle_adjustment_sparsity(self, numCameras, numPoints, cameraIndices, pointIndices):
        """0/1 pattern (2N, 11C+3P), 28 non-zeros per observation (pySBA.py:103-118);
        returned as CSR (the reference fills a lil_matrix with the same pattern)."""
        cameraIndices = np.asarray(cameraIndices)
        m = cameraIndices.size * 2
        n = numCameras * N_CAM_PARAMS + numPoints * 3
        idx = self._get_engine().sparsity_indices(numCameras, numPoints, cameraIndices,
                                                  pointIndices)
        indptr = np.arange(0, 14 * (m + 1), 14, dtype=np.int64 if idx.size >= 2**31 else np.int32)
        return csr_matrix((np.ones(idx.size, dtype=int), idx, indptr), shape=(m, n))

    def optimizedParams(self, params, n_cameras, n_points):
        """Retrieve camera parameters and 3-D coordinates (views of ``params``)."""
        nc = n_cameras * N_CAM_PARAMS
        return params[:nc].reshape((n_cameras, N_CAM_PARAMS)), params[nc:].reshape((n_points, 3))

    # ---- solver (pySBA.py:132-147) ----
    def bundleAdjust(self, ftol=1e-4, xtol=1e-8, gtol=1e-8, max_nfev=None, verbose=2,
                     profile=False, max_iterations=0, _fix_cameras=False, _shared=False,
                     fixed_camera_params=None, fixed_points=None, bounds=None):
        """Returns the bundle adjusted parameters (scipy ``OptimizeResult`` layout) and
        stores them on ``self.cameraArray`` / ``self.points3D``.

        The keyword defaults reproduce the reference call
        ``least_squares(fun, x0, jac_sparsity=A, verbose=2, x_scale='jac', ftol=ftol,
        method='trf', jac='3-point')``.

        ``fixed_camera_params`` (bool, shape (11,) for every camera or (C, 11)) and
        ``fixed_points`` (bool, shape (P,), or integer point indices) hold those parameters at
        their input values: the solve is scipy's ``trf_no_bounds`` on the free sub-vector (scaling,
        trust radius, ``|x|`` and ``|g|_inf`` over free entries, ``max_nfev`` = 100 * free count).
        ``x`` and ``jac`` keep the full layout, held entries of ``x`` equal the input bit for bit,
        ``grad`` is 0 there.  Holding camera 0's extrinsics and three non-collinear points (or one
        scale coordinate) removes the 7-dimensional gauge freedom.

        ``bounds`` (what ``least_squares`` takes: a 2-tuple of scalars or (n,) arrays over the layout
        ``[cameraArray.ravel(), points3D.ravel()]``, or ``scipy.optimize.Bounds``) keeps x in the box: the solve is
        scipy's ``trf_bounds`` (reflective TRF) with the exact Schur solve in place of LSMR; x0 is first moved strictly
        inside as least_squares does.  ``optimality`` is then ``|g v|_inf`` (v: the Coleman-Li vector) and
        ``active_mask`` marks the entries on a bound.  Held entries ignore their bounds.  Every bound infinite:
        the unbounded solve, unchanged."""
        numCameras = self.cameraArray.shape[0]
        numPoints = self.points3D.shape[0]
        cam_fixed, pt_fixed = normalize_fixed(fixed_camera_params, fixed_points, numCameras, numPoints)
        cams0 = np.ascontiguousarray(self.cameraArray, dtype=np.float64)
        pts0 = np.ascontiguousarray(self.points3D, dtype=np.float64)
        nc = numCameras * N_CAM_PARAMS
        held = None
        if cam_fixed is not None or pt_fixed is not None:
            held = np.zeros(nc + 3 * numPoints, dtype=bool)
            if cam_fixed is not None and not _fix_cameras:
                held[:nc] = cam_fixed.ravel()
            if pt_fixed is not None:
                held[nc:] = np.repeat(pt_fixed, 3)
        box = normalize_bounds(bounds, np.hstack((cams0.ravel(), pts0.ravel())), held)
        if _shared:
            # x0 of the reference: the mean (f, k1, k2) for every camera (pySBA.py:300)
            cams0 = cams0.copy()
            cams0[:, 6:9] = np.mean(cams0[:, 6:9], axis=0)
        import time as _time
        t_in0 = _time.perf_counter()
        rank, ws, _ = _dist.world()
        shard = None
        if ws > 1:
            eng, shard = self._ensure_shard(cams0, pts0, rank, ws)
            if verbose and rank != 0:
                verbose = 0
            pt_fixed_local = None if pt_fixed is None else pt_fixed[shard["lo"]:shard["hi"]]
        else:
            eng = self._ensure_problem(cams0, pts0, self.cameraIndices, self.point2DIndices,
                                       self.points2D, self._pointWeights)
            if not self._fresh_problem or _shared:   # observations already resident: new x0 only
                eng.set_params(cams0, pts0)
            pt_fixed_local = pt_fixed
        if cam_fixed is not None or pt_fixed_local is not None or eng.has_fixed:
            eng.set_fixed(cam_fixed, pt_fixed_local)
        if box is not None:
            lo, hi = (0, numPoints) if shard is None else (shard["lo"], shard["hi"])
            eng.set_bounds(box[0][:nc], box[1][:nc], box[0][nc:].reshape(-1, 3)[lo:hi],
                           box[1][nc:].reshape(-1, 3)[lo:hi])
        elif eng.has_bounds:
            eng.set_bounds()
        t_in1 = _time.perf_counter()
        live = None
        if verbose == 2:
            # scipy prints the table while it iterates (least_squares(verbose=2), pySBA.py:141)
            _print_header()
            live = _print_row
        try:
            res, trace = eng.solve(ftol=ftol, xtol=xtol, gtol=gtol, max_nfev=max_nfev or 0,
                                   verbose=verbose, profile=profile,
                                   max_iterations=max_iterations, fix_cameras=_fix_cameras,
                                   shared_intrinsics=_shared, on_iteration=live)
        except _cabi.LcbaError as e:
            if e.code == -5:
                raise ValueError("Residuals are not finite in the initial point.") from e
            raise
        self.last_trace = trace
        t_sol = _time.perf_counter()
        x_direct = None
        if not _fix_cameras and not _shared:
            # the reference's x = [cameras | points]: filled in place, the arrays are views
            x_direct = np.empty(nc + numPoints * 3)
        if shard is None:
            cams, pts = eng.get_params(x_direct)
        else:
            cams, pts = eng.get_params()
            if x_direct is not None:
                x_direct[:nc] = cams.ravel()
                cams = x_direct[:nc].reshape(numCameras, N_CAM_PARAMS)
                pts = _dist.allgather_rows(pts, shard["bounds"], out=x_direct[nc:].reshape(numPoints, 3))
            else:
                pts = _dist.allgather_rows(pts, shard["bounds"])
        # ---- lazy members: the engine is shared (one handle per device), so by the time
        # `res.fun` / `res.grad` / `res.jac` are read it may hold another problem or another x.
        # The readers check the handle's generation counter and, if it moved, put this result's
        # observation set and final x back before evaluating.  On a point-sharded run the
        # residual read is local to the rank (no collective), and a stale handle raises: the
        # other ranks could not follow a re-upload.
        gen, token = eng.generation, self._owner_token
        kept = getattr(self, "_keep", None)
        cams_f, pts_f = cams, pts

        def engine_at_result():
            if eng.h is not None and eng.generation == gen and eng._owner_token is token:
                return eng
            if shard is not None:
                raise RuntimeError("the engine was used again before this member of a point-sharded "
                                   "result was read; read res.fun right after bundleAdjust")
            ci_k, pi_k, p2_k, w_k, _ = kept
            e = self._get_engine()
            e.set_problem(np.ascontiguousarray(cams_f), np.ascontiguousarray(pts_f), p2_k, ci_k, pi_k, w_k)
            e._owner, e._owner_token = None, None
            self._problem_key = None
            return e

        def lazy_fun():
            return engine_at_result().residuals(None, want_cost=False)[0]

        def lazy_grad():
            e = engine_at_result()
            g = e.grad() if e.generation == gen else e.linearize(1.0)["grad"]
            if held is not None:       # the unmasked tap on a re-uploaded problem: held entries -> 0
                g[held] = 0.0
            return g

        # wall-clock split of this call: ingest (H2D + validate/sort/narrow/CSR + plans), solve, results D2H
        self.last_timing = dict(ingest_ms=(t_in1 - t_in0) * 1e3, solve_wall_ms=(t_sol - t_in1) * 1e3,
                                solve_device_ms=float(res.solve_ms), d2h_ms=(_time.perf_counter() - t_sol) * 1e3)
        if _fix_cameras:
            return self._finish_nocam(lazy_fun, lazy_grad, res, pts, shard, verbose)
        if _shared:
            # the reference's parameter order: [f k1 k2 | extrinsics | centroids | points]
            x = np.hstack((cams[0, 6:9], cams[:, :6].ravel(), cams[:, 9:].ravel(), pts.ravel()))
            out = BAResult(x=x, cost=res.cost, optimality=res.optimality,
                           active_mask=np.zeros_like(x), nfev=int(res.nfev), njev=int(res.njev),
                           status=int(res.status))
            out["message"] = TERMINATION_MESSAGES[int(res.status)]
            out["success"] = int(res.status) > 0
            out["solve_ms"] = res.solve_ms
            out["nit"] = int(res.iterations)
            out.set_lazy("fun", lazy_fun)
            if verbose >= 1:
                print(out["message"])
            self.cameraArray = cams
            self.points3D = pts
            return out
        x = x_direct if x_direct is not None else np.hstack((cams.ravel(), pts.ravel()))
        out = BAResult(x=x, cost=res.cost, optimality=res.optimality,
                       nfev=int(res.nfev), njev=int(res.njev), status=int(res.status))
        if box is None:
            out.set_lazy("active_mask", lambda: np.zeros_like(x))
        else:
            from scipy.optimize._lsq.common import find_active_constraints
            active = find_active_constraints(x, box[0], box[1], rtol=xtol)
            if held is not None:
                active[held] = 0
            out["active_mask"] = active
        out["message"] = TERMINATION_MESSAGES[int(res.status)]
        out["success"] = int(res.status) > 0
        out["solve_ms"] = res.solve_ms
        out["nit"] = int(res.iterations)
        out["gpu_launches"] = int(res.gpu_launches)
        ci, pi = np.asarray(self.cameraIndices), np.asarray(self.point2DIndices)
        if shard is not None:
            # sharded run: `fun` / `grad` / `jac` are this rank's shard (observations
            # `fun_obs_index` of the caller's arrays); x, cost, optimality are global
            out["fun_obs_index"] = shard["obs_sel"]
            out.set_lazy("fun", lazy_fun)
            if verbose >= 1:
                print(out["message"])
            camera_params, points_3d = self.optimizedParams(x, numCameras, numPoints)
            self.cameraArray = camera_params
            self.points3D = points_3d
            return out
        out.set_lazy("grad", lazy_grad)
        out.set_lazy("fun", lazy_fun)

        def _jac():
            Jc, Jp = engine_at_result().jacobian_blocks(None)
            A = self.bundle_adjustment_sparsity(numCameras, numPoints, ci, pi)
            return csr_matrix((np.concatenate([Jc, Jp], axis=2).ravel(), A.indices, A.indptr),
                              shape=A.shape)

        out.set_lazy("jac", _jac)
        if verbose >= 1:
            # scipy/optimize/_lsq/least_squares.py:1038-1043
            print(out["message"])
            print("Function evaluations {}, initial cost {:.4e}, final cost {:.4e}, "
                  "first-order optimality {:.2e}.".format(out["nfev"], res.initial_cost,
                                                          res.cost, res.optimality))
        camera_params, points_3d = self.optimizedParams(x, numCameras, numPoints)
        self.cameraArray = camera_params
        self.points3D = points_3d
        return out

    # ---- uncertainty of the solution ----
    def covariance(self, fixed_camera_params=None, fixed_points=None, absolute_sigma=False):
        """Covariance of the least-squares estimate at ``cameraArray`` / ``points3D`` (after ``bundleAdjust``: the
        solution), as ``scipy.optimize.curve_fit`` returns ``pcov``: ``s^2 (J_f^T J_f)^-1`` over the free
        parameters, ``J_f`` the Jacobian of ``fun`` (weights included) over the entries that
        ``fixed_camera_params`` / ``fixed_points`` (as in ``bundleAdjust``) leave free and
        ``s^2 = 2 cost / (m - n_free)``, m = 2 N residuals.  ``absolute_sigma=True``: no ``s^2`` (the weights are
        1 / sigma of the pixel noise).  Bounds are ignored, as curve_fit ignores them.

        Returns an ``OptimizeResult`` with ``camera_cov`` (11 C, 11 C), ``camera_std`` (C, 11), ``point_cov``
        (P, 3, 3) (the 3 x 3 diagonal blocks; no camera-point or point-point cross terms), ``point_std`` (P, 3),
        ``sigma2``, ``dof``, ``cost`` and ``min_pivot`` (the smallest Jacobi-relative pivot ``l_jj^2 / S_jj`` of the
        reduced camera system).  Held entries are 0.  With ``dof <= 0`` and ``absolute_sigma=False`` the free
        entries are ``inf`` and an ``OptimizeWarning`` is issued, as curve_fit does.

        The covariance depends on the gauge: the 7 free modes of the problem (rotation, translation, scale) have
        to be held, e.g. camera 0's extrinsics and three non-collinear points; the result describes the other
        parameters relative to what is held.  Raises ``numpy.linalg.LinAlgError`` when the free parameters are
        not determined (gauge not fixed, an unheld point seen by fewer than two cameras, an unconstrained camera
        entry), ``ValueError`` on malformed masks.  Holding every camera gives the points-only covariance."""
        numCameras = self.cameraArray.shape[0]
        numPoints = self.points3D.shape[0]
        cam_fixed, pt_fixed = normalize_fixed(fixed_camera_params, fixed_points, numCameras, numPoints)
        cams0 = np.ascontiguousarray(self.cameraArray, dtype=np.float64)
        pts0 = np.ascontiguousarray(self.points3D, dtype=np.float64)
        rank, ws, _ = _dist.world()
        shard = None
        if ws > 1:
            eng, shard = self._ensure_shard(cams0, pts0, rank, ws)
            pt_fixed_local = None if pt_fixed is None else pt_fixed[shard["lo"]:shard["hi"]]
        else:
            eng = self._ensure_problem(cams0, pts0, self.cameraIndices, self.point2DIndices,
                                       self.points2D, self._pointWeights)
            if not self._fresh_problem:
                eng.set_params(cams0, pts0)
            pt_fixed_local = pt_fixed
        if cam_fixed is not None or pt_fixed_local is not None or eng.has_fixed:
            eng.set_fixed(cam_fixed, pt_fixed_local)
        try:
            cam_cov, pt6, cost, min_pivot = eng.covariance()
        except _cabi.LcbaError as e:
            if e.code == _cabi.E_SINGULAR:
                raise np.linalg.LinAlgError(str(e)) from e
            raise
        if shard is not None:
            pt6 = _dist.allgather_rows(pt6, shard["bounds"])
        m = 2 * np.asarray(self.cameraIndices).size
        return covariance_result(cam_cov, pt6, cost, min_pivot, m, cam_fixed, pt_fixed, absolute_sigma)

    # ---- variants of the reference that are not on the production path (SURVEY 8f) ----
    # ---- the two dense squared-residual variants (pySBA.py:151-206) ----
    def _dense_variant(self, mode, x0, ftol, verbose):
        """scipy's dense trf loop (tr_solver='exact', x_scale=1) with cost / J^T f / J^T J
        evaluated on the GPU in one pass per call; only n x n arithmetic runs here."""
        from ._trf_dense import trf_dense
        cams = np.ascontiguousarray(self.cameraArray, dtype=np.float64)
        pts = np.ascontiguousarray(self.points3D, dtype=np.float64)
        eng = self._ensure_problem(cams, pts, self.cameraIndices, self.point2DIndices,
                                   self.points2D, self.pointWeights)
        eng.set_params(cams, pts)
        C = cams.shape[0]
        launches0 = [0]

        def evaluate(x, derivs):
            cost, g, H = eng.sq_normal(mode, x, derivs)
            launches0[0] += 3
            if derivs and mode == eng.SQ_CAMONLY:
                D = np.zeros((C * N_CAM_PARAMS, C * N_CAM_PARAMS))
                for c in range(C):
                    a = c * N_CAM_PARAMS
                    D[a:a + N_CAM_PARAMS, a:a + N_CAM_PARAMS] = H[c]
                H = D
            return cost, g, H

        m = 2 * np.asarray(self.cameraIndices).size
        r = trf_dense(evaluate, x0, m, ftol, verbose=verbose,
                      block=N_CAM_PARAMS if mode == eng.SQ_CAMONLY else None)
        out = BAResult(x=r.x, cost=r.cost, grad=r.grad, optimality=r.optimality,
                       active_mask=r.active_mask, nfev=r.nfev, njev=r.njev, status=r.status,
                       message=r.message, success=r.success)
        out["gpu_launches"] = launches0[0]
        return out

    def _squared_fun(self, cams, pts):
        w = np.asarray(self.pointWeights, dtype=np.float64).reshape(-1, 1)
        e = self.project(pts[self.point2DIndices], cams[self.cameraIndices]) - self.points2D
        return (w * e ** 2).ravel()

    def bundle_adjustment_camonly(self, ftol=1e-4, verbose=2):
        """Optimise the cameras with the 3-D points fixed (pySBA.py:158-173).  As in the
        reference the residual is w * (proj - obs)**2 and the solve is scipy's dense
        `least_squares(method='trf')` with default options; `res.x` = cameras (11 C)."""
        C = self.cameraArray.shape[0]
        x0 = np.asarray(self.cameraArray, dtype=np.float64).ravel()
        out = self._dense_variant(_cabi.Engine.SQ_CAMONLY, x0, ftol, verbose)
        self.cameraArray = out.x.reshape((C, N_CAM_PARAMS))
        cams, pts = self.cameraArray, np.asarray(self.points3D, dtype=np.float64)
        out.set_lazy("fun", lambda: self._squared_fun(cams, pts))
        return out

    def _finish_nocam(self, lazy_fun, lazy_grad, res, pts, shard, verbose):
        x = pts.ravel().copy()
        out = BAResult(x=x, cost=res.cost, optimality=res.optimality,
                       active_mask=np.zeros_like(x), nfev=int(res.nfev), njev=int(res.njev),
                       status=int(res.status))
        out["message"] = TERMINATION_MESSAGES[int(res.status)]
        out["success"] = int(res.status) > 0
        out["solve_ms"] = res.solve_ms
        out["nit"] = int(res.iterations)
        out["gpu_launches"] = int(res.gpu_launches)
        out.set_lazy("fun", lazy_fun)
        if shard is None:
            nc = self.cameraArray.shape[0] * N_CAM_PARAMS
            out.set_lazy("grad", lambda: lazy_grad()[nc:])
        else:
            out["fun_obs_index"] = shard["obs_sel"]
        if verbose >= 1:
            print(out["message"])
            print("Function evaluations {}, initial cost {:.4e}, final cost {:.4e}, "
                  "first-order optimality {:.2e}.".format(out["nfev"], res.initial_cost,
                                                          res.cost, res.optimality))
        self.points3D = x.reshape((-1, 3))
        return out

    def bundleAdjust_nocam(self, ftol=1e-7):
        """Returns the optimized 3d positions given current camera parameters, without
        adjusting the camera parameters themselves (pySBA.py:237-250): x = points only."""
        return self.bundleAdjust(ftol, _fix_cameras=True)

    def bundleAdjust_sharedcam(self, ftol=1e-6):
        """Bundle adjustment with one (f, k1, k2) shared by all cameras (pySBA.py:286-325).
        Returns x in the reference's order [f k1 k2 | 6 extrinsics per camera | cx cy per
        camera | points]; ``cameraArray`` gets the shared intrinsics tiled."""
        return self.bundleAdjust(ftol, _shared=True)

    def bundleAdjust_transform_points_3d(self, ftol=1e-3, verbose=2):
        """Fit one 12-parameter affine map [A|t] of all 3-D points with the cameras fixed
        (pySBA.py:176-206; squared residuals, dense solve, x0 = identity); `points3D` is
        replaced by the transformed points, `res.x` = rows of [A|t]."""
        x0 = np.hstack((np.eye(3), np.zeros((3, 1)))).ravel()
        out = self._dense_variant(_cabi.Engine.SQ_TRANSFORM, x0, ftol, verbose)
        M = out.x.reshape((3, 4))
        pts = np.asarray(self.points3D, dtype=np.float64)
        self.points3D = pts @ M[:, :3].T + M[:, 3]
        cams, new_pts = np.asarray(self.cameraArray, dtype=np.float64), self.points3D
        out.set_lazy("fun", lambda: self._squared_fun(cams, new_pts))
        return out

    def getResiduals(self):
        """Residuals at the current parameters with unit weights (pySBA.py:207-213; the
        reference's version raises on a weights broadcast bug — SURVEY App. D)."""
        numCameras = self.cameraArray.shape[0]
        numPoints = self.points3D.shape[0]
        x0 = np.hstack((np.asarray(self.cameraArray).ravel(), np.asarray(self.points3D).ravel()))
        return self.fun(x0, numCameras, numPoints, self.cameraIndices, self.point2DIndices,
                        self.points2D, np.full_like(self.point2DIndices, 1))
