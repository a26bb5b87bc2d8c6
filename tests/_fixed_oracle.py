"""CPU oracle of bundleAdjust with held parameters: scipy's trf_no_bounds restated with an exact
solve (oracle.pysba_oracle.trf_exact_generic) on the FREE sub-vector, with the same residuals.

A held parameter is a constant of the residual function, so the masked problem is the unmasked
one with its Jacobian restricted to the free columns: fun_x embeds the free sub-vector into the
full x, jac_x = jacobian_csr(...)[:, free]."""
import numpy as np
from scipy.sparse import csr_matrix

from oracle import pysba_oracle as O


def _restricted(fun_full, jac_full, x_full, free):
    def fun_x(xf):
        x = x_full.copy()
        x[free] = xf
        return fun_full(x)

    def jac_x(xf):
        x = x_full.copy()
        x[free] = xf
        return jac_full(x)[:, free].tocsr()

    return fun_x, jac_x


def _embed(res, x_full, free):
    x = x_full.copy()
    x[free] = res.x
    g = np.zeros(x_full.size)
    g[free] = res.grad
    res["x_free"], res["grad_free"] = res.x, res.grad
    res["x"], res["grad"] = x, g
    return res


def trf_exact_fixed(cams, pts, points_2d, camera_indices, point_indices, weights=None,
                    cam_fixed=None, pt_fixed=None, ftol=1e-4, xtol=1e-8, gtol=1e-8, max_nfev=None):
    """trf_exact on x = [cams | points] with cam_fixed (C, 11) / pt_fixed (P,) held.  Returns the
    OptimizeResult of trf_exact_generic with x and grad in the full layout (grad 0 at held entries)
    and the reduced ones as x_free / grad_free."""
    C, P = cams.shape[0], pts.shape[0]
    if weights is None:
        weights = O.default_weights(point_indices)
    weights = np.asarray(weights).reshape(-1, 1)
    held = np.zeros(11 * C + 3 * P, dtype=bool)
    if cam_fixed is not None:
        held[:11 * C] = np.asarray(cam_fixed, dtype=bool).ravel()
    if pt_fixed is not None:
        held[11 * C:] = np.repeat(np.asarray(pt_fixed, dtype=bool), 3)
    free = np.flatnonzero(~held)
    x0 = np.hstack((cams.ravel(), pts.ravel())).astype(np.float64)
    args = (C, P, camera_indices, point_indices, points_2d, weights)

    def jac_full(x):
        _, Jc, Jp = O.jacobian_blocks(x[:11 * C].reshape(C, 11), x[11 * C:].reshape(P, 3), camera_indices,
                                      point_indices, weights)
        return O.jacobian_csr(Jc, Jp, C, P, camera_indices, point_indices)

    fun_x, jac_x = _restricted(lambda x: O.fun(x, *args), jac_full, x0, free)
    res = O.trf_exact_generic(fun_x, jac_x, x0[free], ftol, xtol, gtol, max_nfev)
    return _embed(res, x0, free)


def trf_exact_sharedcam_fixed(cams, pts, points_2d, camera_indices, point_indices, pt_fixed, weights=None,
                              ftol=1e-6, xtol=1e-8, gtol=1e-8, max_nfev=None):
    """The shared-intrinsics parameterisation [f k1 k2 | extrinsics | centres | points] with the points of
    pt_fixed held (x, grad returned in that parameterisation)."""
    C, P = cams.shape[0], pts.shape[0]
    if weights is None:
        weights = O.default_weights(point_indices)
    weights = np.asarray(weights).reshape(-1, 1)
    args = (C, P, camera_indices, point_indices, points_2d, weights)
    A = O.sparsity_sharedcam(C, P, camera_indices, point_indices)

    def jac_full(x):
        cm, pt = O.sharedcam_unpack(x, C, P)
        _, Jc, Jp = O.jacobian_blocks(cm, pt, camera_indices, point_indices, weights)
        data = np.concatenate([Jc[:, :, 6:9], Jc[:, :, 0:6], Jc[:, :, 9:11], Jp], axis=2).reshape(-1)
        return csr_matrix((data, A.indices, A.indptr), shape=A.shape)

    x0 = O.sharedcam_pack(cams, pts)
    held = np.zeros(x0.size, dtype=bool)
    held[3 + 8 * C:] = np.repeat(np.asarray(pt_fixed, dtype=bool), 3)
    free = np.flatnonzero(~held)
    fun_x, jac_x = _restricted(lambda x: O.fun_sharedcam(x, *args), jac_full, x0, free)
    res = O.trf_exact_generic(fun_x, jac_x, x0[free], ftol, xtol, gtol, max_nfev)
    return _embed(res, x0, free)
