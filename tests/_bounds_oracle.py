"""CPU oracle of bundleAdjust with box bounds: scipy's trf_bounds (scipy/optimize/_lsq/trf.py:203-412) restated with
the exact solve of the augmented normal equations (J_h^T J_h + diag(diag_h + reg_term)) gn_h = J_h^T f in place of
LSMR, on the FREE sub-vector of tests/_fixed_oracle.py.

Everything else is scipy's: CL_scaling_vector, the Jacobi scaling with running max, the Cauchy reg_term, the 2-D
subspace, select_step (restated below only to record which candidate it chose), make_strictly_feasible, the radius
update and the termination tests.  ``rows`` holds scipy's verbose=2 table (iteration, nfev, cost, cost reduction,
step norm, optimality) and ``choices`` the candidate of every trial: "p" (the subspace step, inside the box or pulled
back from it), "r" (reflected) or "ag" (anti-gradient)."""
import numpy as np
from numpy.linalg import norm
from scipy.linalg import qr
from scipy.optimize import OptimizeResult
from scipy.optimize._lsq.common import (CL_scaling_vector, build_quadratic_1d, check_termination,
                                        evaluate_quadratic, find_active_constraints, in_bounds,
                                        intersect_trust_region, make_strictly_feasible, minimize_quadratic_1d,
                                        solve_trust_region_2d, step_size_to_bound, update_tr_radius)
from scipy.sparse import diags
from scipy.sparse.linalg import splu

from oracle import pysba_oracle as O

from _fixed_oracle import _embed, _restricted


def select_step(x, J_h, diag_h, g_h, p, p_h, d, Delta, lb, ub, theta):
    """scipy's select_step (trf.py:129-200), line for line, returning the chosen candidate's name as well."""
    if in_bounds(x + p, lb, ub):
        p_value = evaluate_quadratic(J_h, g_h, p_h, diag=diag_h)
        return p, p_h, -p_value, "p"
    p_stride, hits = step_size_to_bound(x, p, lb, ub)
    r_h = np.copy(p_h)
    r_h[hits.astype(bool)] *= -1
    r = d * r_h
    p *= p_stride
    p_h *= p_stride
    x_on_bound = x + p
    _, to_tr = intersect_trust_region(p_h, r_h, Delta)
    to_bound, _ = step_size_to_bound(x_on_bound, r, lb, ub)
    r_stride = min(to_bound, to_tr)
    if r_stride > 0:
        r_stride_l = (1 - theta) * p_stride / r_stride
        r_stride_u = theta * to_bound if r_stride == to_bound else to_tr
    else:
        r_stride_l = 0
        r_stride_u = -1
    if r_stride_l <= r_stride_u:
        a, b, c = build_quadratic_1d(J_h, g_h, r_h, s0=p_h, diag=diag_h)
        r_stride, r_value = minimize_quadratic_1d(a, b, r_stride_l, r_stride_u, c=c)
        r_h *= r_stride
        r_h += p_h
        r = r_h * d
    else:
        r_value = np.inf
    p *= theta
    p_h *= theta
    p_value = evaluate_quadratic(J_h, g_h, p_h, diag=diag_h)
    ag_h = -g_h
    ag = d * ag_h
    to_tr = Delta / norm(ag_h)
    to_bound, _ = step_size_to_bound(x, ag, lb, ub)
    ag_stride = theta * to_bound if to_bound < to_tr else to_tr
    a, b = build_quadratic_1d(J_h, g_h, ag_h, diag=diag_h)
    ag_stride, ag_value = minimize_quadratic_1d(a, b, 0, ag_stride)
    ag_h *= ag_stride
    ag *= ag_stride
    if p_value < r_value and p_value < ag_value:
        return p, p_h, -p_value, "p"
    elif r_value < p_value and r_value < ag_value:
        return r, r_h, -r_value, "r"
    return ag, ag_h, -ag_value, "ag"


def trf_bounds_exact_generic(fun_x, jac_x, x0, lb, ub, ftol, xtol=1e-8, gtol=1e-8, max_nfev=None,
                             max_iterations=0):
    """trf_bounds with x_scale='jac', no loss, and the exact augmented solve; x0 is first moved by
    make_strictly_feasible(x0, lb, ub) as least_squares does (least_squares.py:908).  max_iterations > 0 stops after
    that many outer iterations (status 0), like lcba_options.max_iterations."""
    x = make_strictly_feasible(np.asarray(x0, dtype=np.float64), lb, ub)
    f = fun_x(x)
    if not np.all(np.isfinite(f)):
        raise ValueError("Residuals are not finite in the initial point.")
    J = jac_x(x)
    nfev = njev = 1
    m, n = J.shape
    cost = 0.5 * f @ f
    g = J.T @ f
    scale_inv = np.sqrt(np.asarray(J.power(2).sum(axis=0)).ravel())
    scale_inv[scale_inv == 0] = 1
    scale = 1 / scale_inv
    v, dv = CL_scaling_vector(x, g, lb, ub)
    v[dv != 0] *= scale_inv[dv != 0]
    Delta = norm(x * scale_inv / v**0.5)
    if Delta == 0:
        Delta = 1.0
    if max_nfev is None:
        max_nfev = n * 100
    status = None
    iteration = 0
    step_norm = actual = None
    rows, choices = [], []
    while True:
        v, dv = CL_scaling_vector(x, g, lb, ub)
        g_norm = norm(g * v, ord=np.inf)
        if g_norm < gtol:
            status = 1
        rows.append(dict(iteration=iteration, nfev=nfev, cost=cost, cost_reduction=actual, step_norm=step_norm,
                         optimality=g_norm))
        if status is not None or nfev == max_nfev or (max_iterations and iteration >= max_iterations):
            break
        v[dv != 0] *= scale_inv[dv != 0]
        d = v**0.5 * scale
        diag_h = g * dv * scale
        g_h = d * g
        J_h = J @ diags(d)
        a, b = build_quadratic_1d(J_h, g_h, -g_h, diag=diag_h)
        reg_term = -minimize_quadratic_1d(a, b, 0, Delta / norm(g_h))[1] / Delta**2
        gn_h = splu((J_h.T @ J_h + diags(diag_h + reg_term)).tocsc()).solve(J_h.T @ f)
        S, _ = qr(np.vstack((g_h, gn_h)).T, mode="economic")
        JS = J_h @ S
        B_S = JS.T @ JS + (S.T * diag_h) @ S
        g_S = S.T @ g_h
        theta = max(0.995, 1 - g_norm)
        actual = -1
        while actual <= 0 and nfev < max_nfev:
            p_S, _ = solve_trust_region_2d(B_S, g_S, Delta)
            p_h = S @ p_S
            p = d * p_h
            step, step_h, predicted, choice = select_step(x, J_h, diag_h, g_h, p, p_h, d, Delta, lb, ub, theta)
            choices.append(choice)
            x_new = make_strictly_feasible(x + step, lb, ub, rstep=0)
            f_new = fun_x(x_new)
            nfev += 1
            step_h_norm = norm(step_h)
            if not np.all(np.isfinite(f_new)):
                Delta = 0.25 * step_h_norm
                continue
            cost_new = 0.5 * f_new @ f_new
            actual = cost - cost_new
            Delta_new, ratio = update_tr_radius(Delta, actual, predicted, step_h_norm, step_h_norm > 0.95 * Delta)
            step_norm = norm(step)
            status = check_termination(actual, cost, step_norm, norm(x), ratio, ftol, xtol)
            if status is not None:
                break
            Delta = Delta_new
        if actual > 0:
            x, f, cost = x_new, f_new, cost_new
            J = jac_x(x)
            njev += 1
            g = J.T @ f
            scale_inv = np.maximum(np.sqrt(np.asarray(J.power(2).sum(axis=0)).ravel()), scale_inv)
            scale = 1 / scale_inv
        else:
            step_norm = 0
            actual = 0
        iteration += 1
    return OptimizeResult(x=x, cost=cost, fun=f, grad=g, optimality=g_norm,
                          active_mask=find_active_constraints(x, lb, ub, rtol=xtol), nfev=nfev, njev=njev,
                          status=status or 0, rows=rows, choices=choices)


def trf_bounds_fixed(cams, pts, points_2d, camera_indices, point_indices, lb, ub, weights=None, cam_fixed=None,
                     pt_fixed=None, ftol=1e-4, xtol=1e-8, gtol=1e-8, max_nfev=None, max_iterations=0):
    """trf_bounds_exact_generic on x = [cams | points] (lb, ub over that layout) with cam_fixed (C, 11) / pt_fixed (P,)
    held.  x, grad and active_mask come back in the full layout (0 at held entries)."""
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
    lb, ub = np.broadcast_to(lb, x0.shape), np.broadcast_to(ub, x0.shape)
    res = trf_bounds_exact_generic(fun_x, jac_x, x0[free], lb[free], ub[free], ftol, xtol, gtol, max_nfev,
                                   max_iterations)
    am = np.zeros(x0.size, dtype=int)
    am[free] = res.active_mask
    res = _embed(res, x0, free)
    res["active_mask"] = am
    return res
