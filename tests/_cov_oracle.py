"""Dense CPU oracle of the parameter covariance (PySBA.covariance / lcba_covariance): J_f from the numpy oracle's
Jacobian blocks over the free entries, (J_f^T J_f)^-1 by Cholesky, curve_fit's s^2; curve_fit's own SVD formula for
pcov; and the Jacobi-relative pivots l_jj^2 / S_jj of the reduced camera system that lcba_covariance tests."""
import numpy as np
from scipy.linalg import cho_factor, cho_solve

from oracle import pysba_oracle as O


def held_vector(cam_fixed, pt_fixed, C, P):
    """bool (11 C + 3 P,) over [cameraArray.ravel(), points3D.ravel()]"""
    held = np.zeros(11 * C + 3 * P, dtype=bool)
    if cam_fixed is not None:
        held[:11 * C] = np.asarray(cam_fixed).ravel()
    if pt_fixed is not None:
        held[11 * C:] = np.repeat(np.asarray(pt_fixed), 3)
    return held


def jacobian(x, C, P, camera_ind, point_ind, points_2d, weights=None):
    """(J as CSR (2N, 11 C + 3 P), f (2N,)) at x, weights included"""
    w = O.default_weights(point_ind) if weights is None else weights
    cams, pts = x[:11 * C].reshape(C, 11), x[11 * C:].reshape(P, 3)
    _, Jc, Jp = O.jacobian_blocks(cams, pts, camera_ind, point_ind, None if weights is None else weights)
    J = O.jacobian_csr(Jc, Jp, C, P, camera_ind, point_ind)
    f = O.fun(x, C, P, camera_ind, point_ind, points_2d, w)
    return J, f


def covariance(J, f, held, absolute_sigma=False):
    """curve_fit's pcov over the free entries by Cholesky of J_f^T J_f, embedded in the full layout (0 at held
    entries).  Returns (cov, sigma2, dof)."""
    free = ~held
    Jf = J[:, free]
    H = (Jf.T @ Jf).toarray()
    inv = cho_solve(cho_factor(H, lower=True), np.eye(H.shape[0]))
    m, nf = J.shape[0], int(free.sum())
    dof = m - nf
    s2 = 1.0 if absolute_sigma else float(f @ f) / dof
    cov = np.zeros((held.size, held.size))
    cov[np.ix_(free, free)] = s2 * inv
    return cov, s2, dof


def covariance_svd(J, f, held):
    """scipy.optimize.curve_fit's pcov (absolute_sigma=False): the Moore-Penrose inverse of J_f^T J_f from the
    SVD of J_f, singular values below eps max(m, n) s_max dropped, times |f|^2 / (m - n)."""
    free = ~held
    Jf = J[:, free].toarray()
    _, s, VT = np.linalg.svd(Jf, full_matrices=False)
    keep = s > np.finfo(float).eps * max(Jf.shape) * s[0]
    s, VT = s[keep], VT[:keep.size][keep]
    pcov = (VT.T / s ** 2) @ VT
    pcov *= float(f @ f) / (Jf.shape[0] - Jf.shape[1])
    cov = np.zeros((held.size, held.size))
    cov[np.ix_(free, free)] = pcov
    return cov


def reduced_camera_system(J, held, C):
    """S = U - sum_p W_p V_p^-1 W_p^T over the free entries (held camera rows / columns removed, held points
    dropped), in the camera order of lcba_covariance's S"""
    free = ~held
    nc = 11 * C
    cam_free = np.flatnonzero(free[:nc])
    pt_cols = np.flatnonzero(free[nc:]) + nc
    Jc = J[:, cam_free].tocsc()
    U = (Jc.T @ Jc).toarray()
    S = U.copy()
    Jp = J[:, pt_cols].tocsc()
    for k in range(0, pt_cols.size, 3):
        Jk = Jp[:, k:k + 3]
        rows = np.unique(Jk.nonzero()[0])
        A = Jk[rows].toarray()
        B = Jc[rows].toarray()
        V = A.T @ A
        W = B.T @ A
        S -= W @ np.linalg.solve(V, W.T)
    return S


def pivot_ratios(S):
    """l_jj^2 / S_jj of the Cholesky factorisation S = L L^T without pivoting, continued through non-positive
    pivots (LDL^T: l_jj^2 = d_j), as k_chol_fused meets them in row order"""
    A = np.array(S, dtype=np.float64)
    n = A.shape[0]
    d = np.empty(n)
    for j in range(n):
        d[j] = A[j, j]
        if j + 1 < n and d[j] != 0.0:
            l = A[j + 1:, j] / d[j]
            A[j + 1:, j + 1:] -= np.outer(l, A[j + 1:, j])
    return d / np.diag(S)
