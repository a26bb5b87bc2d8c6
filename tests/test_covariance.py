"""CPU checks of the parameter covariance: the dense oracle against curve_fit's SVD formula, the pivot threshold
of lcba_covariance's singularity test on the golden rigs, and PySBA.covariance's argument checks and scaling."""
import warnings

import numpy as np
import pytest
from scipy.optimize import OptimizeWarning

from lasercalib_b200.pySBA import PySBA, covariance_result

import _cov_oracle as CO

# lcba.cu COV_PIVOT_TOL
PIVOT_TOL = 1e-7
GAUGE_RIGS = ["ba_ring8_volume1500", "ba_example18_vis60_800"]


def _gauge(C, P):
    """the gauge mask of tests/test_gpu_fixed_params.py: camera 0's extrinsics and three points"""
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    pt = np.zeros(P, bool)
    pt[[0, P // 3, 2 * P // 3]] = True
    return cam, pt


def _rig(golden, name, n_points=None):
    g = golden(name)
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    x = g["tight_x"].copy()
    ci, pi, p2 = g["camera_ind"], g["point_ind"], g["points_2d"]
    if n_points is not None:           # the first n_points points and their observations
        sel = pi < n_points
        ci, pi, p2 = ci[sel], pi[sel], p2[sel]
        x = np.hstack((x[:11 * C], x[11 * C:11 * C + 3 * n_points]))
        P = n_points
    return x, C, P, ci, pi, p2


@pytest.mark.parametrize("name", GAUGE_RIGS)
def test_oracle_equals_curve_fit_svd_formula(golden, name):
    """(J_f^T J_f)^-1 s^2 by Cholesky equals curve_fit's pcov from the SVD of J_f.  ba_ring8_volume1500 is cut
    to its first 500 points so that the dense SVD stays small; the gauge mask holds three of them."""
    x, C, P, ci, pi, p2 = _rig(golden, name, 500 if name == "ba_ring8_volume1500" else None)
    cam, pt = _gauge(C, P)
    held = CO.held_vector(cam, pt, C, P)
    J, f = CO.jacobian(x, C, P, ci, pi, p2)
    cov, s2, dof = CO.covariance(J, f, held)
    ref = CO.covariance_svd(J, f, held)
    assert dof == 2 * ci.size - int((~held).sum())
    err = np.abs(cov - ref).max() / np.abs(ref).max()
    d = np.sqrt(np.diag(ref))
    d[d == 0] = 1.0
    err_scaled = np.abs((cov - ref) / np.outer(d, d)).max()
    print(name, "relative", err, "correlation-scaled", err_scaled)
    assert err <= 1e-9 and err_scaled <= 1e-9
    assert np.all(cov[held] == 0.0) and np.all(cov[:, held] == 0.0)


# every golden rig with a full-layout solution (tight_x); the other ba_* goldens store the x of the camera-only,
# points-only, shared-intrinsics and transform variants.  Smallest gauge-fixed margin (pivot / tau) asserted per rig:
# the issue's 1e3 on the two rigs it tabulates; ring4 planar (4 cameras, one plane of points, the weakest intrinsics)
# sits at 458 and is held to 3e2.  DESIGN.md section 8 gives the reason tau stays at 1e-7.
PIVOT_RIGS = {"ba_ring8_volume1500": 1e3, "ba_example18_vis60_800": 1e3, "ba_ring4_planar2000": 3e2}


@pytest.mark.parametrize("name", list(PIVOT_RIGS))
def test_pivot_threshold_separates_fixed_from_free_gauge(golden, name):
    """The smallest Jacobi-relative pivot l_jj^2 / S_jj of the free camera rows at the rig's tight solution: with
    the gauge mask at least PIVOT_RIGS[name] times the threshold, with the gauge free non-positive or at most 1e-2
    of it."""
    x, C, P, ci, pi, p2 = _rig(golden, name)
    J, _ = CO.jacobian(x, C, P, ci, pi, p2)
    cam, pt = _gauge(C, P)
    fixed = CO.pivot_ratios(CO.reduced_camera_system(J, CO.held_vector(cam, pt, C, P), C)).min()
    free = CO.pivot_ratios(CO.reduced_camera_system(J, CO.held_vector(None, None, C, P), C)).min()
    print(name, "gauge fixed", fixed, "gauge free", free)
    assert fixed >= PIVOT_RIGS[name] * PIVOT_TOL
    assert free <= 1e-2 * PIVOT_TOL


def _sba(C=3, P=10):
    rng = np.random.default_rng(0)
    ci = np.repeat(np.arange(C), P)
    pi = np.tile(np.arange(P), C)
    return PySBA(rng.random((C, 11)), rng.random((P, 3)), rng.random((ci.size, 2)), ci, pi)


@pytest.mark.parametrize("kw, msg", [
    (dict(fixed_camera_params=np.zeros(10, bool)), "fixed_camera_params must have shape"),
    (dict(fixed_camera_params=np.zeros(11, int)), "must be a bool array"),
    (dict(fixed_points=np.zeros(4, bool)), "a bool fixed_points must have shape"),
    (dict(fixed_points=np.array([0, 10])), "indices must lie in"),
    (dict(fixed_points=np.zeros(10, float)), "bool mask or an integer index array"),
])
def test_covariance_argument_errors_before_the_gpu(kw, msg):
    sba = _sba()
    with pytest.raises(ValueError, match=msg):
        sba.covariance(**kw)
    assert sba._engine is None


def test_covariance_result_scaling_and_dof():
    rng = np.random.default_rng(1)
    C, P = 2, 4
    A = rng.standard_normal((22, 22))
    cam = A @ A.T
    pt6 = rng.random((P, 6))
    cam_fixed = np.zeros((C, 11), bool)
    cam_fixed[0, :6] = True
    cam[cam_fixed.ravel()] = 0.0
    cam[:, cam_fixed.ravel()] = 0.0
    pt_fixed = np.array([True, False, False, False])
    pt6[0] = 0.0
    n_free = 22 - 6 + 3 * 3
    # curve_fit: s^2 = |f|^2 / (m - n), cost = |f|^2 / 2
    r = covariance_result(cam, pt6, 3.0, 0.5, n_free + 5, cam_fixed, pt_fixed)
    assert r.dof == 5 and r.sigma2 == pytest.approx(6.0 / 5)
    np.testing.assert_array_equal(r.camera_cov, cam * (6.0 / 5))
    assert r.point_cov.shape == (P, 3, 3) and np.allclose(r.point_cov, np.swapaxes(r.point_cov, 1, 2))
    assert r.point_cov[1, 0, 2] == pt6[1, 2] * (6.0 / 5) and r.point_cov[1, 2, 1] == pt6[1, 4] * (6.0 / 5)
    np.testing.assert_array_equal(r.camera_std, np.sqrt(np.diag(r.camera_cov)).reshape(C, 11))
    np.testing.assert_array_equal(r.point_std[:, 1], np.sqrt(r.point_cov[:, 1, 1]))
    assert r.min_pivot == 0.5 and r.cost == 3.0
    # absolute_sigma: no scaling, also when dof <= 0
    for m in (n_free + 5, n_free):
        r = covariance_result(cam, pt6, 3.0, 0.5, m, cam_fixed, pt_fixed, absolute_sigma=True)
        assert r.sigma2 == 1.0
        np.testing.assert_array_equal(r.camera_cov, cam)
    # dof <= 0: inf at the free entries with a warning, held entries stay 0
    for m in (n_free, n_free - 3):
        with warnings.catch_warnings(record=True) as w:
            warnings.simplefilter("always")
            r = covariance_result(cam, pt6, 3.0, 0.5, m, cam_fixed, pt_fixed)
        assert any(issubclass(x.category, OptimizeWarning) for x in w)
        free = ~cam_fixed.ravel()
        assert np.all(np.isinf(r.camera_cov[np.ix_(free, free)]))
        assert np.all(r.camera_cov[~free] == 0.0) and np.all(r.point_cov[0] == 0.0)
        assert np.all(np.isinf(r.point_cov[1:]))
