"""GPU tests of the parameter covariance (lcba_covariance, PySBA.covariance): the dense oracle on the golden rigs
on the DFMA and DMMA Schur routes, the int8 route at scale against DMMA and a host formula, held entries, the
refusals, the solver left undisturbed, the statistical meaning on a seeded rig, and two GPUs."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle import pysba_oracle as O
from lasercalib_b200.pySBA import PySBA
from lasercalib_b200.synth import make_rig

import _cov_oracle as CO

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROUTES = {"dfma": {"LCBA_SCHUR_MMA": "0"}, "dmma": {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "0"}}
IU = np.array([[0, 1, 2], [1, 3, 4], [2, 4, 5]])


@pytest.fixture(scope="module")
def Engine():
    from lasercalib_b200._cabi import Engine as E
    return E


def _gauge(C, P):
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    pt = np.zeros(P, bool)
    pt[[0, P // 3, 2 * P // 3]] = True
    return cam, pt


def _entry_err(cov, ref):
    """max over entries of |D (cov - ref) D|_ij / sqrt((D ref D)_ii (D ref D)_jj): every entry of the Jacobi-scaled
    matrix against its own row and column scale (D cancels; held rows, 0 in both, count as 0).  cov, ref: (..., n, n)
    stacks, one normalisation per matrix."""
    d = np.sqrt(np.einsum("...ii->...i", ref))
    d = np.where(d == 0, 1.0, d)
    return np.abs((cov - ref) / (d[..., :, None] * d[..., None, :])).max()


def _point_blocks(ref_full, C, P):
    idx = 11 * C + 3 * np.arange(P)[:, None] + np.arange(3)[None, :]
    return ref_full[idx[:, :, None], idx[:, None, :]]


@pytest.mark.parametrize("route", list(ROUTES))
@pytest.mark.parametrize("name", ["ba_ring8_volume1500", "ba_ring4_planar2000", "ba_example18_vis60_800"])
def test_covariance_matches_dense_oracle(golden, monkeypatch, record_property, name, route):
    """After a gauge-fixed bundleAdjust, camera_cov and every point_cov equal s^2 (J_f^T J_f)^-1 of the dense oracle
    at the same x to 1e-9 in every entry of the Jacobi-scaled matrices, each against its own row and column scale."""
    for k, v in ROUTES[route].items():
        monkeypatch.setenv(k, v)
    g = golden(name)
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cam, pt = _gauge(C, P)
    sba = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    sba.bundleAdjust(1e-8, verbose=0, fixed_camera_params=cam, fixed_points=pt)
    r = sba.covariance(fixed_camera_params=cam, fixed_points=pt)
    x = np.hstack((sba.cameraArray.ravel(), sba.points3D.ravel()))
    held = CO.held_vector(cam, pt, C, P)
    J, f = CO.jacobian(x, C, P, g["camera_ind"], g["point_ind"], g["points_2d"])
    ref, s2, dof = CO.covariance(J, f, held)
    nc = 11 * C
    e_cam = _entry_err(r.camera_cov, ref[:nc, :nc])
    e_pt = _entry_err(r.point_cov, _point_blocks(ref, C, P))
    record_property("camera_err", float(e_cam))
    record_property("point_err", float(e_pt))
    assert e_cam <= 1e-9 and e_pt <= 1e-9, (e_cam, e_pt)
    assert r.dof == dof and abs(r.sigma2 - s2) <= 1e-12 * s2
    assert r.min_pivot >= 3e2 * 1e-7          # lcba.cu COV_PIVOT_TOL; 4.6e-5 on ring4 planar (DESIGN.md section 8)
    np.testing.assert_array_equal(r.camera_std, np.sqrt(np.diag(r.camera_cov)).reshape(C, 11))
    # held entries exactly 0
    hc = cam.ravel()
    assert np.all(r.camera_cov[hc] == 0.0) and np.all(r.camera_cov[:, hc] == 0.0)
    assert np.all(r.point_cov[pt] == 0.0) and np.all(r.point_std[pt] == 0.0)


def test_points_only_covariance_is_s2_inverse_point_blocks(golden):
    """Every camera held: point_cov = s^2 V_p^-1 of the oracle, camera_cov = 0."""
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    x = g["tight_x"]
    sba = PySBA(x[:11 * C].reshape(C, 11).copy(), x[11 * C:].reshape(P, 3).copy(), g["points_2d"],
                g["camera_ind"], g["point_ind"])
    cam = np.ones(11, bool)
    r = sba.covariance(fixed_camera_params=cam)
    assert np.all(r.camera_cov == 0.0)
    held = CO.held_vector(np.ones((C, 11), bool), None, C, P)
    J, f = CO.jacobian(x, C, P, g["camera_ind"], g["point_ind"], g["points_2d"])
    ref, s2, _ = CO.covariance(J, f, held)
    e = _entry_err(r.point_cov, _point_blocks(ref, C, P))
    assert e <= 1e-9, e
    assert r.dof == 2 * g["camera_ind"].size - 3 * P


def test_int8_route_at_scale(Engine, monkeypatch, record_property):
    """ring24 x 50 011 points, where the int8 Schur route is the default: the camera block agrees with the DMMA
    route to 1e-11 in every Jacobi-scaled entry, 1 000 sampled point blocks agree to 1e-10 with V_p^-1 + V_p^-1 W_p^T S^-1 W_p
    V_p^-1 built on the host from lcba_jacobian_blocks and the returned S^-1, and two calls are bit-identical."""
    pb = make_rig("ring24", 50011, seed=7, variant="volume", p_vis=0.95)
    C, P = pb["n_cams"], pb["n_points"]
    ci, pi = pb["camera_ind"], pb["point_ind"]
    cam, pt = _gauge(C, P)
    e = Engine()
    e.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi)
    assert e.i8_fell_back() != -1, "the problem should take the int8 route"
    e.set_fixed(cam, pt)
    e.solve(ftol=1e-6)
    cams, pts = e.get_params()
    S_i8, pt_i8, cost, piv = e.covariance()
    S_2, pt_2, cost2, piv2 = e.covariance()
    assert np.array_equal(S_i8, S_2) and np.array_equal(pt_i8, pt_2) and cost == cost2 and piv == piv2
    Jc, Jp = e.jacobian_blocks()
    e.close()
    monkeypatch.setenv("LCBA_SCHUR_I8", "0")
    e = Engine()
    e.set_problem(cams, pts, pb["points_2d"], ci, pi)
    assert e.i8_fell_back() == -1
    e.set_fixed(cam, pt)
    S_mm, pt_mm, _, _ = e.covariance()
    e.close()
    e_cam = _entry_err(S_i8, S_mm)
    record_property("int8_vs_dmma", float(e_cam))
    assert e_cam <= 1e-11, e_cam
    # host formula on 1 000 sampled unheld points
    rng = np.random.default_rng(0)
    sample = rng.choice(np.flatnonzero(~pt), 1000, replace=False)
    order = np.argsort(pi, kind="stable")
    starts = np.searchsorted(pi[order], np.arange(P + 1))
    worst = 0.0
    for p in sample:
        obs = order[starts[p]:starts[p + 1]]
        V = np.einsum("nka,nkb->ab", Jp[obs], Jp[obs])
        W = np.zeros((11 * C, 3))
        for i in obs:
            W[11 * ci[i]:11 * ci[i] + 11] += Jc[i].T @ Jp[i]
        Vi = np.linalg.inv(V)
        ref = Vi + Vi @ W.T @ S_i8 @ W @ Vi
        worst = max(worst, _entry_err(pt_i8[p][IU], ref))
    record_property("points_vs_host", float(worst))
    assert worst <= 1e-10, worst
    assert np.all(pt_i8[pt] == 0.0)


def test_refusals(golden, Engine):
    """LinAlgError with the library's message: gauge free, an unheld point seen by one camera, a camera that sees no
    point with its entries free; holding everything is the 'every parameter is held' error."""
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    x = g["tight_x"]
    cams, pts = x[:11 * C].reshape(C, 11).copy(), x[11 * C:].reshape(P, 3).copy()
    cam, pt = _gauge(C, P)
    sba = PySBA(cams, pts, g["points_2d"], g["camera_ind"], g["point_ind"])
    with pytest.raises(np.linalg.LinAlgError, match="reduced camera system is singular"):
        sba.covariance()
    # one view of point 5 left
    ci, pi = g["camera_ind"], g["point_ind"]
    first5 = np.flatnonzero(pi == 5)[0]
    keep = (pi != 5) | (np.arange(pi.size) == first5)
    sba = PySBA(cams, pts, g["points_2d"][keep], ci[keep], pi[keep])
    with pytest.raises(np.linalg.LinAlgError, match="fewer than two distinct cameras"):
        sba.covariance(fixed_camera_params=cam, fixed_points=pt)
    pt5 = pt.copy()
    pt5[5] = True                              # held, the same point is fine
    assert sba.covariance(fixed_camera_params=cam, fixed_points=pt5).min_pivot > 1e-4
    # camera C - 1 sees nothing
    keep = ci != C - 1
    sba = PySBA(cams, pts, g["points_2d"][keep], ci[keep], pi[keep])
    with pytest.raises(np.linalg.LinAlgError, match="reduced camera system is singular"):
        sba.covariance(fixed_camera_params=cam, fixed_points=pt)
    cam_last = cam.copy()
    cam_last[C - 1] = True
    assert sba.covariance(fixed_camera_params=cam_last, fixed_points=pt).min_pivot > 1e-4
    # everything held
    sba = PySBA(cams, pts, g["points_2d"], g["camera_ind"], g["point_ind"])
    with pytest.raises(Exception, match="every parameter is held"):
        sba.covariance(fixed_camera_params=np.ones(11, bool), fixed_points=np.ones(P, bool))


def test_solver_not_disturbed_and_bounds_ignored(golden, Engine):
    """solve -> covariance -> solve from the same x0 gives the x, cost, nfev and graph replays of solve -> solve;
    bounds on the handle do not change the covariance."""
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cam, pt = _gauge(C, P)
    out = []
    for with_cov in (False, True):
        e = Engine()
        e.set_problem(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
        e.set_fixed(cam, pt)
        e.solve(ftol=1e-4)
        if with_cov:
            cov = e.covariance()
            lb = np.hstack((e.get_params()[0].ravel() - 10.0, np.full(3 * P, -1e6)))
            e.set_bounds(lb[:11 * C].reshape(C, 11), lb[:11 * C].reshape(C, 11) + 20.0,
                         np.full((P, 3), -1e6), np.full((P, 3), 1e6))
            cov_b = e.covariance()
            for a, b in zip(cov, cov_b):
                assert np.array_equal(a, b)
            e.set_bounds()
        e.set_params(g["cams0"], g["pts0"])
        res, _ = e.solve(ftol=1e-4)
        cams, pts = e.get_params()
        out.append((res.cost, res.nfev, res.reserved[0], cams, pts))
        e.close()
    (c0, n0, g0, cams0, pts0), (c1, n1, g1, cams1, pts1) = out
    assert (c0, n0, g0) == (c1, n1, g1)
    assert g0 > 0
    assert np.array_equal(cams0, cams1) and np.array_equal(pts0, pts1)


def test_predicted_variance_matches_replicates(Engine, record_property):
    """Seeded 8-camera rig, 300 points, Gaussian pixel noise of sigma = 0.5 px, 200 replicates each solved with the
    gauge held at the truth: the mean over free camera entries of empirical / predicted variance is in
    [0.85, 1.15] (predicted: sigma^2 (J_f^T J_f)^-1 at the truth)."""
    sigma, reps = 0.5, 200
    pb = make_rig("ring8", 300, seed=11, variant="volume", p_vis=1.0)
    C, P = pb["n_cams"], pb["n_points"]
    ci, pi = pb["camera_ind"], pb["point_ind"]
    x_gt = np.hstack((pb["cams_gt"].ravel(), pb["pts_gt"].ravel()))
    exact = O.fun(x_gt, C, P, ci, pi, np.zeros((ci.size, 2)), np.ones((ci.size, 1))).reshape(-1, 2)
    cam, pt = _gauge(C, P)
    e = Engine()
    e.set_problem(pb["cams_gt"], pb["pts_gt"], exact, ci, pi)
    e.set_fixed(cam, pt)
    S, _, _, _ = e.covariance(points=False)
    free = ~cam.ravel()
    pred = sigma ** 2 * np.diag(S)[free]
    rng = np.random.default_rng(12)
    sols = []
    for _ in range(reps):
        e.set_problem(pb["cams_gt"], pb["pts_gt"], exact + sigma * rng.standard_normal(exact.shape), ci, pi)
        e.set_fixed(cam, pt)
        e.solve(ftol=1e-12, xtol=1e-12, gtol=1e-12)
        sols.append(e.get_params()[0].ravel()[free])
    e.close()
    emp = np.var(np.array(sols), axis=0, ddof=1)
    ratio = float(np.mean(emp / pred))
    record_property("variance_ratio", ratio)
    assert 0.85 <= ratio <= 1.15, ratio


def test_point_sharded_covariance_matches_single_gpu():
    """Two GPUs (tests/_gpu_dist_cov_worker.py): sharded equals single-GPU to 1e-10, and a gauge-free sharded call
    fails on every rank."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(REPO, "tests", "_gpu_dist_cov_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    for r in range(2):
        assert "rank %d ok" % r in out.stdout
