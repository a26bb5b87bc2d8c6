"""Held parameters (lcba_set_fixed, PySBA.bundleAdjust(fixed_camera_params=..., fixed_points=...)) on the
GPU: one Gauss-Newton step on every pass and Schur route against the damped normal equations of J[:, free],
whole solves against the CPU oracle of the masked problem (tests/_fixed_oracle.py), and the bookkeeping of
the masks on a resident problem (held entries bit-identical, graph replays, clearing)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from oracle import pysba_oracle as O
from lasercalib_b200.synth import make_rig

from _fixed_oracle import trf_exact_fixed, trf_exact_sharedcam_fixed
from test_gpu_step import _check_step, _jacobian, _problem

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# pass routes (LCBA_PT_PASSES) and Schur routes (LCBA_SCHUR_MMA / LCBA_SCHUR_I8) as the other GPU tests select them
ROUTES = {"pt": {}, "generic": {"LCBA_PT_PASSES": "0"},
          "dfma": {"LCBA_SCHUR_MMA": "0"}, "dmma": {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "0"},
          "i8": {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "1"}}
MASKS = ["cam0_extrinsics", "intrinsics", "random30", "whole_camera", "camera_sees_held_points", "points10"]


@pytest.fixture(scope="module")
def Engine():
    from lasercalib_b200._cabi import Engine as E
    return E


def _masks(kind, C, P, ci, pi, seed):
    rng = np.random.default_rng(seed)
    cam = np.zeros((C, 11), bool)
    pt = np.zeros(P, bool)
    if kind == "cam0_extrinsics":
        cam[0, :6] = True
    elif kind == "intrinsics":
        cam[:, 6:] = True
    elif kind == "random30":
        cam = rng.random((C, 11)) < 0.3
    elif kind == "whole_camera":
        cam[C // 2, :] = True
    elif kind == "camera_sees_held_points":
        pt[np.unique(pi[ci == C - 1])] = True
    elif kind == "points10":
        pt = rng.random(P) < 0.1
    return cam, pt


def _held(cam, pt):
    return np.concatenate([cam.ravel(), np.repeat(pt, 3)])


@pytest.mark.parametrize("kind", MASKS)
@pytest.mark.parametrize("C", [3, 8, 24, 64])
def test_masked_step_matches_oracle_on_every_route(Engine, monkeypatch, record_property, C, kind):
    """lcba_debug_step with masks against the damped normal equations of J[:, free] (test_gpu_step._check_step:
    normal-equation residual 1e-11, forward error 1e-11 cond, reg_term / Jg2 / Delta, Gram totals 1e-12,
    subspace scalars), on the pass routes pt / generic and the Schur routes DFMA / DMMA / int8.  Held
    entries of the step are exactly 0; the steps agree over the routes to max(1e-12, 1e-13 cond) scaled.
    Measured on a B200 (1000 W): residual <= 2.8e-14, forward error <= 1.5e-15 cond, Gram totals <= 3.7e-14,
    subspace scalars <= 2.9e-13, routes <= 4.8e-12 (int8)."""
    lam = 1e-3
    pb = _problem(C, seed=100 + C)
    ci, pi = pb["camera_ind"], pb["point_ind"]
    Cn, P = pb["cams0"].shape[0], pb["pts0"].shape[0]
    cam, pt = _masks(kind, Cn, P, ci, pi, seed=C)
    held = _held(cam, pt)
    free = np.flatnonzero(~held)
    J, f, x = _jacobian(pb, 0)
    Jf = J[:, free].tocsr()
    s = np.sqrt(np.asarray(Jf.multiply(Jf).sum(axis=0)).ravel())
    s[s == 0] = 1.0
    H = (Jf.T @ Jf).toarray() + np.diag(lam * s * s)
    p_or = cho_solve(cho_factor(H, lower=True), Jf.T @ f)
    steps = {}
    for route, env in ROUTES.items():
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = Engine()
        e.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi, pb["w"])
        e.set_fixed(cam, pt)
        pc, pp, sc = e.debug_step(lam, 0.0, 0)
        e.close()
        for k in env:
            monkeypatch.delenv(k)
        p = np.hstack((pc, pp))
        assert np.all(p[held] == 0.0), route
        kappa = _check_step(Jf, f, x[free], lam, p_or, p[free], sc, record_property, route)
        steps[route] = p
    p0 = steps["pt"]
    sf = np.ones(held.size)
    sf[free] = s
    for route, p in steps.items():      # the Schur routes round S differently: 1e-13 of its condition
        d = np.abs(sf * (p - p0)).max() / np.abs(sf * p0).max()
        record_property("routes_" + route, float(d))
        assert d <= max(1e-12, 1e-13 * kappa), (route, d, kappa)


def _gauge(C, P):
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    pt = np.zeros(P, bool)
    pt[[0, P // 3, 2 * P // 3]] = True
    return cam, pt


def _solve(Engine, g, cam, pt, ftol=1e-4, **kw):
    e = Engine()
    e.set_problem(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    e.set_fixed(cam, pt)
    res, trace = e.solve(ftol=ftol, **kw)
    cams, pts = e.get_params()
    grad = e.grad()
    e.close()
    return res, trace, cams, pts, grad


# error of every parameter group against the oracle, relative to the group's largest entry: rotvec, t,
# intrinsics (per column), points
def _param_errors(x, xo, C):
    c, co = x[:11 * C].reshape(C, 11), xo[:11 * C].reshape(C, 11)
    out = dict(rotvec=np.abs(c[:, :3] - co[:, :3]).max() / np.abs(co[:, :3]).max(),
               t=np.abs(c[:, 3:6] - co[:, 3:6]).max() / np.abs(co[:, 3:6]).max(),
               points=np.abs(x[11 * C:] - xo[11 * C:]).max() / np.abs(xo[11 * C:]).max())
    intr = np.abs(c[:, 6:] - co[:, 6:]).max(axis=0) / np.maximum(np.abs(co[:, 6:]).max(axis=0), 1e-300)
    out["intrinsics"] = intr.max()
    return out


# measured on a B200 (1000 W): 3.3e-12 at most (intrinsics of ring4 planar), rotvec / t / points <= 6.5e-15
PARAM_RTOL = 1e-9


def _masked_grad(g, x, held):
    """J^T f at x on the CPU, 0 at held entries."""
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    ci, pi = g["camera_ind"], g["point_ind"]
    _, Jc, Jp = O.jacobian_blocks(x[:11 * C].reshape(C, 11), x[11 * C:].reshape(P, 3), ci, pi)
    f = O.fun(x, C, P, ci, pi, g["points_2d"], O.default_weights(pi))
    gr = O.jacobian_csr(Jc, Jp, C, P, ci, pi).T @ f
    gr[held] = 0.0
    return gr


@pytest.mark.parametrize("name", ["ba_ring8_volume1500", "ba_ring4_planar2000", "ba_example18_vis60_800"])
def test_gauge_fixed_solve_matches_oracle_in_every_parameter(Engine, golden, record_property, name):
    """Camera 0's extrinsics and three non-collinear points held: the 7 gauge modes are gone, so not only the
    costs but every parameter (rotvec, t, intrinsics, points) must agree with trf_exact_fixed.  nfev, njev and
    status equal; cost trace rtol 3e-7, final cost rtol 1e-9; parameters within PARAM_RTOL of their group's
    largest entry; held entries bit-identical, gradient 0 there.  |g|_inf over the free entries: at x0 (trace
    row 0) to 1e-8 of J[:, free]^T f computed on the CPU; the returned gradient is J[:, free]^T f at the
    returned x.  The final optimality of the two solves is compared on the scale of the first, as in
    test_gpu_parity: the final iterates differ by round-off while the gradient has shrunk by orders of
    magnitude, so its relative difference is not small.  Measured on a B200 (1000 W): final optimality 1.5e-13
    of the first, returned gradient 1.0e-13 of it from the CPU's."""
    g = golden(name)
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cam, pt = _gauge(C, P)
    ora = trf_exact_fixed(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"],
                          cam_fixed=cam, pt_fixed=pt, ftol=1e-4)
    res, trace, cams, pts, grad = _solve(Engine, g, cam, pt)
    assert (res.nfev, res.njev, res.status) == (ora.nfev, ora.njev, ora.status)
    np.testing.assert_allclose([r["cost"] for r in trace], ora.trace, rtol=3e-7)
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-9)
    x = np.hstack((cams.ravel(), pts.ravel()))
    held = _held(cam, pt)
    x0 = np.hstack((g["cams0"].ravel(), g["pts0"].ravel()))
    assert np.array_equal(x[held].view(np.int64), x0[held].view(np.int64))
    assert np.all(grad[held] == 0.0)
    opt0 = np.abs(_masked_grad(g, x0, held)).max()
    np.testing.assert_allclose(trace[0]["optimality"], opt0, rtol=1e-8)
    record_property("optimality_final_vs_first", float(abs(res.optimality - ora.optimality) / opt0))
    assert abs(res.optimality - ora.optimality) <= 1e-10 * opt0, (res.optimality, ora.optimality, opt0)
    np.testing.assert_allclose(res.optimality, np.abs(grad).max(), rtol=1e-12)
    gx = _masked_grad(g, x, held)
    record_property("grad_vs_cpu", float(np.abs(grad - gx).max() / opt0))
    assert np.abs(grad - gx).max() <= 1e-10 * opt0
    errs = _param_errors(x, ora.x, C)
    for k, v in errs.items():
        record_property("param_" + k, float(v))
    assert max(errs.values()) <= PARAM_RTOL, errs


def test_pysba_masks_hold_entries_and_keep_the_layout(golden):
    """bundleAdjust(fixed_camera_params (11,), fixed_points indices): res.x, cameraArray and points3D equal the
    input bit for bit at held entries; x and jac keep the full layout; grad is 0 at held entries, also when read
    after the engine solved another problem (the unmasked re-linearisation path); optimality = |grad|_inf."""
    from lasercalib_b200.pySBA import PySBA
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cm = np.zeros(11, bool)
    cm[[0, 1, 2, 9, 10]] = True
    idx = np.array([5, 50, 500, 1000])
    sba = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    res = sba.bundleAdjust(1e-4, verbose=0, fixed_camera_params=cm, fixed_points=idx)
    ptm = np.zeros(P, bool)
    ptm[idx] = True
    held = _held(np.tile(cm, (C, 1)), ptm)
    x0 = np.hstack((g["cams0"].ravel(), g["pts0"].ravel()))
    assert res.x.shape == x0.shape and res.jac.shape == (2 * g["camera_ind"].size, x0.size)
    assert np.array_equal(res.x[held].view(np.int64), x0[held].view(np.int64))
    assert np.array_equal(sba.cameraArray[:, cm].view(np.int64), g["cams0"][:, cm].view(np.int64))
    assert np.array_equal(sba.points3D[idx].view(np.int64), g["pts0"][idx].view(np.int64))
    assert not np.array_equal(res.x[~held], x0[~held])
    # lazy grad read after another solve used the shared engine
    other = make_rig("ring4", 300, seed=2)
    sb = PySBA(other["cams0"].copy(), other["pts0"].copy(), other["points_2d"], other["camera_ind"], other["point_ind"])
    sb.bundleAdjust(1e-4, verbose=0)
    gr = res.grad
    assert np.all(gr[held] == 0.0)
    assert abs(np.abs(gr).max() - res.optimality) <= 1e-9 * res.optimality
    full = res.jac.T @ res.fun
    np.testing.assert_allclose(gr[~held], full[~held], rtol=0, atol=1e-9 * np.abs(full).max())
    # the same read on the live engine (no re-upload) gives the same values
    sba2 = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    res2 = sba2.bundleAdjust(1e-4, verbose=0, fixed_camera_params=cm, fixed_points=idx)
    np.testing.assert_array_equal(res2.x, res.x)
    np.testing.assert_allclose(res2.grad, gr, rtol=0, atol=1e-12 * np.abs(gr).max())


def _fresh(Engine, g, cam, pt):
    res, _, cams, pts, _ = _solve(Engine, g, cam, pt)
    return res, np.hstack((cams.ravel(), pts.ravel()))


def test_cleared_masks_and_mask_changes_on_a_resident_problem(Engine, golden):
    """On one resident problem: (a) solve, set masks, clear them, solve again: bit-identical to a fresh handle's
    unmasked solve; (b) two masked solves with different masks, the second a CUDA-graph replay
    (reserved[0] > 0): each bit-identical to a fresh handle with that mask."""
    g = golden("ba_example18_vis60_800")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    m1 = _gauge(C, P)
    m2 = (np.zeros((C, 11), bool), np.zeros(P, bool))
    m2[0][:, 6:9] = True
    m2[1][np.arange(0, P, 7)] = True
    ref0, x_ref0 = _fresh(Engine, g, None, None)
    ref1, x_ref1 = _fresh(Engine, g, *m1)
    ref2, x_ref2 = _fresh(Engine, g, *m2)
    e = Engine()
    e.set_problem(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    e.solve(ftol=1e-4)
    outs = []
    for masks, clear in (((m1[0], m1[1]), True), (m1, False), (m2, False)):
        e.set_params(g["cams0"], g["pts0"])
        e.set_fixed(*masks)
        if clear:
            e.set_fixed(None, None)
        r, _ = e.solve(ftol=1e-4)
        cams, pts = e.get_params()
        outs.append((r, np.hstack((cams.ravel(), pts.ravel()))))
    e.close()
    for (r, x), (rr, xr) in zip(outs, ((ref0, x_ref0), (ref1, x_ref1), (ref2, x_ref2))):
        assert r.reserved[0] > 0
        assert (r.nfev, r.njev, r.status) == (rr.nfev, rr.njev, rr.status)
        assert r.cost == rr.cost
        np.testing.assert_array_equal(x, xr)


def test_point_mask_with_fix_cameras_and_shared_intrinsics(Engine, golden):
    """The point mask under fix_cameras (against the oracle with every camera entry held) and under
    shared_intrinsics (against the shared parameterisation with the points held); a camera mask with
    shared_intrinsics is LCBA_E_UNSUPPORTED; holding every parameter is LCBA_E_ARG."""
    from lasercalib_b200._cabi import LcbaError
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    pt = np.zeros(P, bool)
    pt[np.arange(0, P, 10)] = True
    ora = trf_exact_fixed(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"],
                          cam_fixed=np.ones((C, 11), bool), pt_fixed=pt, ftol=1e-7)
    res, trace, cams, pts, _ = _solve(Engine, g, None, pt, ftol=1e-7, fix_cameras=True)
    assert (res.nfev, res.status) == (ora.nfev, ora.status)
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-9)
    np.testing.assert_array_equal(cams, g["cams0"])
    np.testing.assert_array_equal(pts[pt], g["pts0"][pt])
    np.testing.assert_allclose(pts.ravel(), ora.x[11 * C:], rtol=0, atol=1e-6 * np.abs(ora.x[11 * C:]).max())
    cams_sh = g["cams0"].copy()
    cams_sh[:, 6:9] = cams_sh[:, 6:9].mean(axis=0)
    ora = trf_exact_sharedcam_fixed(cams_sh, g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"], pt, ftol=1e-6)
    e = Engine()
    e.set_problem(cams_sh, g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    e.set_fixed(None, pt)
    res, trace = e.solve(ftol=1e-6, shared_intrinsics=True)
    _, pts = e.get_params()
    assert (res.nfev, res.status) == (ora.nfev, ora.status)
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-9)
    np.testing.assert_array_equal(pts[pt], g["pts0"][pt])
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    e.set_params(cams_sh, g["pts0"])
    e.set_fixed(cam, pt)
    with pytest.raises(LcbaError) as ei:
        e.solve(ftol=1e-6, shared_intrinsics=True)
    assert ei.value.code == -4
    with pytest.raises(LcbaError) as ei:
        e.debug_step(1e-3, 0.0, 2)
    assert ei.value.code == -4
    e.set_fixed(np.ones((C, 11), bool), np.ones(P, bool))
    for kw in ({}, {"fix_cameras": True}):
        with pytest.raises(LcbaError) as ei:
            e.solve(ftol=1e-4, **kw)
        assert ei.value.code == -1
    with pytest.raises(LcbaError) as ei:
        e.debug_step(1e-3, 0.0, 0)
    assert ei.value.code == -1
    with pytest.raises(ValueError):
        e.set_fixed(np.ones((C + 1, 11), bool), None)
    e.set_fixed(None, None)
    e.solve(ftol=1e-4)            # cleared: solves again
    e.close()


def test_int8_route_with_masks_agrees_with_dmma(Engine, monkeypatch):
    """Ring24 x 150 k (the int8 Schur path's default size range) with the gauge mask and 1 % held points: a
    whole solve(ftol=1e-4) on the int8 route and on the DMMA route agree as in test_gpu_i8_scale (equal nfev
    and status, cost rtol 1e-10); held entries bit-identical on both."""
    pb = make_rig("ring24", 150_000, seed=21, variant="volume", p_vis=1.0)
    C, P = pb["n_cams"], pb["n_points"]
    cam, _ = _gauge(C, P)
    pt = np.random.default_rng(3).random(P) < 0.01
    held = _held(cam, pt)
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    out = {}
    for name, env in (("i8", {"LCBA_SCHUR_I8": "1"}), ("dmma", {"LCBA_SCHUR_I8": "0"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = Engine()
        e.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
        e.set_fixed(cam, pt)
        r, _ = e.solve(ftol=1e-4)
        cams, pts = e.get_params()
        e.close()
        for k in env:
            monkeypatch.delenv(k)
        x = np.hstack((cams.ravel(), pts.ravel()))
        assert np.array_equal(x[held], x0[held]), name
        out[name] = r
    a, b = out["i8"], out["dmma"]
    assert (a.nfev, a.status) == (b.nfev, b.status)
    np.testing.assert_allclose(a.cost, b.cost, rtol=1e-10)


def test_point_sharded_masked_solve_matches_single_gpu():
    """Two GPUs (tests/_gpu_dist_fixed_worker.py): held points on both sides of the shard cut and the gauge
    camera mask; same nfev and status as one GPU, cost within 1e-12; different camera masks over the ranks
    fail on every rank."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(REPO, "tests", "_gpu_dist_fixed_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    for r in range(2):
        assert "rank %d ok" % r in out.stdout
