"""Box bounds (lcba_set_bounds, PySBA.bundleAdjust(bounds=...)) on the GPU: infinite bounds change nothing, gauge-fixed
bounded solves against the CPU oracle of trf_bounds (tests/_bounds_oracle.py), the bounds' damping in one step of
every Schur route, and the combinations that are refused."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from lasercalib_b200.pySBA import PySBA
from lasercalib_b200.synth import make_rig

from _bounds_oracle import trf_bounds_fixed
from test_bounds import RIGS as SMALL_RIGS, _binding_box
from test_gpu_fixed_params import PARAM_RTOL, ROUTES, _gauge, _held, _param_errors

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu
RIGS = ["ba_ring8_volume1500", "ba_ring4_planar2000", "ba_example18_vis60_800"]


@pytest.fixture(scope="module")
def Engine():
    from lasercalib_b200._cabi import Engine as E
    return E


def _box(g):
    """k1 within 5e-4 and k2 within 2e-3 of x0, every point above the lowest initial z: binds on the golden rigs."""
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    lb, ub = np.full(11 * C + 3 * P, -np.inf), np.full(11 * C + 3 * P, np.inf)
    c0 = g["cams0"]
    lc, uc = lb[:11 * C].reshape(C, 11), ub[:11 * C].reshape(C, 11)
    lc[:, 7], uc[:, 7] = c0[:, 7] - 5e-4, c0[:, 7] + 5e-4
    lc[:, 8], uc[:, 8] = c0[:, 8] - 2e-3, c0[:, 8] + 2e-3
    lb[11 * C + 2::3] = g["pts0"][:, 2].min()
    return lb, ub


def _set_box(e, lb, ub, C):
    nc = 11 * C
    e.set_bounds(lb[:nc].reshape(C, 11), ub[:nc].reshape(C, 11), lb[nc:].reshape(-1, 3), ub[nc:].reshape(-1, 3))


def _engine(Engine, g, cam=None, pt=None, box=None):
    e = Engine()
    e.set_problem(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    if cam is not None or pt is not None:
        e.set_fixed(cam, pt)
    if box is not None:
        _set_box(e, *box, g["cams0"].shape[0])
    return e


def _x(e):
    cams, pts = e.get_params()
    return np.hstack((cams.ravel(), pts.ravel()))


def test_infinite_bounds_are_bit_identical_to_no_bounds(Engine, golden):
    """All-infinite bounds run the unbounded loop: x, cost, nfev and the trace are the same bits, on a fresh problem
    and on the resident problem's second solve (graph replays)."""
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    inf = np.full(11 * C + 3 * P, np.inf)
    out = []
    for box in (None, (-inf, inf)):
        e = _engine(Engine, g, box=box)
        runs = []
        for _ in range(2):
            e.set_params(g["cams0"], g["pts0"])
            res, trace = e.solve(ftol=1e-4)
            runs.append((_x(e), res.cost, res.nfev, res.reserved[0], np.array([list(r.values()) for r in trace])))
        e.close()
        out.append(runs)
    for a, b in zip(*out):
        assert np.array_equal(a[0].view(np.int64), b[0].view(np.int64))
        assert a[1:4] == b[1:4]
        assert np.array_equal(a[4], b[4], equal_nan=True)
    assert out[0][1][3] > 0     # the second solve replayed graphs


@pytest.mark.parametrize("name", RIGS)
def test_gauge_fixed_bounded_solve_matches_oracle(Engine, golden, record_property, name):
    """Camera 0's extrinsics and three points held, binding k1 / k2 / z bounds: nfev, njev and status equal; the trace
    (cost rtol 3e-7, nfev, step norm and optimality to 1e-6 of the first row's) follows the oracle; every parameter
    within PARAM_RTOL; active_mask equal; x strictly inside the box."""
    g = golden(name)
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cam, pt = _gauge(C, P)
    lb, ub = _box(g)
    ora = trf_bounds_fixed(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"], lb, ub,
                           cam_fixed=cam, pt_fixed=pt, ftol=1e-4)
    e = _engine(Engine, g, cam, pt, (lb, ub))
    res, trace = e.solve(ftol=1e-4)
    x = _x(e)
    am = e.active_mask(1e-8)
    e.close()
    assert (res.nfev, res.njev, res.status) == (ora.nfev, ora.njev, ora.status)
    assert [r["nfev"] for r in trace] == [r["nfev"] for r in ora.rows]
    np.testing.assert_allclose([r["cost"] for r in trace], [r["cost"] for r in ora.rows], rtol=3e-7)
    opt0 = ora.rows[0]["optimality"]
    np.testing.assert_allclose([r["optimality"] for r in trace], [r["optimality"] for r in ora.rows],
                               atol=1e-6 * opt0)
    sn = [r["step_norm"] for r in ora.rows[1:]]
    np.testing.assert_allclose([r["step_norm"] for r in trace[1:]], sn, rtol=1e-6, atol=1e-9 * max(sn))
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-9)
    errs = _param_errors(x, ora.x, C)
    for k, v in errs.items():
        record_property("param_" + k, float(v))
    assert max(errs.values()) <= PARAM_RTOL, errs
    held = _held(cam, pt)
    x0 = np.hstack((g["cams0"].ravel(), g["pts0"].ravel()))
    assert np.array_equal(x[held].view(np.int64), x0[held].view(np.int64))
    assert np.array_equal(am, ora.active_mask)
    assert np.all((x[~held] > lb[~held]) & (x[~held] < ub[~held]))


def test_every_iterate_is_strictly_inside(Engine, golden):
    """After max_iterations = k for every k the solve reaches, x lies strictly inside the box."""
    g = golden("ba_example18_vis60_800")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cam, pt = _gauge(C, P)
    lb, ub = _box(g)
    free = ~_held(cam, pt)
    e = _engine(Engine, g, cam, pt, (lb, ub))
    for k in range(1, 8):
        e.set_params(g["cams0"], g["pts0"])
        e.solve(ftol=1e-4, max_iterations=k)
        x = _x(e)
        assert np.all((x[free] > lb[free]) & (x[free] < ub[free])), k
    e.close()


def test_bounded_step_on_every_route(Engine, golden, monkeypatch):
    """lcba_debug_step with bounds: the Gauss-Newton step solves (J^T J + diag(e)) p = J^T f with the bounded damping
    e = (diag_h + lam) / d^2 (x strictly inside), on the pass routes and the Schur routes DFMA / DMMA / int8."""
    from scipy.optimize._lsq.common import CL_scaling_vector
    from oracle import pysba_oracle as O
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    ci, pi = g["camera_ind"], g["point_ind"]
    lb, ub = _box(g)
    lb[11 * C + 2::3] -= 1.0
    x0 = np.hstack((g["cams0"].ravel(), g["pts0"].ravel()))
    _, Jc, Jp = O.jacobian_blocks(g["cams0"], g["pts0"], ci, pi)
    J = O.jacobian_csr(Jc, Jp, C, P, ci, pi)
    f = O.fun(x0, C, P, ci, pi, g["points_2d"], O.default_weights(pi))
    gr = J.T @ f
    s = np.sqrt(np.asarray(J.multiply(J).sum(axis=0)).ravel())
    s[s == 0] = 1.0
    v, dv = CL_scaling_vector(x0, gr, lb, ub)
    v[dv != 0] *= s[dv != 0]
    d = np.sqrt(v) / s
    lam = 1e-3
    e_diag = (gr * dv / s + lam) / d**2
    H = (J.T @ J).toarray() + np.diag(e_diag)
    p_or = np.linalg.solve(H, gr)
    ref = None
    for route, env in ROUTES.items():
        for k, val in env.items():
            monkeypatch.setenv(k, val)
        eng = _engine(Engine, g, box=(lb, ub))
        pc, pp, sc = eng.debug_step(lam, 0.0, 0)
        eng.close()
        for k in env:
            monkeypatch.delenv(k)
        p = np.hstack((pc, pp))
        r = np.abs(H @ p - gr).max() / (np.abs(H) @ np.abs(p)).max()   # backward error of the solve
        assert r <= 1e-11, (route, r)
        if ref is None:
            ref = p
        assert np.abs(s * (p - ref)).max() <= 1e-7 * np.abs(s * ref).max(), route
    assert np.abs(s * (ref - p_or)).max() <= 1e-6 * np.abs(s * p_or).max()


def test_refused_combinations(Engine, golden):
    """fix_cameras or shared_intrinsics with bounds: LCBA_E_UNSUPPORTED; lb >= ub or x0 outside the box on a free
    entry: LCBA_E_ARG; the same violation on a held entry is ignored, so masks plus bounds solve."""
    from lasercalib_b200._cabi import LcbaError
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    lb, ub = _box(g)
    e = _engine(Engine, g, box=(lb, ub))
    for kw in (dict(fix_cameras=True), dict(shared_intrinsics=True)):
        with pytest.raises(LcbaError) as ei:
            e.solve(ftol=1e-4, **kw)
        assert ei.value.code == -4, kw
    bad_ub = ub.copy()
    bad_ub[11 * C + 5] = lb[11 * C + 5] = 1.0
    _set_box(e, lb, bad_ub, C)
    with pytest.raises(LcbaError) as ei:
        e.solve(ftol=1e-4)
    assert ei.value.code == -1
    lb2, ub2 = _box(g)
    ub2[7] = g["cams0"][0, 7] - 1e-4        # x0 above its upper bound
    _set_box(e, lb2, ub2, C)
    with pytest.raises(LcbaError) as ei:
        e.solve(ftol=1e-4)
    assert ei.value.code == -1
    cam = np.zeros((C, 11), bool)
    cam[0, 7] = True                         # held: its bound is ignored
    e.set_fixed(cam, None)
    res, _ = e.solve(ftol=1e-4)
    assert res.status > 0
    e.close()


def test_pysba_bounds_result(golden):
    """bundleAdjust(bounds=...) on the full layout: optimality is |g v|_inf of the trace, active_mask marks the bound
    entries, x stays in the box, a scalar pair and scipy.optimize.Bounds give the same solve."""
    from scipy.optimize import Bounds
    g = golden("ba_example18_vis60_800")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    lb, ub = _box(g)
    outs = []
    for b in ((lb, ub), Bounds(lb, ub)):
        sba = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
        res = sba.bundleAdjust(1e-4, verbose=0, bounds=b)
        assert np.all((res.x >= lb) & (res.x <= ub))
        assert res.optimality == sba.last_trace[-1]["optimality"]
        assert res.active_mask.shape == res.x.shape
        outs.append(res)
    assert np.array_equal(outs[0].x, outs[1].x) and np.array_equal(outs[0].active_mask, outs[1].active_mask)
    sba = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    res = sba.bundleAdjust(1e-4, verbose=0, bounds=(-np.inf, np.inf))
    sba2 = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    res2 = sba2.bundleAdjust(1e-4, verbose=0)
    assert np.array_equal(res.x, res2.x) and res.nfev == res2.nfev


def test_small_rigs_reach_every_candidate_against_oracle(Engine):
    """The small gauge-fixed ring4 rigs of test_bounds.py, where select_step takes the subspace step, the reflection
    and the anti-gradient: every solve against the oracle (nfev, njev, status, trace nfev, cost rtol 1e-9, every
    parameter within PARAM_RTOL, active_mask), and the three candidates taken over the set."""
    seen = set()
    for seed, kind in SMALL_RIGS:
        pb = make_rig("ring4", 60, seed=seed, variant="volume")
        C, P = pb["cams0"].shape[0], pb["pts0"].shape[0]
        cam, pt = _gauge(C, P)
        lb, ub = _binding_box(pb, C, P, kind)
        ora = trf_bounds_fixed(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], lb, ub,
                               cam_fixed=cam, pt_fixed=pt, ftol=1e-4)
        seen |= set(ora.choices)
        e = _engine(Engine, pb, cam, pt, (lb, ub))
        res, trace = e.solve(ftol=1e-4)
        x = _x(e)
        am = e.active_mask(1e-8)
        e.close()
        tag = (seed, kind)
        assert (res.nfev, res.njev, res.status) == (ora.nfev, ora.njev, ora.status), tag
        assert [r["nfev"] for r in trace] == [r["nfev"] for r in ora.rows], tag
        np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-9, err_msg=str(tag))
        errs = _param_errors(x, ora.x, C)
        assert max(errs.values()) <= PARAM_RTOL, (tag, errs)
        assert np.array_equal(am, ora.active_mask), tag
    assert seen == {"p", "r", "ag"}, seen


def test_debug_step_refuses_x_on_a_bound(Engine, golden):
    """lcba_debug_step needs x strictly inside the box (d = 0 on a bound): an x on a bound is LCBA_E_ARG."""
    from lasercalib_b200._cabi import LcbaError
    g = golden("ba_ring8_volume1500")
    C = g["cams0"].shape[0]
    lb, ub = _box(g)              # the lowest point's z lies on its bound
    e = _engine(Engine, g, box=(lb, ub))
    with pytest.raises(LcbaError) as ei:
        e.debug_step(1e-3, 0.0, 0)
    assert ei.value.code == -1
    lb[11 * C + 2::3] -= 1.0
    _set_box(e, lb, ub, C)
    pc, pp, _ = e.debug_step(1e-3, 0.0, 0)
    assert np.all(np.isfinite(pc)) and np.all(np.isfinite(pp))
    e.close()


def test_int8_route_with_binding_bounds_agrees_with_dmma(Engine, monkeypatch):
    """Ring24 x 150 k (the int8 Schur path's default size range), gauge mask, k1 / k2 within 1e-4 of x0 and every point
    at most 0.1 below its initial z: a whole bounded solve(ftol=1e-4) on the int8 route and on the DMMA route agree as
    in test_gpu_i8_scale (equal nfev and status, cost rtol 1e-10), x strictly inside on both, bounds binding.
    Measured on a B200 (1000 W): 15 evaluations on every route, 37 entries on a bound, int8 / DMMA / DFMA costs within
    3e-15.  A far narrower box (k1 / k2 within 1e-6, z within 1e-3: d -> 0 on the near-active entries) makes the
    trajectory itself sensitive to round-off: there the two FP64 routes DMMA and DFMA already differ by 4.0e-9 in the
    final cost, and int8 by 4.4e-9 from DMMA, so that box measures conditioning, not the route."""
    pb = make_rig("ring24", 150_000, seed=21, variant="volume", p_vis=1.0)
    C, P = pb["n_cams"], pb["n_points"]
    nc = 11 * C
    cam, pt = _gauge(C, P)
    free = ~_held(cam, pt)
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    lb, ub = np.full(x0.size, -np.inf), np.full(x0.size, np.inf)
    for a in (7, 8):
        lb[a:nc:11], ub[a:nc:11] = x0[a:nc:11] - 1e-4, x0[a:nc:11] + 1e-4
    lb[nc + 2::3] = x0[nc + 2::3] - 0.1
    out = {}
    for name, env in (("i8", {"LCBA_SCHUR_I8": "1"}), ("dmma", {"LCBA_SCHUR_I8": "0"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        e = _engine(Engine, pb, cam, pt, (lb, ub))
        r, _ = e.solve(ftol=1e-4)
        x = _x(e)
        active = int(np.count_nonzero(e.active_mask(1e-8)))
        fell_back = e.i8_fell_back()
        e.close()
        for k in env:
            monkeypatch.delenv(k)
        assert np.all((x[free] > lb[free]) & (x[free] < ub[free])), name
        assert active > 0, name
        out[name] = (r, fell_back)
    (a, fa), (b, _) = out["i8"], out["dmma"]
    assert fa is not None and fa >= 0          # the int8 route ran
    assert (a.nfev, a.status) == (b.nfev, b.status)
    np.testing.assert_allclose(a.cost, b.cost, rtol=1e-10)


def test_point_sharded_bounded_solve_matches_single_gpu():
    """Two GPUs (tests/_gpu_dist_bounds_worker.py): bounded points on both sides of the shard cut, binding camera
    bounds, the gauge mask; same nfev and status as one GPU, cost within 1e-12, x within 1e-9; different camera
    bounds over the ranks fail on every rank; a rank without bounds joins the bounded loop of the other."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(REPO, "tests", "_gpu_dist_bounds_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    for r in range(2):
        assert "rank %d ok" % r in out.stdout
