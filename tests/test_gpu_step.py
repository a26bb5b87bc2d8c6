"""The step half of a solver iteration against plain FP64 / extended-precision references: the dense
camera solve (dense.cuh: k_copy_damped_rhs + k_chol_fused) at every size and grid it can run with,
and the whole Gauss-Newton step (point factors, reduced system, camera solve, back-substitution, Gram
sums, 2-D subspace scalars) against the numpy oracle on every pass route.  Errors measured on a B200
are written next to each bound; each run attaches its own to the test report (pytest
`record_property`: `-o junit_family=legacy --junitxml=...` writes them out)."""
import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve
from scipy.optimize._lsq.common import minimize_quadratic_1d, solve_trust_region_2d
from scipy.sparse import csr_matrix

from oracle import pysba_oracle as O
from lasercalib_b200.synth import make_rig

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
CH_NB = 32
# every n up to 70 (all panel remainders, one to three panels), every reduced system size of the
# solver (11 C full, 3 + 8 C shared intrinsics) and the top of the range
SIZES = sorted(set(range(1, 71)) | {11 * c for c in range(1, 65)} | {3 + 8 * c for c in range(1, 65)} | {703, 704})
# 1, 2, 3 CTAs (several panel rows per thread), the solver's own rule (0), and 148 CTAs: more than
# there are trailing tiles for every n here, so some CTAs have none
GRIDS = (1, 2, 3, 0, 148)


@pytest.fixture(scope="module")
def eng():
    from lasercalib_b200._cabi import Engine
    e = Engine()
    yield e
    e.close()


# ------------------------------------------------------------------------------ dense Cholesky
def _unpack(F, n):
    """(L, z) from the work buffer: strict lower L, 1 / l_jj on the diagonal, row n = z."""
    L = np.tril(F[:n], -1) + np.diag(1.0 / np.diag(F[:n]))
    return L, F[n]


def _solve_all_grids(eng, A, b, mu=0.0, d=None):
    """x, factor and fail word, asserted bit-identical over GRIDS and over a repeated call."""
    x0, F0, f0 = eng.debug_chol(A, b, mu, d, grid=GRIDS[0])
    for g in GRIDS[1:] + (GRIDS[0],):
        x, F, f = eng.debug_chol(A, b, mu, d, grid=g)
        assert f == f0, (g, f, f0)
        np.testing.assert_array_equal(x, x0, err_msg="grid %d" % g)
        np.testing.assert_array_equal(F, F0, err_msg="grid %d" % g)
    return x0, F0, f0


def _check_backward(A, b, x, L, record, tag):
    """Normwise backward error (residual in extended precision) and componentwise reconstruction."""
    n = A.shape[0]
    Al, xl = A.astype(np.longdouble), x.astype(np.longdouble)
    r = np.abs(Al @ xl - b.astype(np.longdouble)).max()
    bound = 10 * n * EPS * (np.abs(A).sum(axis=1).max() * np.abs(x).max() + np.abs(b).max())
    record("backward_" + tag, float(r / bound * 10 * n * EPS))
    assert r <= bound, (tag, float(r), float(bound))
    # |L L^T - A|_ij <= c n eps |L| |L^T|_ij <= c n eps sqrt(a_ii a_jj)
    dg = np.sqrt(np.abs(np.diag(A)))
    rec = np.abs(L @ L.T - A) / np.outer(dg, dg)
    record("reconstruct_" + tag, float(rec.max()))
    assert rec.max() <= 10 * n * EPS, (tag, rec.max())


def _spd(rng, n, cond):
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    A = (Q * np.logspace(0, -np.log10(cond), n)) @ Q.T
    return 0.5 * (A + A.T)


@pytest.mark.parametrize("n", SIZES)
def test_chol_matches_exact_and_fp64_references(eng, record_property, n):
    """Three matrix families, each on all GRIDS with bit-identical results:
    * exact: A = L0 L0^T with unit-diagonal L0 of entries in {-1, 0, 1} and b = A x0 with small
      integer x0.  Every intermediate of the factorisation and both substitutions is a small
      integer, so the kernel must return L0, z = L0^T x0 and x0 EXACTLY;
    * random SPD of condition 1e2 and 1e8 (spectrum log-spaced): backward error
      |A x - b| <= 10 n eps (|A| |x| + |b|) (residual in extended precision), reconstruction
      |L L^T - A|_ij <= 10 n eps sqrt(a_ii a_jj), forward error |x - x0| / |x0| <= 10 n eps cond;
    * graded SPD of condition ~1e13: D M D with cond(M) = 10 and D spanning 10^6.5 (Cholesky does
      not see diagonal scaling): the same bounds, the forward error in the scaled variable D x.
    Measured on a B200 (1000 W): the exact family exact at every size; normwise backward error
    <= 1.3e-16, reconstruction <= 2.7e-15, forward error <= 0.02 of its bound."""
    rng = np.random.default_rng(n)
    L0 = np.tril(rng.integers(-1, 2, (n, n)).astype(np.float64), -1) + np.eye(n)
    A = L0 @ L0.T
    x0 = rng.integers(-4, 5, n).astype(np.float64)
    b = A @ x0
    x, F, fail = _solve_all_grids(eng, A, b)
    assert fail == 0
    np.testing.assert_array_equal(x, x0)
    np.testing.assert_array_equal(np.tril(F[:n], -1), np.tril(L0, -1))
    np.testing.assert_array_equal(np.diag(F[:n]), np.ones(n))
    np.testing.assert_array_equal(F[n], L0.T @ x0)
    np.testing.assert_array_equal(np.triu(F[:n], 1), np.triu(A, 1))         # upper triangle untouched
    for cond in (1e2, 1e8):
        A = _spd(rng, n, cond)
        x0 = rng.standard_normal(n)
        b = A @ x0
        x, F, fail = _solve_all_grids(eng, A, b)
        assert fail == 0, cond
        L, _ = _unpack(F, n)
        _check_backward(A, b, x, L, record_property, "cond%.0e" % cond)
        fwd = np.abs(x - x0).max() / np.abs(x0).max()
        record_property("forward_cond%.0e" % cond, float(fwd / (10 * n * EPS * cond)))
        assert fwd <= 10 * n * EPS * cond, (cond, fwd)
    D = 10.0 ** rng.permutation(np.linspace(0, 6.5, n))
    A = _spd(rng, n, 10.0) * np.outer(D, D)
    x0 = rng.standard_normal(n) / D
    b = A @ x0
    x, F, fail = _solve_all_grids(eng, A, b)
    assert fail == 0
    L, _ = _unpack(F, n)
    _check_backward(A, b, x, L, record_property, "graded")
    fwd = np.abs(D * (x - x0)).max() / np.abs(D * x0).max()
    record_property("forward_graded", float(fwd / (10 * n * EPS * 10.0)))
    assert fwd <= 10 * n * EPS * 10.0, fwd


def _first_cameras(pb, C, min_views=3):
    """The problem restricted to its first C cameras (points with too few views left dropped)."""
    keep = pb["camera_ind"] < C
    ci, pi, uv = pb["camera_ind"][keep], pb["point_ind"][keep], pb["points_2d"][keep]
    cnt = np.bincount(pi, minlength=pb["pts0"].shape[0])
    good = cnt >= min_views
    sel = good[pi]
    remap = np.cumsum(good) - 1
    return dict(cams0=pb["cams0"][:C].copy(), pts0=pb["pts0"][good].copy(), points_2d=uv[sel].copy(),
                camera_ind=ci[sel].copy(), point_ind=remap[pi[sel]].copy())


@pytest.mark.parametrize("rig,npts,pvis", [("ring64", 200, 0.5), ("ring24", 300, 0.6), ("example18", 400, 0.6)])
def test_chol_on_real_reduced_systems(eng, record_property, rig, npts, pvis):
    """S from the solver's own linearisation at lam = 1e-8 (gauge modes: nearly singular without the
    damping), d = the camera scaling, mu over the retry schedule of lcba_solve.  Against
    scipy.linalg.cho_solve in the Jacobi-scaled variable within 10 n eps cond(D^-1 S D^-1); backward
    error and reconstruction as above; bit-identical over GRIDS.  Measured on a B200 (1000 W):
    forward error <= 2.3e-4 of its bound, reconstruction <= 1.3e-15."""
    pb = make_rig(rig, npts, seed=1, variant="volume", p_vis=pvis)
    from lasercalib_b200._cabi import Engine
    e = Engine()
    e.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    out = e.linearize(1e-8)
    e.close()
    S, rhs = out["S"], out["rhs"]
    n = S.shape[0]
    d = out["scale_inv"][:n]
    for mu in [0.0] + [10.0 ** k for k in range(-13, -2)]:
        A = S + np.diag(mu * d * d)
        x, F, fail = _solve_all_grids(eng, S, rhs, mu, d)
        assert fail == 0, mu
        L, _ = _unpack(F, n)
        _check_backward(A, rhs, x, L, record_property, "mu%.0e" % mu)
        As = A / np.outer(d, d)
        kappa = np.linalg.cond(As)
        xr = cho_solve(cho_factor(A, lower=True), rhs)
        fwd = np.abs(d * (x - xr)).max() / np.abs(d * xr).max()
        record_property("forward_mu%.0e" % mu, float(fwd / (10 * n * EPS * kappa)))
        assert fwd <= 10 * n * EPS * kappa, (mu, fwd, kappa)


@pytest.mark.parametrize("n", [1, 32, 67, 264, 701, 704])
def test_chol_breakdown_raises_the_fail_bit(eng, n):
    """A zero or negative pivot at column 0, 31, 32, the first column of the last panel and n - 1, and a
    NaN in the lower triangle: bit 0 of the fail word on every grid; bit 1 (barrier timeout) never."""
    rng = np.random.default_rng(n)
    L0 = np.tril(rng.integers(-1, 2, (n, n)).astype(np.float64), -1) + np.eye(n)
    A0 = L0 @ L0.T
    b = rng.standard_normal(n)
    cols = sorted({j for j in (0, 31, 32, CH_NB * ((n - 1) // CH_NB), n - 1) if j < n})
    cases = []
    for j in cols:
        for drop in (1.0, 2.0):                 # exact pivot 1 -> 0 (zero) or -1 (negative)
            A = A0.copy()
            A[j, j] -= drop
            cases.append(A)
    A = A0.copy()
    A[n - 1, n // 2] = np.nan                   # (n-1, n//2) is on or below the diagonal
    cases.append(A)
    for A in cases:
        for g in GRIDS:
            _, _, fail = eng.debug_chol(A, b, grid=g)
            assert fail == 1, (g, fail)


def test_chol_rejects_bad_arguments(eng):
    from lasercalib_b200._cabi import LcbaError
    A = np.eye(4)
    for n in (0, 705):
        with pytest.raises(LcbaError) as ei:
            eng.debug_chol(np.eye(n), np.ones(n))
        assert ei.value.code == -1
    for g in (-1, 1 << 20):
        with pytest.raises(LcbaError) as ei:
            eng.debug_chol(A, np.ones(4), grid=g)
        assert ei.value.code == -1
    with pytest.raises(LcbaError):
        eng.debug_chol(A, np.ones(4), mu=1.0, d=None)            # damping without d


def test_chol_small_grid_covers_every_panel_row(eng):
    """n = 704 on one CTA: 673 panel rows of the first panel for 256 threads.  Every row must be
    solved (the kernel once handled only 256 G of them: a wrong factor on 1 and 2 CTAs)."""
    n = 704
    rng = np.random.default_rng(7)
    L0 = np.tril(rng.integers(-1, 2, (n, n)).astype(np.float64), -1) + np.eye(n)
    x0 = rng.integers(-4, 5, n).astype(np.float64)
    A = L0 @ L0.T
    x, F, fail = eng.debug_chol(A, A @ x0, grid=1)
    assert fail == 0
    np.testing.assert_array_equal(np.tril(F[:n], -1), np.tril(L0, -1))
    np.testing.assert_array_equal(x, x0)


# ------------------------------------------------------------------------------ Gauss-Newton step
def _problem(C, seed, weights_zero=True, shuffle=False, repeat=False):
    """Cameras 0..C-1 of ring24 / ring64 (dense: the tensor-path passes for C >= 8), weights with
    exact zeros, one point reduced to two views, one point without observations."""
    base = make_rig("ring64" if C > 24 else "ring24", 120 if C > 24 else 160, seed=seed, variant="volume", p_vis=0.93)
    pb = _first_cameras(base, C)
    ci, pi, uv = pb["camera_ind"], pb["point_ind"], pb["points_2d"]
    P = pb["pts0"].shape[0]
    two = np.flatnonzero(pi == 1)[2:]           # point 1 keeps its first two views
    keep = np.ones(ci.size, bool)
    keep[two] = False
    ci, pi, uv = ci[keep], pi[keep], uv[keep]
    pts = np.vstack([pb["pts0"], pb["pts0"][:1] + 10.0])   # point P: no observation
    rng = np.random.default_rng(seed)
    if repeat:
        extra = rng.choice(ci.size, ci.size // 10, replace=False)
        ci, pi = np.concatenate([ci, ci[extra]]), np.concatenate([pi, pi[extra]])
        uv = np.concatenate([uv, uv[extra] + rng.normal(0, 0.3, (extra.size, 2))])
    w = rng.uniform(0.5, 2.0, ci.size)
    if weights_zero:
        w[rng.random(ci.size) < 0.05] = 0.0
    out = dict(cams0=pb["cams0"], pts0=pts, points_2d=uv, camera_ind=ci, point_ind=pi, n_obs=ci.size, w=w)
    if shuffle:
        perm = np.random.default_rng(seed + 1).permutation(ci.size)
        out.update(points_2d=uv[perm], camera_ind=ci[perm], point_ind=pi[perm], w=w[perm])
    assert out["pts0"].shape[0] == P + 1
    return out


def _jacobian(pb, mode):
    """(J (CSR), f, x) of the parameterisation of `mode` at x0: 0 = [cams | points], 1 = points,
    2 = the shared-intrinsics vector [f k1 k2 | extrinsics | centres | points] (J_red = J_full T)."""
    cams, pts, ci, pi, w = pb["cams0"], pb["pts0"], pb["camera_ind"], pb["point_ind"], pb["w"]
    C, P = cams.shape[0], pts.shape[0]
    x = np.hstack((cams.ravel(), pts.ravel()))
    f = O.fun(x, C, P, ci, pi, pb["points_2d"], w.reshape(-1, 1))
    _, Jc, Jp = O.jacobian_blocks(cams, pts, ci, pi, w)
    if mode == 2:
        A = O.sparsity_sharedcam(C, P, ci, pi)
        data = np.concatenate([Jc[:, :, 6:9], Jc[:, :, 0:6], Jc[:, :, 9:11], Jp], axis=2).reshape(-1)
        return csr_matrix((data, A.indices, A.indptr), shape=A.shape), f, O.sharedcam_pack(cams, pts)
    J = O.jacobian_csr(Jc, Jp, C, P, ci, pi)
    if mode == 1:
        return J[:, 11 * C:].tocsr(), f, pts.ravel().copy()
    return J, f, x


def _gpu_step(pb, lam, mode, env, monkeypatch):
    from lasercalib_b200._cabi import Engine
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    e = Engine()
    e.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], pb["w"])
    pc, pp, sc = e.debug_step(lam, 0.0, mode)
    e.close()
    for k in env:
        monkeypatch.delenv(k)
    return pc, pp, sc


def _reduce_gpu_p(pb, pc, pp, mode):
    C = pb["cams0"].shape[0]
    if mode == 1:
        assert np.all(pc == 0.0)
        return pp
    if mode == 2:
        c = pc.reshape(C, 11)
        assert np.all(c[:, 6:9] == c[0, 6:9])                  # the shared step, replicated
        return np.hstack((c[0, 6:9], c[:, :6].ravel(), c[:, 9:].ravel(), pp))
    return np.hstack((pc, pp))


def _check_step(J, f, x, lam, p_or, p, sc, record, tag):
    """The GPU step p and scalars sc against the damped normal equations of J."""
    g = J.T @ f
    s = np.sqrt(np.asarray(J.multiply(J).sum(axis=0)).ravel())
    s[s == 0] = 1.0
    d = 1.0 / s
    # damped normal equations (J^T J + lam D^2) p = g at the GPU's p, normalised in the scaled space
    Jp = J @ p
    r = (J.T @ Jp + lam * s * s * p - g) * d
    Ja = abs(J)
    den = ((Ja.T @ (Ja @ np.abs(p)) + lam * s * s * np.abs(p)) * d).max() + np.abs(g * d).max()
    res = np.abs(r).max() / den
    record("residual_" + tag, float(res))
    assert res <= 1e-11, (tag, res)
    # forward error within 1e-11 x the condition number of the Jacobi-scaled system
    H = (J.T @ J).toarray() + np.diag(lam * s * s)
    kappa = np.linalg.cond(H * np.outer(d, d))
    fwd = np.abs(s * (p - p_or)).max() / np.abs(s * p_or).max()
    record("forward_" + tag, float(fwd / kappa))
    assert fwd <= 1e-11 * kappa, (tag, fwd, kappa)
    # Delta, Jg2 and the Cauchy reg_term (trf.py:488-492)
    g_h = d * g
    Jg = J @ (d * g_h)
    Delta = np.linalg.norm(x * s)
    reg = -minimize_quadratic_1d(0.5 * Jg @ Jg, -g_h @ g_h, 0, Delta / np.linalg.norm(g_h))[1] / Delta ** 2
    np.testing.assert_allclose(sc["Delta"], Delta, rtol=1e-12, err_msg=tag)
    np.testing.assert_allclose(sc["Jg2"], Jg @ Jg, rtol=1e-11, err_msg=tag)
    np.testing.assert_allclose(sc["reg_term"], reg, rtol=1e-11, err_msg=tag)
    # the nine Gram totals of k_ctl_sub (trf_exact, oracle/pysba_oracle.py:402-427) at the GPU's p
    a, bh, gt = g_h, p * s, d * g_h
    tot = dict(aa=a @ a, ab=a @ bh, bb=bh @ bh, JAA=Jg @ Jg, JAB=Jg @ Jp, JBB=Jp @ Jp, gtgt=gt @ gt, gtp=gt @ p, pp=p @ p)
    norm = dict(ab=np.sqrt(tot["aa"] * tot["bb"]), JAB=np.sqrt(tot["JAA"] * tot["JBB"]), gtp=np.sqrt(tot["gtgt"] * tot["pp"]))
    worst = 0.0
    for k, v in tot.items():
        err = abs(sc[k] - v) / norm.get(k, abs(v))
        worst = max(worst, err)
        assert err <= 1e-12, (tag, k, sc[k], v)
    record("gram_" + tag, float(worst))
    # the 2-D subspace problem on the oracle's step (basis-sign independent quantities only)
    from scipy.linalg import qr
    Sq, _ = qr(np.vstack((g_h, p_or * s)).T, mode="economic")
    JS = np.stack([J @ (d * Sq[:, 0]), J @ (d * Sq[:, 1])], axis=1)
    B_S, g_S = JS.T @ JS, Sq.T @ g_h
    p_S, _ = solve_trust_region_2d(B_S, g_S, Delta)
    Js = JS @ p_S
    pred = -(0.5 * Js @ Js + g_S @ p_S)
    tol = max(1e-10, 1e-11 * kappa)
    errs = [abs(sc["predicted"] - pred) / abs(pred), abs(sc["step_h_norm"] - np.linalg.norm(p_S)) / np.linalg.norm(p_S),
            abs(sc["step_norm"] - np.linalg.norm(d * (Sq @ p_S))) / np.linalg.norm(d * (Sq @ p_S))]
    record("subspace_" + tag, float(max(errs)))
    assert max(errs) <= tol, (tag, errs, tol)
    assert sc["chol_fail"] == 0.0
    return kappa


ROUTES = {"pt": {}, "generic": {"LCBA_PT_PASSES": "0"}}


@pytest.mark.parametrize("lam", [1e-3, 1e-6])
@pytest.mark.parametrize("C", [3, 8, 13, 24, 29, 64])
def test_step_matches_oracle_on_every_pass_route(monkeypatch, record_property, C, lam):
    """Full step (mode 0) against O.solve_damped_normal_equations on the point-parallel passes
    (k_jdot_pt / k_backsub_pt, default) and the generic ones (k_jdot / k_backsub, LCBA_PT_PASSES=0).
    Weighted with exact zeros, a two-view point, a point without observations
    (its step is exactly 0); C = 13 and 29 shuffled.  Bounds: normal-equation residual 1e-11,
    forward error 1e-11 cond, reg_term / Jg2 1e-11, Gram totals 1e-12, subspace scalars
    max(1e-10, 1e-11 cond); the camera step is bit-identical over the routes (same reduced system),
    the point steps agree to 1e-13 scaled.  Measured on a B200 (1000 W): residual <= 2.3e-14,
    forward error <= 7.4e-15 cond, Gram totals <= 3.5e-14, subspace scalars <= 2.1e-9, point
    steps over the routes <= 7.1e-16."""
    pb = _problem(C, seed=C, shuffle=C in (13, 29))
    ci, pi, w = pb["camera_ind"], pb["point_ind"], pb["w"]
    Cn, P = pb["cams0"].shape[0], pb["pts0"].shape[0]
    J, f, x = _jacobian(pb, 0)
    _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
    U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, Cn, P, ci, pi)
    s = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
    s[s == 0] = 1.0
    p_or, _, _ = O.solve_damped_normal_equations(U, gc, V, gp, W, ci, pi, lam, s)
    steps = {}
    for route, env in ROUTES.items():
        pc, pp, sc = _gpu_step(pb, lam, 0, env, monkeypatch)
        assert np.all(pp[-3:] == 0.0), route                     # the point without observations
        p = _reduce_gpu_p(pb, pc, pp, 0)
        _check_step(J, f, x, lam, p_or, p, sc, record_property, route)
        steps[route] = (pc, pp, s[11 * Cn:])
    pc0, pp0, sp = steps["pt"]
    for route, (pc, pp, _) in steps.items():
        np.testing.assert_array_equal(pc, pc0, err_msg=route)
        d = np.abs(sp * (pp - pp0)).max() / np.abs(sp * pp0).max()
        record_property("routes_" + route, float(d))
        assert d <= 1e-13, (route, d)


def test_step_with_repeated_pairs_matches_oracle(monkeypatch, record_property):
    """Observations that repeat a (camera, point) pair force the generic passes (k_jdot / k_backsub
    with the distinct-pair view of the Schur side).  Same bounds as above.  Measured on a B200
    (1000 W): residual <= 1.6e-14, Gram totals <= 1.3e-14, subspace scalars <= 1.4e-11."""
    for lam in (1e-3, 1e-6):
        pb = _problem(8, seed=5, repeat=True)
        J, f, x = _jacobian(pb, 0)
        ci, pi, w = pb["camera_ind"], pb["point_ind"], pb["w"]
        Cn, P = pb["cams0"].shape[0], pb["pts0"].shape[0]
        _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
        U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, Cn, P, ci, pi)
        s = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
        s[s == 0] = 1.0
        p_or, _, _ = O.solve_damped_normal_equations(U, gc, V, gp, W, ci, pi, lam, s)
        pc, pp, sc = _gpu_step(pb, lam, 0, {}, monkeypatch)
        assert np.all(pp[-3:] == 0.0)
        _check_step(J, f, x, lam, p_or, _reduce_gpu_p(pb, pc, pp, 0), sc, record_property, "repeat%.0e" % lam)


@pytest.mark.parametrize("lam", [1e-3, 1e-6])
@pytest.mark.parametrize("C", [8, 24])
def test_step_fixed_cameras_matches_oracle(monkeypatch, record_property, C, lam):
    """Mode 1 (fix_cameras, PySBA.bundleAdjust_nocam): p = (V + lam Dp^2)^-1 g_p per point as in
    O.trf_exact_nocam; the camera step is exactly zero.  Same bounds as the full step.  Measured on a
    B200 (1000 W): residual <= 1.3e-14, Gram totals <= 1.6e-14, subspace scalars <= 1.7e-14."""
    pb = _problem(C, seed=40 + C)
    J, f, x = _jacobian(pb, 1)
    pi, P = pb["point_ind"], pb["pts0"].shape[0]
    _, _, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], pb["camera_ind"], pi, pb["w"])
    V = np.zeros((P, 3, 3))
    gp = np.zeros((P, 3))
    np.add.at(V, pi, np.einsum("nia,nib->nab", Jp, Jp))
    np.add.at(gp, pi, np.einsum("nia,ni->na", Jp, f.reshape(-1, 2)))
    s = np.sqrt(np.einsum("paa->pa", V)).ravel()
    s[s == 0] = 1.0
    Vd = V.copy()
    Vd[:, np.arange(3), np.arange(3)] += lam * s.reshape(P, 3) ** 2
    p_or = np.linalg.solve(Vd, gp[:, :, None])[:, :, 0].ravel()
    pc, pp, sc = _gpu_step(pb, lam, 1, {}, monkeypatch)
    assert np.all(pp[-3:] == 0.0)
    _check_step(J, f, x, lam, p_or, _reduce_gpu_p(pb, pc, pp, 1), sc, record_property, "nocam")


@pytest.mark.parametrize("C", [3, 8, 24])
def test_step_shared_intrinsics_matches_oracle(monkeypatch, record_property, C):
    """Mode 2 (shared intrinsics, PySBA.bundleAdjust_sharedcam): k_assemble_S_shared, the dense
    solve at n = 3 + 8 C, k_expand_shared and the back-substitution against the dense damped normal
    equations of J_full T (O.trf_exact_sharedcam's Jacobian).  Same bounds as the full step.
    Measured on a B200 (1000 W): residual <= 7.2e-16, Gram totals <= 2.3e-15, subspace scalars
    <= 1.8e-10."""
    pb = _problem(C, seed=60 + C)
    pb["cams0"] = pb["cams0"].copy()
    pb["cams0"][:, 6:9] = pb["cams0"][:, 6:9].mean(axis=0)
    for lam in (1e-3, 1e-6):
        J, f, x = _jacobian(pb, 2)
        s = np.sqrt(np.asarray(J.multiply(J).sum(axis=0)).ravel())
        s[s == 0] = 1.0
        H = (J.T @ J).toarray() + np.diag(lam * s * s)
        p_or = cho_solve(cho_factor(H, lower=True), J.T @ f)
        pc, pp, sc = _gpu_step(pb, lam, 2, {}, monkeypatch)
        assert np.all(pp[-3:] == 0.0)
        _check_step(J, f, x, lam, p_or, _reduce_gpu_p(pb, pc, pp, 2), sc, record_property, "shared%.0e" % lam)
