"""The long-double reference of tests/_ld_reference.py (CPU only): it agrees with the numpy FP64 oracle to FP64
round-off in the Jacobi-scaled space, its Jacobian agrees with the Richardson finite difference of the
reference's own residual, its rotation is right in every regime the kernels branch on, and its scaled
checker sees perturbations that the matrix-relative bounds of the older tests accept."""
import numpy as np
import pytest

import _ld_reference as L
from lasercalib_b200.synth import make_rig
from oracle import pysba_oracle as O

LAM = 1e-4


@pytest.fixture(autouse=True)
def _long_double():
    L.require_long_double()


def _oracle(cams, pts, uv, ci, pi, lam, w=None):
    """The numpy FP64 oracle's linearisation in the layout of L.linearize."""
    C, P = cams.shape[0], pts.shape[0]
    wcol = O.default_weights(pi) if w is None else np.asarray(w, float).reshape(-1, 1)
    f = O.fun(np.hstack((cams.ravel(), pts.ravel())), C, P, ci, pi, uv, wcol)
    _, Jc, Jp = O.jacobian_blocks(cams, pts, ci, pi, wcol)
    U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, C, P, ci, pi)
    sc = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
    sc[sc == 0] = 1
    S, rhs, _ = O.reduced_camera_system(U, gc, V, gp, W, ci, pi, lam, sc)
    return dict(S=S, rhs=rhs, grad=np.hstack((gc.ravel(), gp.ravel())), scale_inv=sc, cost=0.5 * f @ f, r=f,
                Jc=Jc, Jp=Jp)


def _problems():
    out = [("golden:" + g, None) for g in ("model_ring4_planar300", "ba_example18_vis60_800", "ba_ring8_volume1500")]
    out += [("ring4", (300, 1.0, 1e-6)), ("example18", (400, 0.6, 1e-3)), ("ring24", (300, 0.5, 1e-8)),
            ("ring24", (2000, 1.0, 1e-5))]
    return out


@pytest.mark.parametrize("name,spec", _problems(),
                         ids=[n if s is None else "%s-%d" % (n, s[0]) for n, s in _problems()])
def test_reference_matches_numpy_oracle(golden, name, spec):
    """The two restatements agree to FP64 round-off of the oracle, scaled: S <= 1e-14, Jc / Jp per column
    1e-14, scale_inv 1e-14, residual 1e-15 of its scale, cost 1e-16 of sum |r| rscale.  rhs and grad 3e-14:
    the oracle rounds each residual to a few u of its pixel scale, 1.5e3 times |f| here (rho), and that
    reaches g through J^T f as up to u rho s_i |f| = 1.7e-13; its random sum measures 1.8e-14 at most.
    Measured: S <= 5.1e-15, rhs <= 1.2e-14, grad <= 1.8e-14, Jc <= 2.2e-15, Jp <= 8e-16."""
    if spec is None:
        g = golden(name.split(":")[1])
        cams, pts, uv, ci, pi = g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"]
        lam = LAM
    else:
        n, pvis, lam = spec
        pb = make_rig(name, n, seed=1, variant="volume", p_vis=pvis)
        cams, pts, uv, ci, pi = pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"]
    ref = L.linearize(cams, pts, uv, ci, pi, lam)
    L.check("%s oracle vs long double" % name, _oracle(cams, pts, uv, ci, pi, lam), ref,
            dict(S=1e-14, rhs=3e-14, grad=3e-14, scale_inv=1e-14, r=1e-15, cost=1e-16, Jc=1e-14, Jp=1e-14), ci)


def test_jacobian_matches_richardson_truth(golden):
    """The analytic blocks against O.jacobian_truth_longdouble (Richardson-extrapolated central differences
    of the reference's fun in long double): on the golden ring4 truth and on a 4-camera rig re-expressed so
    that camera 0 has r = 0 exactly (the series branch) and then |r| = pi + 0.5.  Per (camera, column) the
    difference stays within 1e-9 of the column's largest entry, the accuracy of the difference quotient
    (measured <= 4.5e-11)."""
    g = golden("model_ring4_planar300")
    ci, pi = g["camera_ind"], g["point_ind"]
    ref = L.obs_blocks(g["cams0"], g["pts0"], ci, pi, g["points_2d"])
    ref["n_cams"] = g["cams0"].shape[0]
    Jt = g["J_truth_blocks"]
    L.check("golden ring4 Richardson truth", dict(Jc=Jt[:, :, :11], Jp=Jt[:, :, 11:]), ref, dict(Jc=1e-9, Jp=1e-9), ci)
    pb = make_rig("ring4", 12, seed=3, variant="volume")
    for r0 in (np.zeros(3), (np.pi + 0.5) * np.array([1.0, -2.0, 0.5]) / np.sqrt(5.25)):
        cams, pts = L.reframe(pb["cams0"], pb["pts0"], r0, b=(30.0, -20.0, 10.0))
        ci, pi, uv = pb["camera_ind"], pb["point_ind"], pb["points_2d"]
        C, P = cams.shape[0], pts.shape[0]
        J = O.jacobian_truth_longdouble(np.hstack((cams.ravel(), pts.ravel())), C, P, ci, pi, uv,
                                        O.default_weights(pi))
        rows = 2 * np.arange(ci.size)[:, None, None] + np.arange(2)[None, :, None]
        Jc = J[rows, 11 * ci[:, None, None] + np.arange(11)]
        Jp = J[rows, 11 * C + 3 * pi[:, None, None] + np.arange(3)]
        ref = L.obs_blocks(cams, pts, ci, pi, uv)
        ref["n_cams"] = C
        L.check("ring4 |r0| = %.3f Richardson truth" % np.linalg.norm(r0), dict(Jc=Jc, Jp=Jp), ref,
                dict(Jc=1e-9, Jp=1e-9), ci)


def test_rotation_regimes():
    """The series (t < 0.1, the branch point of model.cuh) and the closed form agree on both sides of
    t = 0.1 to 5e-17 relative, below FP64 round-off; R and J_r at r and at the equivalent vector
    r (1 - 2 pi / |r|), both in long double, describe the same rotation: R' = R to 1e-17 and
    J_r(r) = J_r(r') dr'/dr to 1e-16 (R(r') = R(r) for all r near, so -R [X]x J_r(r) = -R [X]x J_r(r') dr'/dr)."""
    for t in (0.1 * (1 - 1e-12), 0.1, 0.1 * (1 + 1e-12)):
        s = L.rodrigues_coeffs(t * t, "series")
        c = L.rodrigues_coeffs(t * t, "closed")
        for a, b in zip(s, c):
            assert abs(a - b) <= 5e-17 * abs(a), (t, a, b)
    axes = [np.array([0.0, 0.0, 1.0]), np.array([1.0, -2.0, 0.5]) / np.sqrt(5.25)]
    for ax in axes:
        for t in (0.3, 1.0, np.pi - 1e-9, np.pi, np.pi + 0.5, 5.0):
            r = (L.LD(t) * ax.astype(L.LD))
            t = np.sqrt((r * r).sum())
            rp = r * (1 - 2 * L.PI / t)
            R, Jr = L.rotation(r)
            Rp, Jrp = L.rotation(rp)
            M = (1 - 2 * L.PI / t) * np.eye(3, dtype=L.LD) + 2 * L.PI * np.outer(r, r) / t ** 3
            assert np.abs(R - Rp).max() <= 1e-17, (t, ax)
            assert np.abs(Jr - Jrp @ M).max() <= 1e-16 * np.abs(Jr).max(), (t, ax)
            assert np.abs(R @ R.T - np.eye(3)).max() <= 1e-18
    # the reference's row-wise rotate and the table form give the same rotation
    X = np.random.default_rng(0).normal(size=(5, 3)) * 100
    for t in (0.0, 1e-12, 0.05, 1.0, np.pi, np.pi + 0.5):
        r = t * axes[1]
        R, _ = L.rotation(r)
        got = L.rotate(X, np.tile(r, (5, 1)))
        assert np.abs(got - X.astype(L.LD) @ R.T).max() <= 1e-16 * np.abs(X).max(), t


def test_scaled_checker_sees_what_matrix_relative_bounds_accept():
    """A relative error of 1e-8 in one camera's (f, f) entry of S or its cx entry of rhs, or of 1e-9 in its
    focal column of Jc (1e-8 there exceeds the old bound: 5.6e-9 against 2.8e-9) passes the bounds the older tests assert (max|dS| <= 1e-11 max|S|, max|drhs| <= 1e-10 max|rhs|,
    |dJ| <= 1e-12 max|J|) and fails the scaled checks of the new ones (1e-13) by orders of magnitude."""
    pb = make_rig("ring24", 300, seed=1, variant="volume", p_vis=0.5)
    ci, pi = pb["camera_ind"], pb["point_ind"]
    ref = L.linearize(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi, 1e-8)
    base = L.to_f64(ref)
    base["Jc"] = ref["Jc"].astype(np.float64)
    c = 5
    f_row, cx_row = 11 * c + 6, 11 * c + 9
    Sr, rr, Jr = base["S"], base["rhs"], base["Jc"]
    S = Sr.copy()
    S[f_row, f_row] *= 1 + 1e-8
    rhs = rr.copy()
    rhs[cx_row] *= 1 + 1e-8
    Jc = Jr.copy()
    Jc[ci == c, :, 6] *= 1 + 1e-9
    assert np.abs(S - Sr).max() <= 1e-11 * np.abs(Sr).max()
    assert np.abs(rhs - rr).max() <= 1e-10 * np.abs(rr).max()
    assert np.abs(Jc - Jr).max() <= 1e-12 * np.abs(Jr).max()
    for key, val in (("S", S), ("rhs", rhs), ("Jc", Jc)):
        e = L.scaled_errors({key: val}, ref, ci)[key]
        print("perturbed %s: scaled error %.2e (bound 1e-13)" % (key, e))
        assert e > 1e-10, (key, e)
        with pytest.raises(AssertionError):
            L.check("perturbed " + key, {key: val}, ref, {key: 1e-13}, ci)
    # and the unperturbed FP64 rounding of the reference passes them
    L.check("rounded reference", dict(base), ref, dict(S=2e-16, rhs=2e-16, grad=2e-16, scale_inv=2e-16, Jc=2e-16), ci)


def test_long_double_guard(monkeypatch):
    """With fewer than 63 mantissa bits the reference skips instead of comparing double against double."""
    class Fake:
        nmant = 52
    monkeypatch.setattr(L.np, "finfo", lambda t: Fake)
    with pytest.raises(pytest.skip.Exception, match="mantissa bits"):
        L.require_long_double()
