"""GPU parity tests: the CUDA engine (through the C-ABI / the PySBA drop-in) against the CPU
oracle and the golden fixtures made from the unmodified reference.  Tolerances follow the
protocol of SURVEY.md App. C.4 (P1-P5) and are written next to every assertion."""
import io
import pickle
from contextlib import redirect_stdout

import numpy as np
import pytest

from oracle import pysba_oracle as O
from lasercalib_b200.synth import make_rig, shuffle_observations

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def PySBA():
    from lasercalib_b200.pySBA import PySBA as cls
    return cls


@pytest.fixture(scope="module")
def Engine():
    from lasercalib_b200._cabi import Engine as cls
    return cls


def _x0(g):
    return np.hstack((g["cams0"].ravel(), g["pts0"].ravel()))


def _sba(PySBA, g, weights=None):
    return PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"],
                 g["point_ind"], pointWeights=weights)


# ----------------------------------------------------------------------------- P1 model
def test_project_rotate_match_reference_outputs(PySBA, golden):
    g = golden("model_example17")
    M = int(g["cam_rows_per_point"])
    rows = np.repeat(g["cams"], M, axis=0)
    sba = PySBA(g["cams"], g["pts"], np.zeros((1, 2)), np.zeros(1, dtype=int), np.zeros(1, dtype=int))
    proj = sba.project(g["pts"], rows)
    # P1: 1e-9 * max(1, |proj|)
    assert np.all(np.abs(proj - g["proj"]) <= 1e-9 * np.maximum(1.0, np.abs(g["proj"])))
    np.testing.assert_allclose(sba.rotate(g["pts"], rows[:, :3]), g["rot"], rtol=0, atol=1e-11)
    r = sba.rotate(g["pts"][:6], g["rv_small"])
    assert np.all(np.isfinite(r))
    np.testing.assert_array_equal(r[0], g["pts"][0])            # theta = 0 => identity
    np.testing.assert_allclose(r, g["rot_small"], rtol=0, atol=1e-11)
    np.testing.assert_allclose(sba.project(g["pts"][:6], g["cam_small"]), g["proj_small"],
                               rtol=0, atol=1e-9)
    # inputs untouched, empty input ok
    assert sba.project(np.zeros((0, 3)), np.zeros((0, 11))).shape == (0, 2)


def test_fun_matches_reference(PySBA, golden):
    g = golden("model_ring4_planar300")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    sba = _sba(PySBA, g)
    assert sba.pointWeights.dtype == np.int64 and sba.pointWeights.shape == (g["point_ind"].size, 1)
    f = sba.fun(_x0(g), C, P, g["camera_ind"], g["point_ind"], g["points_2d"], sba.pointWeights)
    assert f.shape == g["f0"].shape
    proj_mag = np.maximum(1.0, np.abs(np.repeat(g["proj"], 1, axis=0)).ravel())
    assert np.all(np.abs(f - g["f0"]) <= 1e-9 * proj_mag)        # P1
    # float weights
    sw = _sba(PySBA, g, weights=g["weights"])
    fw = sw.fun(_x0(g), C, P, g["camera_ind"], g["point_ind"], g["points_2d"], sw.pointWeights)
    assert np.all(np.abs(fw - g["f0_w"]) <= 2e-9 * proj_mag)
    # another parameter vector through the same resident problem
    x1 = _x0(g) * (1 + 1e-4)
    f1 = sba.fun(x1, C, P, g["camera_ind"], g["point_ind"], g["points_2d"], sba.pointWeights)
    ref1 = O.fun(x1, C, P, g["camera_ind"], g["point_ind"], g["points_2d"], sba.pointWeights)
    np.testing.assert_allclose(f1, ref1, rtol=0, atol=1e-8)


def test_fun_sees_in_place_edits_of_the_observations(PySBA):
    pb = make_rig("ring4", 200, seed=1)
    C, P = pb["n_cams"], pb["n_points"]
    p2 = pb["points_2d"].copy()
    sba = PySBA(pb["cams0"], pb["pts0"], p2, pb["camera_ind"], pb["point_ind"])
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    f0 = sba.fun(x0, C, P, pb["camera_ind"], pb["point_ind"], p2, sba.pointWeights)
    p2 += 1.0                                        # same buffer, new content
    f1 = sba.fun(x0, C, P, pb["camera_ind"], pb["point_ind"], p2, sba.pointWeights)
    np.testing.assert_allclose(f1, f0 - 1.0, atol=1e-9)


def test_sparse_in_place_edits_are_never_served_stale(PySBA):
    """The reference re-reads its arrays on every call (pySBA.py:92-101, :132-147).  One edited
    observation in the middle of points2D and one edited weight must show up in `fun` and in
    `bundleAdjust`; with `observations_static = True` the caller promises no such edits and
    `invalidate()` is the explicit way to announce one."""
    pb = make_rig("ring8", 600, seed=2, variant="volume", p_vis=0.9)
    C, P, N = pb["n_cams"], pb["n_points"], pb["n_obs"]
    p2 = pb["points_2d"].copy()
    w = np.ones(N)
    sba = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), p2, pb["camera_ind"], pb["point_ind"], pointWeights=w)
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    f0 = sba.fun(x0, C, P, pb["camera_ind"], pb["point_ind"], p2, sba.pointWeights)
    mid = N // 2 + 7
    p2[mid, 1] += 40.0                                 # one outlier pixel coordinate
    f1 = sba.fun(x0, C, P, pb["camera_ind"], pb["point_ind"], p2, sba.pointWeights)
    d = f1 - f0
    assert abs(d[2 * mid + 1] + 40.0) < 1e-9 and np.count_nonzero(d) == 1
    w[mid] = 0.0                                       # ... down-weighted in place
    f2 = sba.fun(x0, C, P, pb["camera_ind"], pb["point_ind"], p2, sba.pointWeights)
    assert f2[2 * mid] == 0.0 and f2[2 * mid + 1] == 0.0
    np.testing.assert_array_equal(np.delete(f2, [2 * mid, 2 * mid + 1]), np.delete(f0, [2 * mid, 2 * mid + 1]))
    # bundleAdjust sees the same edits: outlier active -> higher cost than outlier removed
    w[mid] = 1.0
    r_out = sba.bundleAdjust(1e-4, verbose=0)
    sba.cameraArray, sba.points3D = pb["cams0"].copy(), pb["pts0"].copy()
    w[mid] = 0.0
    r_in = sba.bundleAdjust(1e-4, verbose=0)
    ora = O.trf_exact(pb["cams0"], pb["pts0"], p2, pb["camera_ind"], pb["point_ind"], weights=w, ftol=1e-4)
    np.testing.assert_allclose(r_in.cost, ora.cost, rtol=1e-8)
    assert r_out.cost > r_in.cost + 100.0
    # opt-in residency: the device copy is kept for the same array objects until invalidate()
    sba.observations_static = True
    sba.cameraArray, sba.points3D = pb["cams0"].copy(), pb["pts0"].copy()
    a = sba.bundleAdjust(1e-4, verbose=0)
    sba.cameraArray, sba.points3D = pb["cams0"].copy(), pb["pts0"].copy()
    b = sba.bundleAdjust(1e-4, verbose=0)
    assert not sba._fresh_problem and b.cost == a.cost
    w[mid] = 1.0
    sba.invalidate()
    sba.cameraArray, sba.points3D = pb["cams0"].copy(), pb["pts0"].copy()
    c = sba.bundleAdjust(1e-4, verbose=0)
    assert sba._fresh_problem
    np.testing.assert_allclose(c.cost, r_out.cost, rtol=1e-12)


def test_lazy_result_members_survive_engine_reuse(PySBA):
    """res.fun / res.grad / res.jac are produced on first access from the shared per-device
    engine; if another solve (another PySBA object) used the engine in between they must still
    be THIS result's residuals, gradient and Jacobian."""
    pa = make_rig("ring8", 300, seed=4, variant="volume", p_vis=0.9)
    pb = make_rig("ring4", 500, seed=5)
    sa = PySBA(pa["cams0"].copy(), pa["pts0"].copy(), pa["points_2d"], pa["camera_ind"], pa["point_ind"])
    ra = sa.bundleAdjust(1e-4, verbose=0)
    sb = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    rb = sb.bundleAdjust(1e-4, verbose=0)               # the engine now holds problem b
    assert "fun" in ra and "jac" in ra.keys()
    fa = ra.fun
    assert fa.shape == (2 * pa["n_obs"],)
    np.testing.assert_allclose(0.5 * fa @ fa, ra.cost, rtol=1e-12)
    w = O.default_weights(pa["point_ind"])
    np.testing.assert_allclose(fa, O.fun(ra.x, pa["n_cams"], pa["n_points"], pa["camera_ind"], pa["point_ind"],
                                         pa["points_2d"], w), atol=1e-8)
    fb = rb.fun                                          # and b's members after a's restore
    np.testing.assert_allclose(0.5 * fb @ fb, rb.cost, rtol=1e-12)
    ga = ra.grad
    np.testing.assert_allclose(ra.jac.T @ fa, ga, rtol=0, atol=1e-9 * np.abs(ga).max())
    assert abs(ra.optimality - np.abs(ga).max()) <= 1e-9 * ra.optimality


def test_repeated_camera_point_rows_are_accepted(PySBA, Engine):
    """Rows that repeat a (camera, point) pair are one more residual pair each in the reference
    (its 3-dataset concatenation makes them, calibrate_camera.py:41-44; SURVEY 8f rank 2).
    Dense rig -> tensor-path Schur; sparse rig -> DFMA Schur; weighted and unweighted."""
    for rig, npts, pvis in (("ring8", 500, 0.95), ("example18", 500, 0.5)):
        pb = make_rig(rig, npts, seed=9, variant="volume", p_vis=pvis)
        rng = np.random.default_rng(1)
        extra = rng.choice(pb["n_obs"], 150, replace=False)
        extra = np.concatenate([extra, extra[:40]])      # some pairs three times
        ci = np.concatenate([pb["camera_ind"], pb["camera_ind"][extra]])
        pi = np.concatenate([pb["point_ind"], pb["point_ind"][extra]])
        uv = np.concatenate([pb["points_2d"], pb["points_2d"][extra] + rng.normal(0, 0.3, (extra.size, 2))])
        for w in (None, rng.uniform(0.5, 2.0, ci.size)):
            C, P = pb["n_cams"], pb["n_points"]
            wcol = O.default_weights(pi) if w is None else w.reshape(-1, 1)
            x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
            f = O.fun(x0, C, P, ci, pi, uv, wcol)
            _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
            U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, C, P, ci, pi)
            sc = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
            S_or, rhs_or, _ = O.reduced_camera_system(U, gc, V, gp, W, ci, pi, 1e-4, sc)
            eng = Engine()
            eng.set_problem(pb["cams0"], pb["pts0"], uv, ci, pi, w)
            out = eng.linearize(1e-4)
            r, cost = eng.residuals()
            eng.close()
            np.testing.assert_allclose(r, f, atol=1e-8)
            np.testing.assert_allclose(cost, 0.5 * f @ f, rtol=1e-12)
            assert np.abs(out["S"] - S_or).max() <= 1e-11 * np.abs(S_or).max()
            assert np.abs(out["rhs"] - rhs_or).max() <= 1e-10 * np.abs(rhs_or).max()
        sba = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), uv, ci, pi)
        res = sba.bundleAdjust(1e-4, verbose=0)
        ora = O.trf_exact(pb["cams0"], pb["pts0"], uv, ci, pi, ftol=1e-4)
        assert res.nfev == ora.nfev and res.status == ora.status
        np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-8)


def test_fun_on_shuffled_observations(PySBA):
    pb = make_rig("example18", 600, seed=3, variant="volume", p_vis=0.7)
    sh = shuffle_observations(pb, seed=5)
    C, P = pb["n_cams"], pb["n_points"]
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    w = O.default_weights(sh["point_ind"])
    ref = O.fun(x0, C, P, sh["camera_ind"], sh["point_ind"], sh["points_2d"], w)
    sba = PySBA(pb["cams0"], pb["pts0"], sh["points_2d"], sh["camera_ind"], sh["point_ind"])
    f = sba.fun(x0, C, P, sh["camera_ind"], sh["point_ind"], sh["points_2d"], sba.pointWeights)
    np.testing.assert_allclose(f, ref, rtol=0, atol=1e-8)


# ----------------------------------------------------------------------------- P2 Jacobian
def test_jacobian_blocks_vs_truth_and_fd(Engine, golden):
    g = golden("model_ring4_planar300")
    eng = Engine()
    eng.set_problem(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    Jc, Jp = eng.jacobian_blocks(_x0(g))
    J = np.concatenate([Jc, Jp], axis=2)
    Jt = g["J_truth_blocks"]
    # P2(i): element-wise vs the extended-precision truth of the reference's own fun
    assert np.abs(J - Jt).max() <= 1e-9 * np.abs(Jt).max()
    # P2(ii): Frobenius-relative vs scipy's 3-point finite difference
    Jfd = g["J_fd_blocks"]
    assert np.linalg.norm(J - Jfd) / np.linalg.norm(Jfd) <= 1e-9
    # and against the analytic oracle, tightly
    _, Jc_o, Jp_o = O.jacobian_blocks(g["cams0"], g["pts0"], g["camera_ind"], g["point_ind"],
                                      O.default_weights(g["point_ind"]))
    np.testing.assert_allclose(Jc, Jc_o, rtol=0, atol=1e-12 * np.abs(Jt).max())
    np.testing.assert_allclose(Jp, Jp_o, rtol=0, atol=1e-12 * np.abs(Jt).max())
    eng.close()


def test_jacobian_blocks_weighted_and_shuffled(Engine):
    pb = shuffle_observations(make_rig("ring8", 500, seed=2, variant="volume", p_vis=0.8), seed=9)
    rng = np.random.default_rng(1)
    w = rng.uniform(0.5, 2.0, pb["n_obs"])
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], w)
    Jc, Jp = eng.jacobian_blocks()
    _, Jc_o, Jp_o = O.jacobian_blocks(pb["cams0"], pb["pts0"], pb["camera_ind"], pb["point_ind"], w)
    scale = np.abs(Jc_o).max()
    np.testing.assert_allclose(Jc, Jc_o, rtol=0, atol=1e-12 * scale)
    np.testing.assert_allclose(Jp, Jp_o, rtol=0, atol=1e-12 * scale)
    eng.close()


# ----------------------------------------------------------------------------- P5 structure
def test_sparsity_pattern_identical(PySBA, golden):
    g = golden("model_ring4_planar300")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    sba = _sba(PySBA, g)
    A = sba.bundle_adjustment_sparsity(C, P, g["camera_ind"], g["point_ind"])
    assert tuple(A.shape) == tuple(g["A_shape"]) and A.nnz == 28 * g["camera_ind"].size
    assert str(A.dtype) == str(g["A_dtype"])
    assert np.array_equal(A.indices, g["A_indices"]) and np.array_equal(A.indptr, g["A_indptr"])
    Ao = O.bundle_adjustment_sparsity(C, P, g["camera_ind"], g["point_ind"])
    assert (A != Ao).nnz == 0


# ------------------------------------------------------------------ reduced camera system
@pytest.mark.parametrize("rig,npts,pvis,lam", [("ring4", 300, 1.0, 1e-6), ("example18", 400, 0.6, 1e-3),
                                               ("ring24", 300, 0.5, 1e-8), ("ring64", 200, 0.5, 1e-5)])
def test_reduced_camera_system_vs_oracle(Engine, rig, npts, pvis, lam):
    pb = make_rig(rig, npts, seed=1, variant="volume", p_vis=pvis)
    C, P = pb["n_cams"], pb["n_points"]
    ci, pi = pb["camera_ind"], pb["point_ind"]
    w = O.default_weights(pi)
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    f = O.fun(x0, C, P, ci, pi, pb["points_2d"], w)
    _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
    U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, C, P, ci, pi)
    g_or = np.hstack((gc.ravel(), gp.ravel()))
    sc_or = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
    S_or, rhs_or, _ = O.reduced_camera_system(U, gc, V, gp, W, ci, pi, lam, sc_or)
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi)
    out = eng.linearize(lam)
    np.testing.assert_allclose(out["cost"], 0.5 * f @ f, rtol=1e-13)
    np.testing.assert_allclose(out["grad"], g_or, rtol=0, atol=1e-11 * np.abs(g_or).max())
    np.testing.assert_allclose(out["scale_inv"], sc_or, rtol=1e-12)
    assert np.abs(out["S"] - out["S"].T).max() == 0.0
    assert np.abs(out["S"] - S_or).max() <= 1e-11 * np.abs(S_or).max()
    assert np.abs(out["rhs"] - rhs_or).max() <= 1e-10 * np.abs(rhs_or).max()
    eng.close()


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


@pytest.mark.parametrize("C", [8, 10, 12, 13, 15, 18, 22, 24, 32, 40, 48, 64])
def test_tensor_path_schur_equals_dfma_path(Engine, monkeypatch, C):
    """The two Schur kernels (DMMA tiles, schur_mma.cuh; DFMA duo blocks, schur.cuh) against each
    other and the oracle for every shape of the last tile group (11 C + 1 rows mod 48), with
    weights, with Y precomputed in HBM (k_make_Y) and evaluated by the producers in place."""
    base = make_rig("ring64" if C > 24 else "ring24", 260, seed=5, variant="volume", p_vis=0.93)
    pb = _first_cameras(base, C)
    ci, pi = pb["camera_ind"], pb["point_ind"]
    w = np.random.default_rng(C).uniform(0.5, 2.0, ci.size)
    outs = {}
    for name, env in (("dfma", {"LCBA_SCHUR_MMA": "0"}), ("mma_pre", {"LCBA_SCHUR_MMA": "1", "LCBA_MMA_PRE": "1"}),
                      ("mma_inplace", {"LCBA_SCHUR_MMA": "1", "LCBA_MMA_PRE": "0"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        eng = Engine()
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi, w)
        outs[name] = eng.linearize(1e-3)
        eng.close()
        for k in env:
            monkeypatch.delenv(k)
    ref = outs["dfma"]
    for name in ("mma_pre", "mma_inplace"):
        o = outs[name]
        assert np.abs(o["S"] - o["S"].T).max() == 0.0
        assert np.abs(o["S"] - ref["S"]).max() <= 1e-12 * np.abs(ref["S"]).max()
        assert np.abs(o["rhs"] - ref["rhs"]).max() <= 1e-11 * np.abs(ref["rhs"]).max()
    np.testing.assert_array_equal(outs["mma_pre"]["S"], outs["mma_inplace"]["S"])     # same arithmetic
    P = pb["pts0"].shape[0]
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    f = O.fun(x0, C, P, ci, pi, pb["points_2d"], w.reshape(-1, 1))
    _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
    U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, C, P, ci, pi)
    sc = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
    S_or, rhs_or, _ = O.reduced_camera_system(U, gc, V, gp, W, ci, pi, 1e-3, sc)
    assert np.abs(outs["mma_pre"]["S"] - S_or).max() <= 1e-11 * np.abs(S_or).max()
    assert np.abs(outs["mma_pre"]["rhs"] - rhs_or).max() <= 1e-10 * np.abs(rhs_or).max()


@pytest.mark.parametrize("C", [8, 9, 13, 16, 18, 24, 29, 32, 48, 64])
def test_int8_tensor_core_schur_equals_fp64_paths(Engine, monkeypatch, C):
    """The tcgen05 path (schur_i8.cuh: int8 digit planes of Y, exact int32 products in TMEM, FP64
    recombination) against the DMMA path and the oracle, for camera counts that exercise every
    tile shape of its plan (partial last row tile, folded 16/32-column tiles, 48-column tiles),
    with weights and partial visibility.  FP64-grade: 1e-13 between kernels, 1e-11 / 1e-10 vs numpy."""
    base = make_rig("ring64" if C > 24 else "ring24", 300, seed=6, variant="volume", p_vis=0.9)
    pb = _first_cameras(base, C)
    ci, pi = pb["camera_ind"], pb["point_ind"]
    w = np.random.default_rng(C).uniform(0.5, 2.0, ci.size)
    outs = {}
    for name, env in (("dmma", {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "0"}), ("i8", {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "1"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        eng = Engine()
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi, w)
        outs[name] = eng.linearize(1e-3)
        eng.close()
        for k in env:
            monkeypatch.delenv(k)
    a, b = outs["i8"], outs["dmma"]
    assert np.abs(a["S"] - a["S"].T).max() == 0.0
    assert np.abs(a["S"] - b["S"]).max() <= 1e-13 * np.abs(b["S"]).max()
    assert np.abs(a["rhs"] - b["rhs"]).max() <= 1e-12 * np.abs(b["rhs"]).max()
    d = np.sqrt(np.abs(np.diag(b["S"])))
    assert (np.abs(a["S"] - b["S"]) / np.outer(d, d)).max() <= 1e-12          # Jacobi-scaled
    P = pb["pts0"].shape[0]
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    f = O.fun(x0, C, P, ci, pi, pb["points_2d"], w.reshape(-1, 1))
    _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
    U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, C, P, ci, pi)
    sc = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
    S_or, rhs_or, _ = O.reduced_camera_system(U, gc, V, gp, W, ci, pi, 1e-3, sc)
    assert np.abs(a["S"] - S_or).max() <= 1e-11 * np.abs(S_or).max()
    assert np.abs(a["rhs"] - rhs_or).max() <= 1e-10 * np.abs(rhs_or).max()


def test_int8_tensor_core_schur_at_depth_and_trajectory(Engine, monkeypatch):
    """ring24 x 20011 dense points (953 K blocks, ragged last block) vs the oracle, then a full
    trajectory on ring24 x 5000 against oracle.trf_exact.  On 148 SMs the longest K range of the plan
    is 96 blocks, under I8_FLUSH = 224: every CTA flushes TMEM once.  The multi-flush path and the
    default dispatch at >= 32768 points are tested in test_gpu_i8_scale.py."""
    monkeypatch.setenv("LCBA_SCHUR_I8", "1")
    pb = make_rig("ring24", 20011, seed=7, variant="volume", p_vis=1.0)
    S_or, rhs_or, cost_or = _oracle_reduced(pb, 1e-5)
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    o = eng.linearize(1e-5)
    o2 = eng.linearize(1e-5)
    eng.close()
    assert np.array_equal(o["S"], o2["S"])                                     # deterministic
    assert np.abs(o["S"] - S_or).max() <= 1e-11 * np.abs(S_or).max()
    assert np.abs(o["rhs"] - rhs_or).max() <= 1e-10 * np.abs(rhs_or).max()
    pb = make_rig("ring24", 5000, seed=11, variant="volume", p_vis=1.0)
    ora = O.trf_exact(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], ftol=1e-4)
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    res, trace = eng.solve(ftol=1e-4)
    f, _ = eng.residuals()
    eng.close()
    assert res.nfev == ora.nfev and res.njev == ora.njev and res.status == ora.status
    costs_o = [rec["cost"] for rec in ora.trace] + [ora.cost]
    np.testing.assert_allclose([row["cost"] for row in trace], costs_o, rtol=3e-7)
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-8)
    assert abs(O.rmse_px(f) - O.rmse_px(ora.fun)) < 1e-6


def _oracle_reduced(pb, lam, w=None):
    C, P = pb["n_cams"], pb["n_points"]
    ci, pi = pb["camera_ind"], pb["point_ind"]
    wcol = O.default_weights(pi) if w is None else w.reshape(-1, 1)
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    f = O.fun(x0, C, P, ci, pi, pb["points_2d"], wcol)
    _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
    U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, C, P, ci, pi)
    sc = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
    S, rhs, _ = O.reduced_camera_system(U, gc, V, gp, W, ci, pi, lam, sc)
    return S, rhs, 0.5 * f @ f


@pytest.mark.parametrize("npts,weighted", [(20000, False), (20011, True)])
def test_tensor_path_dense_many_ring_laps_vs_oracle(Engine, monkeypatch, npts, weighted):
    """The headline configuration of the tensor-path Schur kernel at depth: ring24, full
    visibility, ~400 points (25 chunks of 16) per point slice, so the 2-stage ring of
    k_schur_mma wraps many times, k_make_Y loops over many tiles and every slice reduces many
    chunk partials.  20011 points leave a ragged tail (not a multiple of 16 x nslices).
    S / rhs against the numpy oracle (O.reduced_camera_system): 1e-11 / 1e-10 matrix-relative,
    with Y from HBM (k_make_Y) and evaluated in place by the producers."""
    pb = make_rig("ring24", npts, seed=7, variant="volume", p_vis=1.0)
    assert pb["n_obs"] >= 0.99 * 24 * pb["n_points"]          # dense: the DMMA path by default
    w = np.random.default_rng(3).uniform(0.5, 2.0, pb["n_obs"]) if weighted else None
    S_or, rhs_or, cost_or = _oracle_reduced(pb, 1e-5, w)
    outs = {}
    for name, env in (("mma_pre", {"LCBA_MMA_PRE": "1"}), ("mma_inplace", {"LCBA_MMA_PRE": "0"}),
                      ("dfma", {"LCBA_SCHUR_MMA": "0"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        eng = Engine()
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], w)
        outs[name] = eng.linearize(1e-5)
        eng.close()
        for k in env:
            monkeypatch.delenv(k)
    for name, o in outs.items():
        np.testing.assert_allclose(o["cost"], cost_or, rtol=1e-12, err_msg=name)
        assert np.abs(o["S"] - o["S"].T).max() == 0.0, name
        assert np.abs(o["S"] - S_or).max() <= 1e-11 * np.abs(S_or).max(), name
        assert np.abs(o["rhs"] - rhs_or).max() <= 1e-10 * np.abs(rhs_or).max(), name
    np.testing.assert_array_equal(outs["mma_pre"]["S"], outs["mma_inplace"]["S"])     # same arithmetic


def test_dense_ring24_trajectory_matches_oracle(Engine):
    """One full bundleAdjust(1e-4) trajectory on the dense 24-camera rig (5000 points: every
    point slice several ring laps deep) against the same algorithm on the CPU."""
    pb = make_rig("ring24", 5000, seed=11, variant="volume", p_vis=1.0)
    ora = O.trf_exact(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"],
                      ftol=1e-4)
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    res, trace = eng.solve(ftol=1e-4)
    f, _ = eng.residuals()
    eng.close()
    assert res.nfev == ora.nfev and res.njev == ora.njev and res.status == ora.status
    costs_o = [rec["cost"] for rec in ora.trace] + [ora.cost]
    np.testing.assert_allclose([row["cost"] for row in trace], costs_o, rtol=3e-7)
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-8)
    assert abs(O.rmse_px(f) - O.rmse_px(ora.fun)) < 1e-6      # north-star RMSE tolerance


# ------------------------------------------------------------------------- P3 / P4 solver
def _run_engine(Engine, g, **kw):
    eng = Engine()
    eng.set_problem(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    res, trace = eng.solve(**kw)
    cams, pts = eng.get_params()
    f, cost = eng.residuals()
    eng.close()
    return res, trace, cams, pts, f


@pytest.mark.parametrize("name", ["ba_ring8_volume1500", "ba_ring4_planar2000", "ba_example18_vis60_800"])
def test_trajectory_matches_exact_trf_oracle(Engine, golden, name):
    """Same algorithm on CPU (oracle.trf_exact) and GPU: iteration-by-iteration agreement."""
    g = golden(name)
    C = g["cams0"].shape[0]
    ora = O.trf_exact(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"], ftol=1e-4)
    res, trace, cams, pts, f = _run_engine(Engine, g, ftol=1e-4)
    assert res.nfev == ora.nfev and res.njev == ora.njev and res.status == ora.status
    costs_o = [rec["cost"] for rec in ora.trace] + [ora.cost]
    costs_g = [row["cost"] for row in trace]
    assert len(costs_g) == len(costs_o)
    # iterates that follow a nearly undamped step (reg_term ~ 1e-12: the gauge modes make the
    # reduced system almost singular, so one ulp in its Cholesky factor moves the iterate by
    # ~1e-7: observed 1.1e-7 on one ring4 iterate) agree to 3e-7; everything else to round-off
    np.testing.assert_allclose(costs_g, costs_o, rtol=3e-7)
    regs_o = [rec["reg_term"] for rec in ora.trace]
    got = [row["reg_term"] for row in trace[1:]]
    np.testing.assert_allclose(got[:2], regs_o[:2], rtol=1e-7)
    np.testing.assert_allclose(got, regs_o, rtol=1e-2)      # later ones: tiny, noisy gradients
    # the other columns of scipy's table: optimality of every row; step norm and cost reduction of
    # the trial that ended the previous iteration (0 when it was rejected).  Rows 0 and 1 (x0 and
    # the first step from it) agree to round-off: measured on a B200 (1000 W) 2.5e-10 relative at
    # most.  After that the ~1e-7 differences of the iterates explained above move the gradient and
    # the next step by that order of their INITIAL size, while both shrink by orders of magnitude:
    # measured at most 6.6e-7 of row 0's optimality and 1.6e-6 of |x0| for the step norm (ring4),
    # hence bounds of 2e-6 and 5e-6 on those scales.  The cost reduction is a difference of two
    # costs: the cost tolerance against the row's cost (measured 9.6e-8).
    x0n = np.linalg.norm(_x0(g))
    opt_o = np.array([rec["g_norm"] for rec in ora.trace] + [ora.optimality])
    opt_g = np.array([row["optimality"] for row in trace])
    np.testing.assert_allclose(opt_g[:2], opt_o[:2], rtol=1e-8)
    assert np.all(np.abs(opt_g - opt_o) <= 2e-6 * opt_o[0]), (opt_g, opt_o)
    last = [rec["trials"][-1] for rec in ora.trace]
    red_o = np.array([t["actual"] if t["actual"] > 0 else 0.0 for t in last])
    step_o = np.array([t["step_norm"] if t["actual"] > 0 else 0.0 for t in last])
    assert np.isnan(trace[0]["cost_reduction"]) and np.isnan(trace[0]["step_norm"])
    step_g = np.array([row["step_norm"] for row in trace[1:]])
    np.testing.assert_allclose(step_g[0], step_o[0], rtol=1e-9)
    assert np.all(np.abs(step_g - step_o) <= 5e-6 * x0n), (step_g, step_o)
    red_g = np.array([row["cost_reduction"] for row in trace[1:]])
    np.testing.assert_allclose(red_g[0], red_o[0], rtol=1e-9)
    assert np.all(np.abs(red_g - red_o) <= 3e-7 * np.array(costs_o[:-1])), (red_g, red_o)
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-9)
    # final reprojection RMSE within 1e-6 px (north-star tolerance); observed ~1e-10
    assert abs(O.rmse_px(f) - O.rmse_px(ora.fun)) < 1e-6
    co = ora.x[: C * 11].reshape(C, 11)
    rel = np.abs(cams[:, 6:] - co[:, 6:]).max(axis=0) / np.abs(co[:, 6:]).max(axis=0)
    assert rel.max() < 1e-6, rel                                  # intrinsics, relative


@pytest.mark.parametrize("rig,npts,pvis,variant", [("wide8", 400, 1.0, "volume"),      # config 4 geometry
                                                   ("ring64", 150, 0.5, "volume"),     # config 5 geometry
                                                   ("ring24", 300, 0.6, "planar"),     # two-plane points
                                                   ("ring4", 2500, 1.0, "volume")])    # config 1 geometry
def test_trajectory_matches_oracle_on_baseline_rigs(Engine, rig, npts, pvis, variant):
    """BASELINE.json configs 1/3/4/5 geometries at oracle-sized point counts."""
    pb = make_rig(rig, npts, seed=21, variant=variant, p_vis=pvis)
    ora = O.trf_exact(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"],
                      ftol=1e-4)
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    res, trace = eng.solve(ftol=1e-4)
    f, _ = eng.residuals()
    eng.close()
    assert res.nfev == ora.nfev and res.status == ora.status
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-8)
    assert abs(O.rmse_px(f) - O.rmse_px(ora.fun)) < 1e-6


def test_first_step_and_final_rmse_vs_tight_scipy(Engine, golden):
    """P3: one step from the common x0 against scipy with tight LSMR; P4: final RMSE."""
    g = golden("ba_ring8_volume1500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    res, trace, cams, pts, f = _run_engine(Engine, g, ftol=1e-4, max_nfev=2)
    t1 = g["tight_x1"]
    ct = t1[: C * 11].reshape(C, 11)
    rel = np.abs(cams[:, 6:] - ct[:, 6:]).max(axis=0) / np.abs(ct[:, 6:]).max(axis=0)
    assert rel.max() < 1e-6, rel                                  # intrinsics <= 1e-6 relative
    assert np.abs(pts.ravel() - t1[C * 11:]).max() < 1e-4          # points, mm
    for sl in (slice(0, 3), slice(3, 6)):                          # rotvec / t as blocks
        assert np.abs(cams[:, sl] - ct[:, sl]).max() / np.abs(ct[:, sl]).max() < 1e-6
    res, trace, cams, pts, f = _run_engine(Engine, g, ftol=1e-4)
    assert res.nfev == int(g["tight_nfev"]) and res.status == int(g["tight_status"])
    w = O.default_weights(g["point_ind"])
    f_t = O.fun(g["tight_x"], C, P, g["camera_ind"], g["point_ind"], g["points_2d"], w)
    assert abs(O.rmse_px(f) - O.rmse_px(f_t)) < 1e-6               # north-star RMSE tolerance
    np.testing.assert_allclose(res.cost, float(g["tight_cost"]), rtol=1e-6)
    # the reference's default (LSMR atol=btol=1e-6) stops slightly above: report-only bound
    f_r = O.fun(g["ref_x"], C, P, g["camera_ind"], g["point_ind"], g["points_2d"], w)
    assert 0 <= O.rmse_px(f_r) - O.rmse_px(f) < 1e-4


def test_zero_residual_at_noise_free_ground_truth(Engine):
    pb = make_rig("ring24", 2000, seed=4, variant="volume", p_vis=0.5, noise_px=0.0)
    eng = Engine()
    eng.set_problem(pb["cams_gt"], pb["pts_gt"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    r, cost = eng.residuals()
    assert np.abs(r).max() < 1e-8
    res, trace = eng.solve(ftol=1e-8)
    assert res.status in (1, 2, 3, 4) and res.cost <= cost + 1e-20
    eng.close()


def test_recovers_ground_truth_from_perturbed_start(Engine):
    pb = make_rig("ring8", 3000, seed=6, variant="volume", noise_px=0.0)
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    res, trace = eng.solve(ftol=1e-15, xtol=1e-15, gtol=1e-12, max_nfev=60)
    r, cost = eng.residuals()
    assert O.rmse_px(r) < 1e-6                     # noise-free: reprojection error -> 0
    assert all(b["cost"] <= a["cost"] for a, b in zip(trace, trace[1:]))   # monotone
    eng.close()


# ----------------------------------------------------------------------------- drop-in API
def test_bundleAdjust_drop_in_surface(PySBA, golden):
    g = golden("ba_ring4_planar2000")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    sba = _sba(PySBA, g)
    buf = io.StringIO()
    with redirect_stdout(buf):
        res = sba.bundleAdjust(1e-4)
    log = buf.getvalue().splitlines()
    assert log[0].split() == ["Iteration", "Total", "nfev", "Cost", "Cost", "reduction", "Step",
                              "norm", "Optimality"]
    assert log[1].split()[:3] == ["0", "1", "%.4e" % res_initial(g)]
    assert "termination condition is satisfied" in buf.getvalue()
    # the rows are printed live from inside the solve (scipy prints while iterating)
    seen = []
    eng = sba._get_engine()
    eng.set_params(g["cams0"], g["pts0"])
    eng.solve(ftol=1e-4, on_iteration=lambda row: seen.append((row["iteration"], row["nfev"])))
    assert seen[0] == (0, 1) and len(seen) >= 2 and [it for it, _ in seen] == list(range(len(seen)))
    sba = _sba(PySBA, g)
    with redirect_stdout(io.StringIO()):
        res = sba.bundleAdjust(1e-4)
    for k in ("x", "cost", "fun", "jac", "grad", "optimality", "active_mask", "nfev", "njev",
              "status", "message", "success"):
        assert k in res or hasattr(res, k), k
    assert res.success and res.status == 2 and res.x.shape == (11 * C + 3 * P,)
    assert sba.cameraArray.shape == (C, 11) and sba.points3D.shape == (P, 3)
    assert sba.cameraArray.base is res.x or np.shares_memory(sba.cameraArray, res.x)   # views of res.x
    assert res.fun.shape == (2 * g["camera_ind"].size,)
    np.testing.assert_allclose(res.cost, 0.5 * res.fun @ res.fun, rtol=1e-12)
    J = res.jac
    assert J.shape == (2 * g["camera_ind"].size, 11 * C + 3 * P) and J.nnz == 28 * g["camera_ind"].size
    np.testing.assert_allclose(J.T @ res.fun, res.grad, rtol=0, atol=1e-9 * np.abs(res.grad).max())
    assert abs(res.optimality - np.abs(res.grad).max()) <= 1e-9 * res.optimality
    # cost no worse than the reference's own run, within 1e-4 relative of it
    assert res.cost <= float(g["ref_cost"]) * (1 + 1e-9)
    np.testing.assert_allclose(res.cost, float(g["ref_cost"]), rtol=1e-4)
    # the object (and the result) must stay picklable (calibrate_camera.py:86-88)
    sba2 = pickle.loads(pickle.dumps(sba))
    np.testing.assert_array_equal(sba2.cameraArray, sba.cameraArray)
    r2 = pickle.loads(pickle.dumps(res))
    np.testing.assert_array_equal(r2["x"], res.x)
    # sba_print.py:17 usage
    r = sba.project(sba.points3D[sba.point2DIndices], sba.cameraArray[sba.cameraIndices]) - sba.points2D
    np.testing.assert_allclose(r.ravel(), res.fun, atol=1e-8)


def res_initial(g):
    w = O.default_weights(g["point_ind"])
    f = O.fun(_x0(g), g["cams0"].shape[0], g["pts0"].shape[0], g["camera_ind"], g["point_ind"],
              g["points_2d"], w)
    return 0.5 * f @ f


def test_weighted_bundle_adjust_vs_oracle(PySBA):
    pb = make_rig("ring8", 800, seed=8, variant="volume", p_vis=0.8)
    rng = np.random.default_rng(2)
    w = rng.uniform(0.5, 2.0, pb["n_obs"])
    ora = O.trf_exact(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"],
                      weights=w, ftol=1e-4)
    sba = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), pb["points_2d"], pb["camera_ind"],
                pb["point_ind"], pointWeights=w)
    res = sba.bundleAdjust(1e-4, verbose=0)
    assert res.nfev == ora.nfev and res.status == ora.status
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-9)


def test_unsorted_input_gives_same_solution(PySBA):
    pb = make_rig("example18", 500, seed=3, variant="volume", p_vis=0.7)
    sh = shuffle_observations(pb, seed=11)
    a = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    b = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), sh["points_2d"], sh["camera_ind"], sh["point_ind"])
    ra, rb = a.bundleAdjust(1e-4, verbose=0), b.bundleAdjust(1e-4, verbose=0)
    assert ra.nfev == rb.nfev
    np.testing.assert_allclose(ra.cost, rb.cost, rtol=1e-12)
    np.testing.assert_allclose(ra.x, rb.x, rtol=1e-9, atol=1e-9)
    # residual vector comes back in the caller's order
    perm_cost = 0.5 * rb.fun @ rb.fun
    np.testing.assert_allclose(perm_cost, rb.cost, rtol=1e-12)


def test_bundleAdjust_nocam_points_only(PySBA, golden):
    """SURVEY 8f rank 1: PySBA.bundleAdjust_nocam (pySBA.py:237-250) — cameras fixed."""
    g = golden("ba_nocam_ring8_600")
    ora = O.trf_exact_nocam(g["cams"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"],
                            ftol=1e-7)
    sba = PySBA(g["cams"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    cams_before = sba.cameraArray.copy()
    res = sba.bundleAdjust_nocam(1e-7)
    assert res.x.shape == (3 * g["pts0"].shape[0],) and sba.points3D.shape == g["pts0"].shape
    np.testing.assert_array_equal(sba.cameraArray, cams_before)            # cameras untouched
    assert res.nfev == ora.nfev and res.status == ora.status
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-11)
    np.testing.assert_allclose(res.x, ora.x, rtol=0, atol=1e-7)
    # against the reference's own run (scipy, inexact LSMR): same optimum
    np.testing.assert_allclose(res.cost, float(g["ref_cost"]), rtol=1e-9)
    np.testing.assert_allclose(res.x, g["ref_x"], rtol=0, atol=1e-4)       # mm
    np.testing.assert_allclose(res.cost, 0.5 * res.fun @ res.fun, rtol=1e-12)
    assert res.grad.shape == res.x.shape


def test_bundleAdjust_sharedcam(PySBA, golden):
    """SURVEY 8f rank 1: PySBA.bundleAdjust_sharedcam (pySBA.py:286-325) — one (f, k1, k2)."""
    g = golden("ba_sharedcam_ring8_500")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    args = (g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    ora = O.trf_exact_sharedcam(*args, ftol=1e-4)
    sba = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    res = sba.bundleAdjust_sharedcam(1e-4)
    assert res.x.shape == (3 + 8 * C + 3 * P,)
    assert np.all(sba.cameraArray[:, 6:9] == sba.cameraArray[0, 6:9])      # intrinsics stay tied
    np.testing.assert_array_equal(res.x[:3], sba.cameraArray[0, 6:9])
    assert res.nfev == ora.nfev and res.status == ora.status
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-8)
    np.testing.assert_allclose(res.x[:3], ora.x[:3], rtol=1e-5)
    w = O.default_weights(g["point_ind"])
    f = O.fun_sharedcam(res.x, C, P, g["camera_ind"], g["point_ind"], g["points_2d"], w)
    np.testing.assert_allclose(0.5 * f @ f, res.cost, rtol=1e-10)
    # run to the reference's own tolerance: the exact solver ends at or below the reference cost
    sba2 = PySBA(g["cams0"].copy(), g["pts0"].copy(), g["points_2d"], g["camera_ind"], g["point_ind"])
    res2 = sba2.bundleAdjust_sharedcam(1e-6)
    assert res2.cost <= float(g["ref_cost"]) * (1 + 1e-9)
    np.testing.assert_allclose(res2.cost, float(g["ref_cost"]), rtol=2e-3)


def test_unproject_matches_reference(golden):
    """SURVEY 8f rank 4: rigid_body.Unproject (OpenCV undistortPoints + ray/plane) on the GPU."""
    from lasercalib_b200.io import Unproject
    g, cal = golden("unproject_example"), golden("io_example17")
    for n, i in enumerate(g["cam_ids"]):
        out = Unproject(g["pts"][n], g["Z"][n], cal["camera_matrix"][i], cal["distortion"][i],
                        cal["rc_ext"][i], cal["tc_ext"][i])
        np.testing.assert_allclose(out, g["out"][n], rtol=0, atol=1e-8)      # mm
    out2 = Unproject(g["pts2"], [106.0], cal["camera_matrix"][0], g["d2"], cal["rc_ext"][0],
                     cal["tc_ext"][0])
    np.testing.assert_allclose(out2, g["out2"], rtol=0, atol=1e-8)
    assert Unproject(np.zeros((0, 2)), [0.0], cal["camera_matrix"][0], g["d2"], cal["rc_ext"][0],
                     cal["tc_ext"][0]).shape == (0, 3)


def test_calibrate_camera_script_flow(PySBA, golden):
    """The sequence of scripts/calibrate_camera.py:32-99 around the path: two laser datasets
    -> concatenation -> cameras from the example calibration files -> PySBA -> bundleAdjust ->
    readable / red export -> pickle of the object."""
    from lasercalib_b200 import io as lio
    cal = golden("io_example17")
    C = cal["cams"].shape[0]
    cams_gt = np.array([lio.camera_vector_from_calibration(cal["camera_matrix"][i], cal["distortion"][i],
                                                           cal["rc_ext"][i], cal["tc_ext"][i])
                        for i in range(C)])
    np.testing.assert_allclose(cams_gt[:, 3:], cal["cams"][:, 3:], atol=0)
    rng = np.random.default_rng(4)
    datasets = []
    for z in (0.0, 106.0):                                   # example/config.json z_gt
        n = 300
        pts = np.column_stack([rng.uniform(-600, 600, n), rng.uniform(-600, 600, n), np.full(n, z)])
        uv = O.project(np.repeat(pts, C, axis=0), np.tile(cams_gt, (n, 1))).reshape(n, C, 2)
        vis = (uv[..., 0] > 0) & (uv[..., 0] < 3208) & (uv[..., 1] > 0) & (uv[..., 1] < 2200)
        vis &= rng.random((n, C)) < 0.8
        keep = (vis.sum(axis=1) >= 4) & vis[:, 0]
        pts, uv, vis = pts[keep], uv[keep], vis[keep]
        pi, ci = np.nonzero(vis)
        datasets.append(dict(n_cams=C, n_pts=pts.shape[0], points_3d=pts + rng.normal(0, 2.0, pts.shape),
                             points_2d=uv[pi, ci] + rng.normal(0, 0.3, (pi.size, 2)),
                             camera_ind=ci, point_ind=pi))
    n_cams, points_3d, points_2d, camera_ind, point_ind = lio.concat_points_dataset(datasets)
    cams0 = cams_gt.copy()
    cams0[:, :3] += rng.normal(0, 1e-3, (C, 3))
    cams0[:, 3:6] += rng.normal(0, 1.0, (C, 3))
    sba = PySBA(cams0, points_3d, points_2d, camera_ind, point_ind)
    r0 = sba.project(sba.points3D[sba.point2DIndices], sba.cameraArray[sba.cameraIndices]) - sba.points2D
    res = sba.bundleAdjust(1e-4, verbose=0)
    r1 = sba.project(sba.points3D[sba.point2DIndices], sba.cameraArray[sba.cameraIndices]) - sba.points2D
    assert res.success and np.sqrt((r1 ** 2).sum(1)).mean() < 0.1 * np.sqrt((r0 ** 2).sum(1)).mean()
    ora = O.trf_exact(cams0, points_3d, points_2d, camera_ind, point_ind, ftol=1e-4)
    assert res.nfev == ora.nfev
    np.testing.assert_allclose(res.cost, ora.cost, rtol=1e-7)
    cam_list = [lio.sba_to_readable_format(sba.cameraArray[i, :]) for i in range(n_cams)]
    red = lio.readable_to_red_format(cam_list)
    assert red.shape == (C, 25) and np.all(np.isfinite(red))
    assert pickle.loads(pickle.dumps(sba)).cameraArray.shape == (C, 11)


# ------------------------------------------------ dense squared-residual variants (8f rank 1)
def test_sq_normal_matches_oracle(Engine, golden):
    """lcba_sq_normal (cost, J^T f, J^T J in one pass) against the analytic numpy restatement;
    weighted and unweighted, shuffled input, 18 cameras with partial visibility."""
    for pb, weights in ((make_rig("ring8", 500, seed=2, p_vis=0.8), None),
                        (shuffle_observations(make_rig("example18", 400, seed=3, p_vis=0.6), seed=1), "w")):
        ci, pi, uv = pb["camera_ind"], pb["point_ind"], pb["points_2d"]
        w = None if weights is None else np.random.default_rng(0).uniform(0.5, 2.0, ci.size)
        eng = Engine()
        eng.set_problem(pb["cams_gt"], pb["pts0"], uv, ci, pi, w)
        cost, g, H = eng.sq_normal(eng.SQ_CAMONLY, pb["cams0"])
        oc, og, oH = O.sq_normal_camonly(pb["cams0"], pb["pts0"], uv, ci, pi, w)
        np.testing.assert_allclose(cost, oc, rtol=1e-12)
        np.testing.assert_allclose(g, og, rtol=1e-9, atol=1e-9 * np.abs(og).max())
        np.testing.assert_allclose(H, oH, rtol=1e-9, atol=1e-9 * np.abs(oH).max())
        c2, g2, H2 = eng.sq_normal(eng.SQ_CAMONLY, pb["cams0"], derivs=False)
        assert g2 is None and H2 is None
        np.testing.assert_allclose(c2, oc, rtol=1e-12)
        th = np.hstack((np.eye(3) + 0.01, np.array([[1.0], [-2.0], [0.5]]))).ravel()
        cost, g, H = eng.sq_normal(eng.SQ_TRANSFORM, th)
        oc, og, oH = O.sq_normal_transform(th, pb["cams_gt"], pb["pts0"], uv, ci, pi, w)
        np.testing.assert_allclose(cost, oc, rtol=1e-12)
        np.testing.assert_allclose(g, og, rtol=1e-9, atol=1e-9 * np.abs(og).max())
        np.testing.assert_allclose(H, oH, rtol=1e-9, atol=1e-9 * np.abs(oH).max())
        np.testing.assert_allclose(eng.sq_normal(eng.SQ_TRANSFORM, th, derivs=False)[0], oc, rtol=1e-12)
        eng.close()


def test_camonly_matches_reference_run(PySBA, golden):
    """PySBA.bundle_adjustment_camonly against the reference's own run (golden) and against
    scipy fed the analytic Jacobian (the oracle arm that has no finite-difference noise)."""
    from scipy.optimize import least_squares
    g = golden("ba_camonly_ring8_400")
    ci, pi, uv, pts = g["camera_ind"], g["point_ind"], g["points_2d"], g["pts_gt"]
    C, N = g["cams0"].shape[0], ci.size
    sba = PySBA(g["cams0"].copy(), pts.copy(), uv, ci, pi)
    buf = io.StringIO()
    with redirect_stdout(buf):
        res = sba.bundle_adjustment_camonly(1e-4)
    assert (res.nfev, res.njev, res.status) == (int(g["ref_nfev"]), int(g["ref_njev"]), int(g["ref_status"]))
    np.testing.assert_allclose(res.cost, g["ref_cost"], rtol=1e-5)      # reference: 2-point FD
    assert buf.getvalue().splitlines()[0].split() == g["ref_log"].item().splitlines()[0].split()
    assert len(buf.getvalue().splitlines()) == len(g["ref_log"].item().splitlines())
    uv_a = O.project(pts[pi], sba.cameraArray[ci])
    uv_b = O.project(pts[pi], g["ref_cams"][ci])
    assert np.abs(uv_a - uv_b).max() < 1e-2
    np.testing.assert_allclose(res.fun, O.fun_camonly(res.x, C, ci, pi, uv, np.ones((N, 1)), pts),
                               rtol=1e-9, atol=1e-12)

    def jac(x, *a):
        p, Jc, _ = O.jacobian_blocks(x.reshape(C, 11), pts, ci, pi)
        Jd = 2 * (p - uv)[:, :, None] * Jc
        D = np.zeros((2 * N, 11 * C))
        for d in range(2):
            for a_ in range(11):
                D[2 * np.arange(N) + d, ci * 11 + a_] = Jd[:, d, a_]
        return D

    ref = least_squares(O.fun_camonly, g["cams0"].ravel(), jac=jac, ftol=1e-4, method="trf",
                        args=(C, ci, pi, uv, np.ones((N, 1)), pts))
    assert (res.nfev, res.njev, res.status) == (ref.nfev, ref.njev, ref.status)
    np.testing.assert_allclose(res.cost, ref.cost, rtol=1e-9)
    np.testing.assert_allclose(res.x, ref.x, rtol=1e-5, atol=1e-8)


def test_transform_points_3d_matches_reference_run(PySBA, golden):
    g = golden("ba_transform_ring8_400")
    ci, pi, uv = g["camera_ind"], g["point_ind"], g["points_2d"]
    sba = PySBA(g["cams_gt"].copy(), g["moved"].copy(), uv, ci, pi)
    res = sba.bundleAdjust_transform_points_3d(1e-3, verbose=0)
    assert (res.nfev, res.njev, res.status) == (int(g["ref_nfev"]), int(g["ref_njev"]), int(g["ref_status"]))
    np.testing.assert_allclose(res.cost, g["ref_cost"], rtol=1e-5)
    np.testing.assert_allclose(sba.points3D, g["ref_points"], rtol=1e-5, atol=1e-4)
    # the known map is recovered up to the pixel noise
    M = res.x.reshape(3, 4)
    np.testing.assert_allclose(M[:, :3], g["A"], atol=2e-3)
    np.testing.assert_allclose(M[:, 3], g["t"], atol=0.5)
    # a second call starts from the transformed points: the identity is (nearly) optimal
    res2 = sba.bundleAdjust_transform_points_3d(1e-3, verbose=0)
    np.testing.assert_allclose(res2.x.reshape(3, 4)[:, :3], np.eye(3), atol=1e-3)


# ----------------------------------------------------------------------------- error paths
def test_error_behaviour(PySBA, Engine):
    from lasercalib_b200._cabi import LcbaError
    pb = make_rig("ring4", 50, seed=0)
    bad = pb["pts0"].copy()
    bad[0, 0] = np.nan
    sba = PySBA(pb["cams0"].copy(), bad, pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    with pytest.raises(ValueError, match="Residuals are not finite in the initial point"):
        sba.bundleAdjust(1e-4, verbose=0)
    eng = Engine()
    ci = pb["camera_ind"].copy()
    ci[3] = 99
    with pytest.raises(LcbaError, match="out of range"):
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pb["point_ind"])
    with pytest.raises(LcbaError, match="no problem"):
        Engine().solve()
    with pytest.raises(LcbaError, match="64 cameras"):
        eng.set_problem(np.zeros((65, 11)), pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    with pytest.raises(ValueError, match="wrong size"):
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
        eng.sq_normal(eng.SQ_TRANSFORM, np.zeros(11))
    eng.close()


def test_point_without_observations_is_left_alone(Engine):
    pb = make_rig("ring4", 200, seed=0)
    pts = np.vstack([pb["pts0"], [[1.0, 2.0, 3.0]]])          # extra point nobody sees
    eng = Engine()
    eng.set_problem(pb["cams0"], pts, pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    res, _ = eng.solve(ftol=1e-4)
    _, out = eng.get_params()
    np.testing.assert_array_equal(out[-1], [1.0, 2.0, 3.0])
    assert res.status > 0
    eng.close()


def test_repeated_solves_replay_cuda_graphs_bit_identically(Engine):
    """From the second solve on a resident problem the static launch sequences of an iteration run
    as CUDA graphs (lcba.cu run_graphed).  Direct launches and graph replays must give bit-identical
    trajectories, also after switching the solver mode (the graphs are keyed on it) and back."""
    for rig, npts, pvis in (("ring8", 1500, 0.9), ("example18", 800, 0.6)):
        pb = make_rig(rig, npts, seed=13, variant="volume", p_vis=pvis)
        eng = Engine()
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
        runs = []
        for i in range(4):
            eng.set_params(pb["cams0"], pb["pts0"])
            if i == 2:                                       # another mode in between: points only
                r_nc, _ = eng.solve(ftol=1e-6, fix_cameras=True)
                assert r_nc.status > 0
                eng.set_params(pb["cams0"], pb["pts0"])
            res, trace = eng.solve(ftol=1e-4)
            cams, pts = eng.get_params()
            runs.append((res.nfev, res.njev, res.status, res.cost, [t["cost"] for t in trace], cams.copy(), pts.copy(),
                         int(res.gpu_launches)))
        for r in runs[1:]:
            assert r[:3] == runs[0][:3] and r[3] == runs[0][3] and r[4] == runs[0][4]
            np.testing.assert_array_equal(r[5], runs[0][5])
            np.testing.assert_array_equal(r[6], runs[0][6])
            assert r[7] == runs[0][7]                        # the launch count is the same claim either way
        eng.close()


# ------------------------------------------------------------------ full-size properties
def test_full_size_properties(Engine):
    """Config-3 scale (24 cameras, 1 M points; SURVEY 8d) through size-independent
    properties: fun on device == fun via the row-wise project kernel on a sample,
    J^T f from the linearise pass == directional finite difference of the cost, monotone
    cost, determinism of the (atomics-free) reductions."""
    pb = make_rig("ring24", 1_000_000, seed=0, variant="volume", p_vis=0.5)
    C, P, N = pb["n_cams"], pb["n_points"], pb["n_obs"]
    assert N > 5_000_000
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    r, cost = eng.residuals()
    np.testing.assert_allclose(0.5 * r @ r, cost, rtol=1e-12)
    sel = np.random.default_rng(0).choice(N, 5000, replace=False)
    ref = O.project(pb["pts0"][pb["point_ind"][sel]], pb["cams0"][pb["camera_ind"][sel]]) - pb["points_2d"][sel]
    np.testing.assert_allclose(r.reshape(-1, 2)[sel], ref, rtol=0, atol=1e-8)
    lin = eng.linearize(1e-6)
    g = lin["grad"]
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    v = np.random.default_rng(1).normal(size=x0.size)
    v[: 11 * C] *= np.maximum(1e-6, np.abs(x0[: 11 * C])) * 1e-3
    h = 1e-4
    _, cp = eng.residuals(x0 + h * v, want_r=False)
    _, cm = eng.residuals(x0 - h * v, want_r=False)
    np.testing.assert_allclose((cp - cm) / (2 * h), g @ v, rtol=1e-6)
    lin2 = eng.linearize(1e-6)
    assert np.array_equal(lin["S"], lin2["S"]) and np.array_equal(lin["grad"], lin2["grad"])   # deterministic
    res, trace = eng.solve(ftol=1e-4)
    assert res.status > 0 and all(b["cost"] <= a["cost"] for a, b in zip(trace, trace[1:]))
    f, c = eng.residuals()
    # sigma = 0.3 px per axis; ~12 views fit 3 point parameters => rmse ~ 0.424*sqrt(1-3/24)
    assert 0.37 < O.rmse_px(f) < 0.43
    eng.close()
