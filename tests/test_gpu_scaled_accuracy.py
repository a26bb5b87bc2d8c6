"""The linearisation entry by entry in the solver's Jacobi-scaled space against the long-double reference
(tests/_ld_reference.py), at the camera model's edge geometries (A), over the Schur routes and shapes (B),
and for the squared-residual variants (C).

Error model (u = 2^-53).  In the scaled space (s = scale_inv, the column norms of J) every Jacobian column has
norm 1, so an FP64 sum of the products that make S_ij / (s_i s_j) carries about u sqrt(terms) of random-walk
round-off (terms <= 3 P: 4e-14 at P = 33 k) plus u cond(V_p + lam D_p^2) from each point factor; the inputs
of B keep that condition <= 1e4 (asserted) and measure <= 40 in the Jacobi-scaled space, hence the bound
1e-13 for S.  rhs and grad: the same sums times residuals, which the kernel rounds to a few u of their pixel
scale, rho = 1.5e3 times |f| on these rigs (_ld_reference.check stretches the 1e-13 bound by rho / 2e3 where
rho is larger).  The int8 route quantises Y to 48-bit digits: 2^-47 m_r m_c per entry with m_r <= s_r,
about 7e-15 scaled, below the same bound.  Jc / Jp per column: a few u of the column's largest entry, after
dividing out the condition kappa of z_c (kappa ~ 1e4 for the points near a camera plane): 1e-13.  Residual
and project: 1e-14 of the residual scale.  rotate: 4e-15 of |X|.  Cost: 1e-15 of sum |r_i| rscale_i.
scale_inv: 1e-14 relative (grad and scale_inv divided by the largest kappa of the column).  sq_normal: 1e-14
after dividing out the residual condition (_ld_reference.sq_errors).

Measured on a B200 (1000 W power limit), largest over each test:
  A: residual 6.3e-16, Jc 2.4e-15, Jp 1.7e-15, grad 8.9e-15, scale_inv 3.8e-15, cost 7.6e-17, rotate 9.7e-16;
  B: FP64 routes S 1.0e-14, rhs 1.4e-14, grad 1.2e-14, scale_inv 1.5e-15, cost 6.3e-18; int8 routes S 1.5e-14,
     rhs 1.5e-14, grad 7.2e-15; at depth int8 (ring24 x 33 000) S 4.1e-15, rhs 1.2e-14, DMMA (ring24 x 20 011)
     S 2.9e-15, rhs 8.8e-15;
  C: H 3.1e-16, g 2.5e-17, cost 1.1e-16.
The old matrix-relative bounds accept errors 1e5 to 1e6 times larger on the focal, translation and centre
blocks.  A 1e-8 relative error in one series coefficient of rodrigues_coeffs fails the two cases at
|r| = 0.1 (1 - 1e-9) here and passes every older test.

Every GPU test prints its observed errors as fractions of their bounds (pytest -s)."""
import numpy as np
import pytest

import _ld_reference as L
from lasercalib_b200.synth import make_rig, shuffle_observations
from oracle import pysba_oracle as O

pytestmark = pytest.mark.gpu

ENV_KEYS = ("LCBA_SCHUR_MMA", "LCBA_SCHUR_I8", "LCBA_MMA_PRE", "LCBA_PT_PASSES", "LCBA_I8_PLAN", "LCBA_I8_SCHED",
            "LCBA_I8_GUARD", "LCBA_MMA_DENSITY", "LCBA_SCHUR_CFG")
LIN_BOUNDS = dict(S=1e-13, rhs=1e-13, grad=1e-13, scale_inv=1e-14, cost=1e-15)
EDGE_BOUNDS = dict(r=1e-14, Jc=1e-13, Jp=1e-13, grad=1e-13, scale_inv=1e-14, cost=1e-15)
SQ_BOUNDS = dict(H=1e-14, g=1e-14, cost=1e-14)
# pass routes of A: dense one-pass linearisation (k_linearize_dense), the point-parallel passes, the
# observation-major ones
ROUTES = {"dense": {}, "pt": {"LCBA_SCHUR_MMA": "0"}, "obs": {"LCBA_SCHUR_MMA": "0", "LCBA_PT_PASSES": "0"}}
OBLIQUE = np.array([1.0, -2.0, 0.5]) / np.sqrt(5.25)
AXIS = np.array([0.0, 0.0, 1.0])
ROT_MAGS = [0.0, 1e-12, 1e-6, 0.1 * (1 - 1e-9), 0.1 * (1 + 1e-9), 1.0, np.pi - 1e-9, np.pi, np.pi + 0.5]


@pytest.fixture(autouse=True)
def _long_double():
    L.require_long_double()


@pytest.fixture(scope="module")
def Engine():
    from lasercalib_b200._cabi import Engine as cls
    return cls


def _open(Engine, monkeypatch, pb, w=None, env=None):
    """An engine holding pb, with `env` in force while the problem is set (where the routes are chosen)."""
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], w)
    finally:
        for k in env or {}:
            monkeypatch.delenv(k)
    return eng


def _problem(cams, pts, uv, ci, pi, **kw):
    return dict(cams0=np.ascontiguousarray(cams), pts0=np.ascontiguousarray(pts), points_2d=np.ascontiguousarray(uv),
                camera_ind=np.asarray(ci, dtype=np.int64), point_ind=np.asarray(pi, dtype=np.int64),
                n_cams=cams.shape[0], n_points=pts.shape[0], n_obs=int(np.asarray(ci).size), **kw)


# --------------------------------------------------------------------------------- A. edge problems
def _rot_problem(r0, b=(0.0, 0.0, 0.0)):
    pb = make_rig("ring8", 150, seed=61, variant="volume", p_vis=1.0)
    cams, pts = L.reframe(pb["cams0"], pb["pts0"], r0, b)
    return _problem(cams, pts, pb["points_2d"], pb["camera_ind"], pb["point_ind"])


def _distortion_problem(k1, k2):
    """wide8 (the 65 MP wide-angle rig) with strong radial distortion; the observations regenerated from the
    distorted model with 0.3 px noise.  With k1 = -0.4, k2 = -0.2 the observations where d = 1 + k1 n + k2 n^2
    falls below 0.1 are dropped, so d reaches about 0.1 on the kept ones."""
    pb = make_rig("wide8", 150, seed=62, variant="volume", p_vis=1.0)
    gt, cams = pb["cams_gt"].copy(), pb["cams0"].copy()
    gt[:, 7], gt[:, 8] = k1, k2
    cams[:, 7], cams[:, 8] = k1, k2
    ci, pi = pb["camera_ind"], pb["point_ind"]
    Xc = np.einsum("nij,nj->ni", np.stack([L.rotation(c[:3])[0].astype(float) for c in gt])[ci], pb["pts_gt"][pi]) \
        + gt[ci, 3:6]
    n = ((Xc[:, :2] / Xc[:, 2:]) ** 2).sum(1)
    keep = 1 + k1 * n + k2 * n * n >= 0.1
    ci, pi = ci[keep], pi[keep]
    uv = O.project(pb["pts_gt"][pi], gt[ci]) + np.random.default_rng(7).normal(0, 0.3, (ci.size, 2))
    return _problem(cams, pb["pts0"], uv, ci, pi)


def _near_problem():
    """ring8 with 8 extra points in front of camera 3 at z_c = 1e-1, 1e-2, 1e-3 of their distance (and the
    same at 1e-3 once more on the other side) and 2 behind it, each observed by every camera (observations
    projected from the ground truth with noise: the model projects a point behind a camera without
    complaint)."""
    pb = make_rig("ring8", 150, seed=63, variant="volume", p_vis=1.0)
    gt = pb["cams_gt"]
    R = L.rotation(gt[3, :3])[0].astype(float)
    centre = -R.T @ gt[3, 3:6]
    rng = np.random.default_rng(8)
    new = []
    for eps, side in ((1e-1, 1), (1e-2, 1), (1e-3, 1), (1e-3, -1), (-0.5, 1), (-0.2, -1), (5e-3, 1), (2e-2, -1)):
        lateral = side * R[0] * np.sqrt(1 - min(1.0, eps * eps))
        new.append(centre + 1500.0 * (lateral + eps * R[2]))
    new = np.array(new)
    P0, C = pb["n_points"], pb["n_cams"]
    ci = np.concatenate([pb["camera_ind"], np.tile(np.arange(C), len(new))])
    pi = np.concatenate([pb["point_ind"], P0 + np.repeat(np.arange(len(new)), C)])
    uv_new = O.project(new[pi[pb["n_obs"]:] - P0], gt[ci[pb["n_obs"]:]]) + rng.normal(0, 0.3, (len(new) * C, 2))
    uv = np.concatenate([pb["points_2d"], uv_new])
    pts = np.vstack([pb["pts0"], new + rng.normal(0, 0.5, new.shape)])
    return _problem(pb["cams0"], pts, uv, ci, pi)


def _large_problem():
    """ring8 scaled 50x (points to 3.5e4 mm, cameras at 7.5e4 mm), f = 1e4, cx = cy = 0, and the world frame
    moved by 2e4 mm: translations and points near 1e4 to 1e5 mm."""
    pb = make_rig("ring8", 150, seed=64, variant="volume", p_vis=1.0)
    gt, cams = pb["cams_gt"].copy(), pb["cams0"].copy()
    for c in (gt, cams):
        c[:, 3:6] *= 50.0
        c[:, 9:11] = 0.0
    gt[:, 6] = 1e4
    cams[:, 6] = 1e4 + np.random.default_rng(9).normal(0, 20.0, cams.shape[0])
    ci, pi = pb["camera_ind"], pb["point_ind"]
    uv = O.project(50.0 * pb["pts_gt"][pi], gt[ci]) + np.random.default_rng(10).normal(0, 0.3, (ci.size, 2))
    c2, p2 = L.reframe(cams, 50.0 * pb["pts0"], cams[0, :3], b=(2e4, -1e4, 5e3))
    return _problem(c2, p2, uv, ci, pi)


def _weights(kind, n):
    if kind == "int64":
        return np.ones(n, dtype=np.int64)
    rng = np.random.default_rng(11)
    w = rng.choice([0.0, 1e-3, 1.0, 1e3], n, p=[0.1, 0.3, 0.3, 0.3])
    return w


def _edge_cases():
    out = []
    for ax_name, ax in (("axis", AXIS), ("oblique", OBLIQUE)):
        for t in ROT_MAGS:
            out.append(("r%.12g-%s" % (t, ax_name), ("rot", t * ax)))
    for k1, k2 in ((-0.4, -0.2), (-0.4, 0.1), (0.3, -0.2), (0.3, 0.1)):
        out.append(("k1=%g,k2=%g" % (k1, k2), ("dist", (k1, k2))))
    out += [("near-plane", ("near", None)), ("large", ("large", None)), ("weights", ("weights", "mixed")),
            ("weights-int64", ("weights", "int64"))]
    return out


EDGE = _edge_cases()


def _edge(kind, arg):
    """(problem, weights or None) of one edge case."""
    if kind == "rot":
        return _rot_problem(arg), None
    if kind == "dist":
        return _distortion_problem(*arg), None
    if kind == "near":
        return _near_problem(), None
    if kind == "large":
        return _large_problem(), None
    pb = _rot_problem(np.array([0.3, -0.2, 0.1]))
    return pb, _weights(arg, pb["n_obs"])


@pytest.mark.parametrize("name,case", EDGE, ids=[n for n, _ in EDGE])
def test_model_edges_on_every_pass_route(Engine, monkeypatch, name, case):
    """Residuals (with x given and resident, and the cost-only pass), Jacobian blocks (sorted input: bulk
    store; shuffled: scatter), grad, scale_inv and cost of linearize on the dense, point-parallel and
    observation-major routes, and project / rotate, on problems at the edges of the camera model (EDGE)
    against the long-double reference; bounds in the module docstring."""
    pb, w = _edge(*case)
    ci, pi = pb["camera_ind"], pb["point_ind"]
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    ref = L.linearize(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi, 1e-3, w, schur=False)
    if case[0] == "dist" and case[1] == (-0.4, -0.2):
        dmin = float(ref["d"].min())
        print("%s: min d %.3f" % (name, dmin))
        assert 0.1 <= dmin < 0.15
    for route, env in ROUTES.items():
        eng = _open(Engine, monkeypatch, pb, w, env)
        try:
            r_x, cost_x = eng.residuals(x0)
            r_res, cost_res = eng.residuals()
            _, cost_only = eng.residuals(want_r=False)
            Jc, Jp = eng.jacobian_blocks()
            lin = eng.linearize(1e-3)
        finally:
            eng.close()
        lab = "%s %s" % (name, route)
        L.check(lab + " residuals(x)", dict(r=r_x, cost=cost_x), ref, dict(r=EDGE_BOUNDS["r"], cost=EDGE_BOUNDS["cost"]))
        L.check(lab + " residuals()", dict(r=r_res, cost=cost_res, Jc=Jc, Jp=Jp), ref,
                {k: EDGE_BOUNDS[k] for k in ("r", "cost", "Jc", "Jp")}, ci)
        L.check(lab + " cost only", dict(cost=cost_only), ref, dict(cost=EDGE_BOUNDS["cost"]))
        L.check(lab + " linearize", {k: lin[k] for k in ("grad", "scale_inv", "cost")}, ref,
                {k: EDGE_BOUNDS[k] for k in ("grad", "scale_inv", "cost")})
    sh = shuffle_observations(pb, seed=3)
    ws = None if w is None else w[np.random.default_rng(3).permutation(pb["n_obs"])]   # shuffle_observations' order
    ref_s = L.obs_blocks(sh["cams0"], sh["pts0"], sh["camera_ind"], sh["point_ind"], sh["points_2d"], ws)
    ref_s["n_cams"] = pb["n_cams"]
    eng = _open(Engine, monkeypatch, sh, ws)
    try:
        Jc, Jp = eng.jacobian_blocks()
        r_s, _ = eng.residuals()
    finally:
        eng.close()
    L.check("%s shuffled" % name, dict(Jc=Jc, Jp=Jp, r=r_s), ref_s,
            {k: EDGE_BOUNDS[k] for k in ("Jc", "Jp", "r")}, sh["camera_ind"])
    # the reference's row-wise project / rotate at the same rotation vectors
    eng = Engine()
    try:
        rows, X = pb["cams0"][ci], pb["pts0"][pi]
        proj = eng.project(X, rows)
        rot = eng.rotate(X, rows[:, :3])
    finally:
        eng.close()
    ref_p = L.obs_blocks(pb["cams0"], pb["pts0"], ci, pi, np.zeros((ci.size, 2)))
    ref_p["n_cams"] = pb["n_cams"]
    ref_p["r"] = L.project(X, rows)
    L.check("%s project" % name, dict(r=proj), ref_p, dict(r=EDGE_BOUNDS["r"]))
    e_rot = float((np.abs(rot - L.rotate(X, rows[:, :3])).max(axis=1) / np.abs(X).max(axis=1)).max())
    print("%s rotate: %.2e = %.3f of 4e-15" % (name, e_rot, e_rot / 4e-15))
    assert e_rot <= 4e-15


# -------------------------------------------------------------------------- B. routes x shapes sweep
def _first_cameras(base, C, min_views):
    keep = base["camera_ind"] < C
    ci, pi, uv = base["camera_ind"][keep], base["point_ind"][keep], base["points_2d"][keep]
    cnt = np.bincount(pi, minlength=base["pts0"].shape[0])
    good = cnt >= min_views
    sel = good[pi]
    remap = np.cumsum(good) - 1
    return _problem(base["cams0"][:C].copy(), base["pts0"][good].copy(), uv[sel], ci[sel], remap[pi[sel]])


def _sweep_problem(C, P, vis, extras, seed):
    """C cameras of ring24 / ring64 (the first C), exactly P points seen by >= min(3, C) of them, visibility
    vis, and the extras: 'rep' repeats 10 % of the observations (a third of those twice more) with new noise,
    'shuf' shuffles the observations, 'lonely' adds a point nobody observes, 'w' draws weights in [0.5, 2]."""
    rig = "ring64" if C > 24 else "ring24"
    base = make_rig(rig, int(P / max(vis, 0.3) ** 2 * 3) + 200, seed=seed, variant="volume", p_vis=vis)
    pb = _first_cameras(base, C, min(3, C))
    assert pb["n_points"] >= P, (C, P, vis, pb["n_points"])
    keep = pb["point_ind"] < P
    pb = _problem(pb["cams0"], pb["pts0"][:P], pb["points_2d"][keep], pb["camera_ind"][keep], pb["point_ind"][keep])
    rng = np.random.default_rng(seed)
    ci, pi, uv = pb["camera_ind"], pb["point_ind"], pb["points_2d"]
    pts = pb["pts0"]
    if "rep" in extras:
        extra = rng.choice(ci.size, max(3, ci.size // 10), replace=False)
        extra = np.concatenate([extra, extra[: extra.size // 3]])
        ci, pi = np.concatenate([ci, ci[extra]]), np.concatenate([pi, pi[extra]])
        uv = np.concatenate([uv, uv[extra] + rng.normal(0, 0.3, (extra.size, 2))])
    if "lonely" in extras:
        pts = np.vstack([pts, pts.mean(axis=0) + 10.0])
    pb = _problem(pb["cams0"], pts, uv, ci, pi)
    if "shuf" in extras:
        pb = shuffle_observations(pb, seed=seed)
    w = rng.uniform(0.5, 2.0, pb["n_obs"]) if "w" in extras else None
    return pb, w


DFMA = {"LCBA_SCHUR_MMA": "0"}
DMMA_PRE = {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "0", "LCBA_MMA_PRE": "1"}
DMMA_INPLACE = {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "0", "LCBA_MMA_PRE": "0"}


def _i8(plan=None, sched=None):
    env = {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "1", "LCBA_I8_GUARD": "0"}
    if plan:
        env["LCBA_I8_PLAN"] = plan
    if sched:
        env["LCBA_I8_SCHED"] = sched
    return env


# (route, env, C, P, visibility, lam, extras).  Every route meets a camera count, a point-count border,
# visibility 1 / 0.93 / 0.3 (DFMA skips invisible duo blocks below 80 % pairs), every lam, repeated pairs,
# shuffled input and a point without observations.  Camera counts 1 - 7 take the DFMA kernel by default
# (one camera is half a duo); DMMA and int8 run from 8 cameras, as their own tests do.
SWEEP = [
    ("dfma", DFMA, 1, 60, 1.0, 1.0, ""),
    ("dfma", DFMA, 2, 80, 1.0, 1e-3, "rep"),
    ("dfma", DFMA, 3, 90, 0.93, 1e-10, "shuf"),
    ("dfma-skip", DFMA, 5, 70, 0.3, 1e-3, "lonely"),
    ("dfma", DFMA, 7, 100, 1.0, 1.0, "w"),
    ("dfma-skip", DFMA, 13, 120, 0.3, 1e-10, "w,shuf"),
    ("dfma", DFMA, 64, 90, 0.93, 1e-3, "rep,lonely"),
    ("dmma-pre", DMMA_PRE, 8, 37, 1.0, 1e-10, ""),
    ("dmma-pre", DMMA_PRE, 25, 150, 0.93, 1.0, "shuf"),
    ("dmma-pre", DMMA_PRE, 48, 100, 1.0, 1e-3, "rep,w"),
    ("dmma-inplace", DMMA_INPLACE, 9, 60, 0.3, 1e-3, "lonely"),
    ("dmma-inplace", DMMA_INPLACE, 33, 101, 1.0, 1e-10, "w"),
    ("dmma-inplace", DMMA_INPLACE, 63, 90, 0.93, 1.0, "rep,shuf"),
    ("int8-cover-kmajor", _i8("cover"), 24, 20, 1.0, 1e-3, "w"),
    ("int8-strip-kmajor", _i8("strip"), 13, 21, 0.93, 1e-10, ""),
    ("int8-cover-range", _i8("cover", "range"), 64, 22, 0.3, 1.0, "shuf"),
    ("int8-strip-range", _i8("strip", "range"), 8, 300, 1.0, 1e-3, "rep,shuf"),
    ("int8", _i8(), 48, 200, 1.0, 1e-10, "w,lonely"),
]


def _run_lin(Engine, monkeypatch, pb, w, env, lam):
    eng = _open(Engine, monkeypatch, pb, w, env)
    try:
        out = eng.linearize(lam)
        out["fell_back"] = eng.i8_fell_back()
    finally:
        eng.close()
    return out


@pytest.mark.parametrize("route,env,C,P,vis,lam,extras", SWEEP,
                         ids=["%s-C%d-P%d-v%g-lam%g%s" % (r, c, p, v, l, "-" + e if e else "")
                              for r, _, c, p, v, l, e in SWEEP])
def test_schur_routes_and_shapes(Engine, monkeypatch, route, env, C, P, vis, lam, extras):
    """linearize(lam): S, rhs, grad, scale_inv and cost against the long-double reference on every Schur route
    (DFMA with and without visibility skipping, DMMA with Y precomputed and in place, int8 with both tile plans
    on both schedules, resolution guard off so the int8 result is the one checked) at the shapes of SWEEP.
    Precondition: every damped point block has cond(V_p + lam D_p^2) <= 1e4."""
    pb, w = _sweep_problem(C, P, vis, extras.split(","), seed=70 + C)
    ci, pi = pb["camera_ind"], pb["point_ind"]
    ref = L.linearize(pb["cams0"], pb["pts0"], pb["points_2d"], ci, pi, lam, w)
    cond = float(ref["cond_V"].max())
    assert cond <= 1e4, cond
    out = _run_lin(Engine, monkeypatch, pb, w, env, lam)
    assert out["fell_back"] == (0 if route.startswith("int8") else -1), out["fell_back"]
    assert np.abs(out["S"] - out["S"].T).max() == 0.0
    L.check("%s C=%d P=%d vis %g lam %g %s (cond V %.1e)" % (route, C, P, vis, lam, extras, cond),
            {k: out[k] for k in LIN_BOUNDS}, ref, LIN_BOUNDS)


@pytest.mark.parametrize("route,P", [("int8-default", 33_000), ("dmma-default", 20_011)])
def test_schur_default_routes_at_depth(Engine, monkeypatch, route, P):
    """The int8 route where it runs by default (ring24 x 33 000 points, >= 32 768 per shard) and DMMA where it
    does (ring24 x 20 011), against the long-double reference with the sweep's bounds: the int8 quantisation
    error stays inside the scaled bound at depth."""
    base = make_rig("ring24", P + 1500, seed=77, variant="volume", p_vis=1.0)
    keep = base["point_ind"] < P
    pb = _problem(base["cams0"], base["pts0"][:P], base["points_2d"][keep], base["camera_ind"][keep],
                  base["point_ind"][keep])
    ref = L.linearize(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], 1e-5)
    cond = float(ref["cond_V"].max())
    assert cond <= 1e4, cond
    out = _run_lin(Engine, monkeypatch, pb, None, {}, 1e-5)
    assert out["fell_back"] == (0 if route == "int8-default" else -1), out["fell_back"]
    L.check("ring24 x %d %s (cond V %.1e)" % (P, route, cond), {k: out[k] for k in LIN_BOUNDS}, ref, LIN_BOUNDS)


# ------------------------------------------------------------------------------------- C. sq_normal
@pytest.mark.parametrize("name,case", EDGE, ids=[n for n, _ in EDGE])
def test_sq_normal_on_model_edges(Engine, name, case):
    """lcba_sq_normal in camera-only mode (cameras cams0 over the problem's points) and transform mode (an
    affine map of the points, cameras cams0) on the edge problems of A: H scaled by sqrt(H_ii H_jj), g by
    sqrt(H_ii) |f|, cost relative; each divided by the residual condition of these squared residuals
    (L.sq_errors)."""
    pb, w = _edge(*case)
    ci, pi, uv = pb["camera_ind"], pb["point_ind"], pb["points_2d"]
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], uv, ci, pi, w)
        theta_c = pb["cams0"].copy()
        theta_c[:, 3:6] += 0.5
        cost, g, H = eng.sq_normal(eng.SQ_CAMONLY, theta_c)
        th = np.hstack((np.eye(3) * (1 + 1e-3) + 1e-3, np.array([[1.0], [-2.0], [0.5]]))).ravel()
        cost_t, g_t, H_t = eng.sq_normal(eng.SQ_TRANSFORM, th)
    finally:
        eng.close()
    ref = L.sq_normal_camonly(theta_c, pb["pts0"], uv, ci, pi, w)
    L.check_sq("%s camonly" % name, dict(cost=cost, g=g, H=H), ref, SQ_BOUNDS)
    ref_t = L.sq_normal_transform(th, pb["cams0"], pb["pts0"], uv, ci, pi, w)
    L.check_sq("%s transform" % name, dict(cost=cost_t, g=g_t, H=H_t), ref_t, SQ_BOUNDS)
