"""Extended-precision (np.longdouble) restatement of the linearisation.  TEST INFRASTRUCTURE ONLY.

The trust-region step is solved in the Jacobi-scaled space (x_scale='jac': s = scale_inv, the column norms
of J), so an error in S_ij matters as |dS_ij| / (s_i s_j), and one in rhs_i or g_i as |d_i| / (s_i |f|).
A bound relative to max|S| (or max|J|, max|g|) is 6 to 7 orders of magnitude looser than that on the focal,
translation and centre blocks.  Everything here is evaluated in long double (64-bit mantissa on x86-64,
binary128 in software on aarch64) from the same FP64 inputs the GPU gets, so it is about 2^11 more accurate
than any FP64 evaluation and can judge the kernels entry by entry in the scaled space.

What it restates (same formulas as oracle/pysba_oracle.py and lasercalib_b200/csrc/model.cuh):
  * the camera table of cam_table_build: R = I + a K + b K^2, J_r = I - b K + c K^2 (series below t = 0.1,
    long-double sin / cos above), and the reference's row-wise rotate / project;
  * the weighted residual and the analytic Jc / Jp blocks;
  * U, g_c, V, g_p, W, the damped point blocks inverted by adjugate (np.linalg has no long double), the
    reduced camera system S, rhs, and grad, scale_inv (0 -> 1), cost;
  * sq_normal_camonly and sq_normal_transform.
``check`` measures a GPU output against it in the scaled space and prints each error as a fraction of its
bound, the way tests/test_gpu_i8_scale._check does."""
import numpy as np
import pytest

LD = np.longdouble
NCP = 11
PI = LD("3.14159265358979323846264338327950288")


def require_long_double():
    """Skip unless np.longdouble carries at least 63 mantissa bits: comparing double against double would
    look like a pass and say nothing."""
    nm = np.finfo(LD).nmant
    if nm < 63:
        pytest.skip("np.longdouble has %d mantissa bits on this platform (< 63): no extended-precision "
                    "reference" % nm)


# ------------------------------------------------------------------------------------------- model
def rodrigues_coeffs(t2, form=None):
    """a = sin t / t, b = (1 - cos t) / t^2, c = (t - sin t) / t^3 of t2 = t^2, in long double.
    form None: series below t2 = 0.01 (the branch point of model.cuh), closed form above;
    'series' / 'closed' force one form (the series converges for any t, slowly above 1)."""
    t2 = LD(t2)
    if form is None:
        form = "series" if t2 < LD("0.01") else "closed"
    if form == "series":
        a = b = c = LD(0)
        term = LD(1)
        for k in range(24):                     # t2 <= 0.01: the 24th term is < 1e-60
            a += term / _fact(2 * k + 1)
            b += term / _fact(2 * k + 2)
            c += term / _fact(2 * k + 3)
            term *= -t2
        return a, b, c
    t = np.sqrt(t2)
    s, co = np.sin(t), np.cos(t)
    return s / t, (1 - co) / t2, (t - s) / (t * t2)


_FACT = [LD(1)]


def _fact(n):
    while len(_FACT) <= n:
        _FACT.append(_FACT[-1] * len(_FACT))
    return _FACT[n]


def skew(r):
    r = np.asarray(r, dtype=LD)
    return np.array([[0, -r[2], r[1]], [r[2], 0, -r[0]], [-r[1], r[0], 0]], dtype=LD)


def rotation(r, form=None):
    """(R, J_r) of one rotation vector (FP64 or long double), the cam_table_build form."""
    r = np.asarray(r)
    r = r if r.dtype == LD else r.astype(np.float64).astype(LD)
    a, b, c = rodrigues_coeffs((r * r).sum(), form)
    K = skew(r)
    K2 = K @ K
    eye = np.eye(3, dtype=LD)
    return eye + a * K + b * K2, eye - b * K + c * K2


def rotate(points, rot_vecs):
    """The reference's row-wise Rodrigues rotation (pySBA.py:61-73, model.cuh rotate_row)."""
    p = np.asarray(points, dtype=np.float64).astype(LD)
    r = np.asarray(rot_vecs, dtype=np.float64).astype(LD)
    th = np.sqrt((r * r).sum(axis=1))[:, None]
    axis = np.where(th > 0, r / np.where(th > 0, th, 1), LD(0))
    c, s = np.cos(th), np.sin(th)
    along = (p * axis).sum(axis=1)[:, None]
    return c * p + s * np.cross(axis, p) + along * (1 - c) * axis


def project(points, cam_rows):
    """The reference's project (pySBA.py:76-89) with its rotate, per row."""
    cam = np.asarray(cam_rows, dtype=np.float64).astype(LD)
    pc = rotate(points, cam[:, 0:3]) + cam[:, 3:6]
    xy = pc[:, 0:2] / pc[:, 2:3]
    n = (xy * xy).sum(axis=1)
    d = 1 + cam[:, 7] * n + cam[:, 8] * n * n
    return xy * (d * cam[:, 6])[:, None] + cam[:, 9:11]


def _eval_cond(R, X, t, Xc):
    """First-order sensitivity of (x, y) = Xc[:2] / Xc[2] to the FP64 rounding of Xc = R X + t, in units of
    u: |dx| <= u (A_x + |x| A_z) / |z_c| with A = |R| |X| + |t| per row.  Near the camera plane or behind a
    large translation this is far above |x|, and every output downstream of (x, y) inherits it."""
    A = np.einsum("nij,nj->ni", np.abs(R), np.abs(X)) + np.abs(t)
    az = np.abs(Xc[:, 2])
    x, y = Xc[:, 0] / Xc[:, 2], Xc[:, 1] / Xc[:, 2]
    return (A[:, 0] + np.abs(x) * A[:, 2]) / az, (A[:, 1] + np.abs(y) * A[:, 2]) / az, A[:, 2] / az


def obs_blocks(cams, pts, ci, pi, uv, w=None):
    """Residual (N,2), Jc (N,2,11), Jp (N,2,3) (weights applied), the residual scale (N,2) and the
    evaluation condition kappa (N,) of every observation.

    Residual scale: w (|E| dxy + |f x| (1 + |k1| n + |k2| n^2) + |f d x| + |c| + |uv_obs|) per component,
    with E = d(u,v)/d(x,y) and dxy of _eval_cond: the magnitudes an FP64 evaluation rounds, so that an
    error of a few u of this scale is what correct FP64 code makes.  On a well-placed point it is about
    w (3 |f d x| + |c| + |uv_obs|).  kappa = max(1, (|R_z| |X| + |t_z|) / |z_c|): the relative error of
    z_c, and with it of every Jacobian entry, that the FP64 rounding of R X + t alone causes."""
    cams = np.asarray(cams, dtype=np.float64)
    C, N = cams.shape[0], ci.size
    w = np.ones(N, dtype=LD) if w is None else np.asarray(w, dtype=np.float64).reshape(-1).astype(LD)
    Rs = np.empty((C, 3, 3), dtype=LD)
    Jr = np.empty((C, 3, 3), dtype=LD)
    for c in range(C):
        Rs[c], Jr[c] = rotation(cams[c, :3])
    cm = cams.astype(LD)[ci]
    X = np.asarray(pts)
    X = (X if X.dtype == LD else X.astype(np.float64).astype(LD))[pi]
    R = Rs[ci]
    Xc = np.einsum("nij,nj->ni", R, X) + cm[:, 3:6]
    iz = 1 / Xc[:, 2]
    x, y = Xc[:, 0] * iz, Xc[:, 1] * iz
    n = x * x + y * y
    f, k1, k2 = cm[:, 6], cm[:, 7], cm[:, 8]
    d = 1 + n * (k1 + k2 * n)
    dp = k1 + 2 * k2 * n
    uvo = np.asarray(uv, dtype=np.float64).astype(LD)
    r = np.stack([f * d * x + cm[:, 9] - uvo[:, 0], f * d * y + cm[:, 10] - uvo[:, 1]], axis=1) * w[:, None]
    E = np.empty((N, 2, 2), dtype=LD)
    E[:, 0, 0] = f * (d + 2 * x * x * dp)
    E[:, 0, 1] = E[:, 1, 0] = 2 * f * x * y * dp
    E[:, 1, 1] = f * (d + 2 * y * y * dp)
    D = np.zeros((N, 2, 3), dtype=LD)
    D[:, 0, 0] = iz
    D[:, 1, 1] = iz
    D[:, 0, 2] = -x * iz
    D[:, 1, 2] = -y * iz
    G = E @ D
    Xx = np.zeros((N, 3, 3), dtype=LD)                  # [X]x
    Xx[:, 0, 1], Xx[:, 0, 2] = -X[:, 2], X[:, 1]
    Xx[:, 1, 0], Xx[:, 1, 2] = X[:, 2], -X[:, 0]
    Xx[:, 2, 0], Xx[:, 2, 1] = -X[:, 1], X[:, 0]
    Jc = np.zeros((N, 2, NCP), dtype=LD)
    Jc[:, :, 0:3] = G @ (-(R @ Xx @ Jr[ci]))           # d(R X)/dr = -R [X]x J_r
    Jc[:, :, 3:6] = G
    Jc[:, 0, 6], Jc[:, 1, 6] = d * x, d * y
    Jc[:, 0, 7], Jc[:, 1, 7] = f * n * x, f * n * y
    Jc[:, 0, 8], Jc[:, 1, 8] = f * n * n * x, f * n * n * y
    Jc[:, 0, 9] = 1
    Jc[:, 1, 10] = 1
    Jp = G @ R
    dx, dy, kz = _eval_cond(R, X, cm[:, 3:6], Xc)
    aE = np.abs(E)
    dd = np.abs(f) * (1 + np.abs(k1) * n + np.abs(k2) * n * n)
    rs = np.stack([aE[:, 0, 0] * dx + aE[:, 0, 1] * dy + dd * np.abs(x) + np.abs(f * d * x) + np.abs(cm[:, 9])
                   + np.abs(uvo[:, 0]),
                   aE[:, 1, 0] * dx + aE[:, 1, 1] * dy + dd * np.abs(y) + np.abs(f * d * y) + np.abs(cm[:, 10])
                   + np.abs(uvo[:, 1])], axis=1) * np.abs(w)[:, None]
    return dict(r=r, Jc=Jc * w[:, None, None], Jp=Jp * w[:, None, None], rscale=rs,
                kappa=np.maximum(kz, LD(1)), d=d)


def inv3(A):
    """Inverse of stacked 3x3 matrices by adjugate / determinant."""
    a, b, c = A[:, 0, 0], A[:, 0, 1], A[:, 0, 2]
    d, e, f = A[:, 1, 0], A[:, 1, 1], A[:, 1, 2]
    g, h, i = A[:, 2, 0], A[:, 2, 1], A[:, 2, 2]
    adj = np.stack([e * i - f * h, c * h - b * i, b * f - c * e,
                    f * g - d * i, a * i - c * g, c * d - a * f,
                    d * h - e * g, b * g - a * h, a * e - b * d], axis=1).reshape(-1, 3, 3)
    det = a * adj[:, 0, 0] + b * adj[:, 1, 0] + c * adj[:, 2, 0]
    return adj / det[:, None, None]


def linearize(cams, pts, uv, ci, pi, lam, w=None, schur=True, chunk=2000):
    """Everything lcba_linearize returns at x = (cams, pts), damping lam, in long double: dict of S (11C,11C),
    rhs (11C), grad (11C+3P), scale_inv (11C+3P, zero columns -> 1), cost, fnorm = |f|, plus the observation
    blocks of obs_blocks, kappa_col (the largest kappa of each column's observations) and cond_V, the FP64 2-norm condition of each damped point block V_p + lam D_p^2.
    Repeated (camera, point) rows add up, as in oracle.normal_blocks; a point without observations has
    V = 0, scale 1 and contributes nothing.  schur=False skips S and rhs."""
    ci = np.asarray(ci, dtype=np.int64)
    pi = np.asarray(pi, dtype=np.int64)
    C, P = np.asarray(cams).shape[0], np.asarray(pts).shape[0]
    ob = obs_blocks(cams, pts, ci, pi, uv, w)
    r, Jc, Jp = ob["r"], ob["Jc"], ob["Jp"]
    U = np.zeros((C, NCP, NCP), dtype=LD)
    gc = np.zeros((C, NCP), dtype=LD)
    V = np.zeros((P, 3, 3), dtype=LD)
    gp = np.zeros((P, 3), dtype=LD)
    np.add.at(U, ci, np.einsum("nia,nib->nab", Jc, Jc))
    np.add.at(gc, ci, np.einsum("nia,ni->na", Jc, r))
    np.add.at(V, pi, np.einsum("nia,nib->nab", Jp, Jp))
    np.add.at(gp, pi, np.einsum("nia,ni->na", Jp, r))
    s = np.sqrt(np.concatenate([np.einsum("caa->ca", U).ravel(), np.einsum("paa->pa", V).ravel()]))
    s[s == 0] = 1
    cost = (r * r).sum() / 2
    kc = np.ones(C, dtype=LD)
    kp = np.ones(P, dtype=LD)
    np.maximum.at(kc, ci, ob["kappa"])
    np.maximum.at(kp, pi, ob["kappa"])
    out = dict(ob, grad=np.concatenate([gc.ravel(), gp.ravel()]), scale_inv=s, cost=cost,
               fnorm=np.sqrt(2 * cost), n_cams=C, kappa_col=np.concatenate([np.repeat(kc, NCP), np.repeat(kp, 3)]))
    sc, sp = s[:NCP * C].reshape(C, NCP), s[NCP * C:].reshape(P, 3)
    Vd = V.copy()
    Vd[:, [0, 1, 2], [0, 1, 2]] += LD(lam) * sp * sp
    out["cond_V"] = np.linalg.cond(Vd.astype(np.float64))
    if not schur:
        return out
    Vi = inv3(Vd)
    W = np.einsum("nia,nib->nab", Jc, Jp)
    S = np.zeros((NCP * C, NCP * C), dtype=LD)
    for c in range(C):
        S[NCP * c:NCP * (c + 1), NCP * c:NCP * (c + 1)] = U[c] + LD(lam) * np.diag(sc[c] ** 2)
    rhs = gc.ravel().copy()
    order = np.argsort(pi, kind="stable")
    starts = np.searchsorted(pi[order], np.arange(0, P + chunk, chunk))
    for k in range(len(starts) - 1):
        p0, p1 = k * chunk, min(P, (k + 1) * chunk)
        sel = order[starts[k]:starts[k + 1]]
        if sel.size == 0:
            continue
        E = np.zeros((p1 - p0, C, NCP, 3), dtype=LD)
        np.add.at(E, (pi[sel] - p0, ci[sel]), W[sel])
        E = E.reshape(p1 - p0, NCP * C, 3)
        T = E @ Vi[p0:p1]                                      # E_p V_p^-1
        rhs -= np.einsum("pac,pc->a", T, gp[p0:p1])
        S -= T.transpose(1, 0, 2).reshape(NCP * C, -1) @ E.transpose(1, 0, 2).reshape(NCP * C, -1).T
    out.update(S=S, rhs=rhs)
    return out


def _sq_rho(e, wl, rscale, J, kappa):
    """rho_H, rho_f: the relative FP64 error of e^2 and e^4, 2 u rscale / |e| and 4 u rscale / |e|, in units
    of u, averaged with the weights e^2 and e^4 that H and the cost give each residual; kappa_H: kappa of
    obs_blocks averaged with each observation's share of trace(H) (the Jacobian rows of a point near a camera
    plane carry kappa u relative error)."""
    a = np.abs(e)
    w2 = (wl * wl)[:, None]
    q = (J * J).reshape(J.shape[0], -1).sum(axis=1)
    return float((w2 * a * rscale).sum() / (w2 * a * a).sum()), \
        float((w2 * a ** 3 * rscale).sum() / (w2 * a ** 4).sum()), float((q * kappa).sum() / q.sum())


def sq_normal_camonly(cams, pts, uv, ci, pi, w=None):
    """(cost, g (11C), H (C,11,11)) of fun_camonly (f = w e^2, J = 2 w e dproj), |f| and the residual
    conditions rho_H, rho_f (see sq_errors)."""
    C = np.asarray(cams).shape[0]
    ob = obs_blocks(cams, pts, ci, pi, uv, None)
    wl = np.ones(ci.size, dtype=LD) if w is None else np.asarray(w, dtype=np.float64).reshape(-1).astype(LD)
    e = ob["r"]
    f = wl[:, None] * e * e
    J = 2 * (wl[:, None] * e)[:, :, None] * ob["Jc"]
    H = np.zeros((C, NCP, NCP), dtype=LD)
    g = np.zeros((C, NCP), dtype=LD)
    np.add.at(H, ci, np.einsum("nia,nib->nab", J, J))
    np.add.at(g, ci, np.einsum("nia,ni->na", J, f))
    rH, rf, kH = _sq_rho(e, wl, ob["rscale"], J, ob["kappa"])
    return dict(cost=(f * f).sum() / 2, g=g.ravel(), H=H, fnorm=np.sqrt((f * f).sum()), rho_H=rH, rho_f=rf,
                kappa_H=kH)


def sq_normal_transform(theta, cams, pts, uv, ci, pi, w=None):
    """(cost, g (12), H (12,12)) of fun_transform_points_3d, |f| and rho_H, rho_f."""
    M = np.asarray(theta, dtype=np.float64).astype(LD).reshape(3, 4)
    pl = np.asarray(pts, dtype=np.float64).astype(LD)
    X = pl @ M[:, :3].T + M[:, 3]
    ob = obs_blocks(cams, X, ci, pi, uv, None)
    wl = np.ones(ci.size, dtype=LD) if w is None else np.asarray(w, dtype=np.float64).reshape(-1).astype(LD)
    e = ob["r"]
    f = wl[:, None] * e * e
    Xh = np.concatenate([pl, np.ones((pl.shape[0], 1), dtype=LD)], axis=1)[pi]
    Jt = np.einsum("ndk,nj->ndkj", ob["Jp"], Xh).reshape(-1, 2, 12)
    Jf = (2 * (wl[:, None] * e)[:, :, None] * Jt).reshape(-1, 12)
    # the transformed points are rounded to FP64 on the GPU: a rounding of u |M| |X_h| per coordinate, which the
    # residual scale of obs_blocks already holds through |R| |X|
    rH, rf, kH = _sq_rho(e, wl, ob["rscale"], Jf.reshape(-1, 2, 12), ob["kappa"])
    return dict(cost=(f * f).sum() / 2, g=Jf.T @ f.ravel(), H=Jf.T @ Jf, fnorm=np.sqrt((f * f).sum()), rho_H=rH,
                rho_f=rf, kappa_H=kH)


def reframe(cams, pts, r0, b=(0.0, 0.0, 0.0)):
    """The same problem in another world frame, X' = Q X + b, R_c' = R_c Q^T, t_c' = t_c - R_c Q^T b, with Q
    chosen so that camera 0 gets the rotation vector r0 (any length: |r0| > pi is the equivalent vector of a
    rotation by 2 pi - |r0|).  Every reprojection is unchanged, so the conditioning of the problem is too.
    FP64; returns (cams', pts')."""
    from lasercalib_b200.synth import rotmat_to_rotvec, rotvec_to_rotmat
    cams = np.array(cams, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    Qt = rotvec_to_rotmat(cams[0, :3]).T @ rotvec_to_rotmat(r0)
    out = cams.copy()
    for c in range(cams.shape[0]):
        Rq = rotvec_to_rotmat(cams[c, :3]) @ Qt
        out[c, :3] = rotmat_to_rotvec(Rq)
        out[c, 3:6] = cams[c, 3:6] - Rq @ b
    out[0, :3] = r0
    return out, np.asarray(pts, dtype=np.float64) @ Qt + b


# ------------------------------------------------------------------------------------- the checker
def _ratio(err, scale):
    """err / scale with scale 0 -> the error must be exactly 0 there."""
    err = np.asarray(err, dtype=LD)
    scale = np.asarray(scale, dtype=LD)
    return np.where(scale > 0, err / np.where(scale > 0, scale, 1), np.where(err > 0, LD(np.inf), LD(0)))


def scaled_errors(got, ref, ci=None):
    """Errors of the GPU outputs in `got` against the long-double reference `ref`, in the scaled space:
      S          max |dS_ij| / (s_i s_j)
      rhs, grad  max |d_i| / (s_i |f|)
      Jc, Jp     per (camera, column): max |dJ| / kappa over the camera's observations, relative to the
                 column's largest entry for that camera (kappa: evaluation condition, obs_blocks)
      r          per element, relative to the residual scale of obs_blocks
      cost       |d cost| / sum_i |r_i| rscale_i: a residual r_i that is a difference of pixel values 1e3
                 times larger carries an FP64 error of a few u rscale_i, so relative to the cost itself two
                 correct FP64 evaluations differ by ~1e-14 (numpy against this reference: 9e-15 on ring4)
      scale_inv  relative
    grad and scale_inv are further divided by kappa_col, the largest evaluation condition of the column's
    observations (1 to 3 on well-placed points, 1e4 for a point near a camera plane, whose column norm and
    gradient come from its own Jacobian rows).  s = ref["scale_inv"], |f| = ref["fnorm"]."""
    e = {}
    s = ref.get("scale_inv")
    nc = NCP * ref["n_cams"]
    if "S" in got:
        e["S"] = _ratio(np.abs(got["S"] - ref["S"]), np.outer(s[:nc], s[:nc])).max()
    if "rhs" in got:
        e["rhs"] = _ratio(np.abs(got["rhs"] - ref["rhs"]), s[:nc] * ref["fnorm"]).max()
    kcol = ref.get("kappa_col", 1)
    if "grad" in got:
        e["grad"] = _ratio(np.abs(got["grad"] - ref["grad"]), s * ref["fnorm"] * kcol).max()
    if "cost" in got:
        e["cost"] = _ratio(abs(LD(got["cost"]) - ref["cost"]), (np.abs(ref["r"]) * ref["rscale"]).sum()).max()
    if "scale_inv" in got:
        e["scale_inv"] = _ratio(np.abs(got["scale_inv"] - s), s * kcol).max()
    if "r" in got:
        e["r"] = _ratio(np.abs(np.asarray(got["r"]).reshape(-1, 2) - ref["r"]), ref["rscale"]).max()
    for key in ("Jc", "Jp"):
        if key in got:
            J = ref[key]
            dJ = np.abs(np.asarray(got[key]) - J) / ref["kappa"][:, None, None]
            k = J.shape[2]
            cmax = np.zeros((ref["n_cams"], k), dtype=LD)
            emax = np.zeros((ref["n_cams"], k), dtype=LD)
            np.maximum.at(cmax, ci, np.abs(J).max(axis=1))
            np.maximum.at(emax, ci, dJ.max(axis=1))
            e[key] = _ratio(emax, cmax).max()
    return {k: float(v) for k, v in e.items()}


def residual_rho(ref):
    """rho = |rscale| / |f|: how much larger the pixel values are than the residuals that are their
    differences (about 1.5e3 on the synthetic rigs at x0)."""
    return float(np.sqrt((ref["rscale"] ** 2).sum()) / ref["fnorm"])


def check(label, got, ref, bounds, ci=None):
    """Prints every scaled error of `got` as a fraction of its bound, then asserts the bounds (a dict keyed
    like scaled_errors; keys of `got` without a bound are printed only).  Returns the errors.

    The rhs and grad bounds are stretched by max(1, rho / 2e3) (residual_rho): the rounding of each residual,
    a few u of its pixel scale, reaches g_i through J^T f as about u rho s_i |f|, whatever the kernel does
    afterwards.  On the synthetic rigs rho < 2e3 and the bounds stand as given."""
    err = scaled_errors(got, ref, ci)
    rho = residual_rho(ref) if "fnorm" in ref and ref["fnorm"] > 0 else 1.0
    bounds = {k: (b * max(1.0, rho / 2e3) if k in ("rhs", "grad") else b) for k, b in bounds.items()}
    msg = "; ".join("%s %.2e" % (k, v) + ("" if bounds.get(k) is None else " = %.3f of %.0e" % (v / bounds[k], bounds[k]))
                    for k, v in err.items())
    print("%s (rho %.1e): %s" % (label, rho, msg))
    for k, b in bounds.items():
        assert k in err, (label, k)
        assert err[k] <= b, "%s: %s" % (label, msg)
    return err


def sq_errors(got, ref):
    """sq_normal outputs in the scaled space: H by sqrt(H_ii H_jj), g by sqrt(H_ii) |f|, cost relative, each
    then divided by the residual condition that bounds it (max(1, rho_H) kappa_H for H, max(1, rho_H, rho_f)
    kappa_H for g, max(1, rho_f) for the cost: _sq_rho).  Camera-only H comes as (C,11,11) diagonal blocks, each
    scaled by its own diagonal."""
    H = ref["H"]
    Hg = np.asarray(got["H"]).reshape(H.shape)
    hd = np.sqrt(np.abs(np.einsum("...ii->...i", H)))
    hd = np.where(hd > 0, hd, 1)
    eH = _ratio(np.abs(Hg - H), hd[..., :, None] * hd[..., None, :]).max()
    eg = _ratio(np.abs(np.asarray(got["g"]) - ref["g"]), hd.ravel() * ref["fnorm"]).max()
    ec = _ratio(abs(LD(got["cost"]) - ref["cost"]), ref["cost"]).max()
    rH, rf, kH = max(1.0, ref["rho_H"]), max(1.0, ref["rho_f"]), ref["kappa_H"]
    return dict(H=float(eH) / (rH * kH), g=float(eg) / (max(rH, rf) * kH), cost=float(ec) / rf)


def check_sq(label, got, ref, bounds):
    """sq_errors printed as fractions of their bounds, then asserted."""
    err = sq_errors(got, ref)
    msg = "; ".join("%s %.2e = %.3f of %.0e" % (k, v, v / bounds[k], bounds[k]) for k, v in err.items())
    print("%s (rho_H %.1e, rho_f %.1e, kappa_H %.1e): %s" % (label, ref["rho_H"], ref["rho_f"], ref["kappa_H"], msg))
    for k, b in bounds.items():
        assert err[k] <= b, "%s: %s" % (label, msg)
    return err


def to_f64(ref, keys=("S", "rhs", "grad", "scale_inv")):
    """A copy of the given long-double outputs rounded to FP64 (for perturbation tests)."""
    return {k: np.asarray(ref[k], dtype=np.float64).copy() for k in keys if k in ref}
