"""The int8 tensor-core Schur path (schur_i8.cuh: k_i8_rowmax, k_i8_make, k_i8_syrk, k_i8_gather) at the
shard sizes where it runs by default (>= 32768 points per shard, lcba.cu), against the FP64 DMMA path and
the numpy oracle: deep K ranges that flush TMEM several times per CTA, the dispatch switch, ragged and tiny
K, inputs with a hard dynamic range, and point-sharded runs.

Every GPU test prints its observed errors as a fraction of their bounds (run pytest with -s to see them).
The GPU tests of this file take about 45 s on one B200."""
import ctypes
import math
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle import pysba_oracle as O
from lasercalib_b200.synth import RIGS, make_rig, project_one_camera, rotvec_to_rotmat

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
I8_FLUSH = 224            # K blocks between TMEM flushes in k_i8_syrk (schur_i8.cuh I8_FLUSH)
I8_SWITCH = 32768         # smallest shard that takes the int8 path by default (lcba.cu)
LAM = 1e-5

# (rig, points, visibility, weighted): camera counts 24 / 64 / 8 at sizes where the longest K range of the
# plan on a 148-SM B200 needs >= 3 TMEM flushes (4 / 5 / 3), so the epilogue sums several flushes and the
# MMA warp waits on both parities of bar_tempty
DEPTH_CASES = [("ring24", 150_000, 1.0, False), ("ring64", 40_000, 0.5, True), ("ring8", 600_000, 1.0, True)]
HARD_KINDS = ["weights", "outliers", "twoview", "near", "nocam", "combined"]


# ----------------------------------------------------------------------------------------- helpers
def _subset(pb, P):
    """The problem restricted to its first P points (observations of the other points dropped), so that a
    test gets an exact point count: make_rig drops every point camera 0 does not see.  The first P points keep
    their numbers, so the point indices need no remapping."""
    assert pb["n_points"] >= P, (pb["n_points"], P)
    keep = pb["point_ind"] < P
    out = dict(pb)
    out.update(n_points=P, n_obs=int(keep.sum()), pts0=pb["pts0"][:P].copy(), pts_gt=pb["pts_gt"][:P].copy(),
               points_2d=np.ascontiguousarray(pb["points_2d"][keep]), camera_ind=pb["camera_ind"][keep].copy(),
               point_ind=pb["point_ind"][keep].copy())
    return out


def _run(monkeypatch, pb, lam, w=None, env=None, repeat=False):
    """linearize(lam) at x0 under the environment `env` (read when the problem is set), and the names of the
    kernels that one solver iteration launched: "i8_rowmax" is there exactly when the int8 path ran.
    out["fell_back"]: 1 when the resolution guard of the int8 path handed that linearize to DMMA, 0 when the
    int8 result stood, -1 on the DMMA path."""
    from lasercalib_b200._cabi import Engine
    env = env or {}
    for k in ("LCBA_SCHUR_I8", "LCBA_SCHUR_MMA", "LCBA_I8_GUARD"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], w)
        eng.solve(max_iterations=1, profile=True)
        kernels = set(eng.profile())
        eng.set_params(pb["cams0"], pb["pts0"])
        out = eng.linearize(lam)
        out["fell_back"] = eng.i8_fell_back()
        if repeat:
            out["again"] = eng.linearize(lam)
    finally:
        eng.close()
        for k in env:
            monkeypatch.delenv(k)
    return out, kernels


def _plan(lib, C, P, sm_count):
    tiles = np.zeros((256, 8), dtype=np.int32)
    work = np.zeros((512, 3), dtype=np.int32)
    nwork, nrg, nkb = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int64()
    nt = lib.lcba_debug_i8_plan(C, P, sm_count, tiles.ctypes.data_as(ctypes.c_void_p), 256,
                                work.ctypes.data_as(ctypes.c_void_p), 512, ctypes.byref(nwork), ctypes.byref(nrg),
                                ctypes.byref(nkb))
    assert nt >= 1, (C, P, nt)
    return tiles[:nt], work[:nwork.value], nkb.value


def _flushes(C, P, sm_count=None):
    """TMEM flushes of the CTA with the longest K range in the plan of C cameras x P points."""
    from lasercalib_b200 import _cabi
    if sm_count is None:
        import torch
        sm_count = torch.cuda.get_device_properties(0).multi_processor_count
    _, work, _ = _plan(_cabi.load(), C, P, sm_count)
    return math.ceil(int((work[:, 2] - work[:, 1]).max()) / I8_FLUSH)


def _oracle(pb, lam, w=None):
    """S, rhs, cost and column scales at x0 from numpy (O.reduced_camera_system, chunked over points).
    Columns without data get scale 1, the rule of the solver (oracle.trf_exact, scipy's trf)."""
    C, P = pb["n_cams"], pb["n_points"]
    ci, pi = pb["camera_ind"], pb["point_ind"]
    wcol = O.default_weights(pi) if w is None else w.reshape(-1, 1)
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    f = O.fun(x0, C, P, ci, pi, pb["points_2d"], wcol)
    _, Jc, Jp = O.jacobian_blocks(pb["cams0"], pb["pts0"], ci, pi, w)
    U, gc, V, gp, W = O.normal_blocks(f.reshape(-1, 2), Jc, Jp, C, P, ci, pi)
    sc = np.hstack((np.sqrt(np.einsum("caa->ca", U)).ravel(), np.sqrt(np.einsum("paa->pa", V)).ravel()))
    sc[sc == 0] = 1
    S, rhs, _ = O.reduced_camera_system(U, gc, V, gp, W, ci, pi, lam, sc)
    return dict(S=S, rhs=rhs, cost=0.5 * f @ f, scale_inv=sc)


def _check(label, a, ref, S=None, rhs=None, jacobi=None, cost=None):
    """max|dS| / max|S|, Jacobi-scaled max |dS_ij| / sqrt(S_ii S_jj), max|drhs| / max|rhs| and the relative
    cost difference of `a` against `ref`; prints each with its bound, then asserts the bounds given."""
    Sr = ref["S"]
    d = np.sqrt(np.abs(np.diag(Sr)))
    dS = np.abs(a["S"] - Sr)
    err = dict(S=dS.max() / np.abs(Sr).max(), jacobi=(dS / np.outer(d, d)).max(),
               rhs=np.abs(a["rhs"] - ref["rhs"]).max() / np.abs(ref["rhs"]).max(),
               cost=abs(a["cost"] - ref["cost"]) / abs(ref["cost"]))
    bounds = dict(S=S, jacobi=jacobi, rhs=rhs, cost=cost)
    msg = "; ".join("%s %.2e" % (k, e) + ("" if bounds[k] is None else " = %.3f of %.0e" % (e / bounds[k], bounds[k]))
                    for k, e in err.items())
    print("%s: %s" % (label, msg))
    for k, b in bounds.items():
        if b is not None:
            assert err[k] <= b, "%s: %s" % (label, msg)
    return err


def _assert_symmetric(out):
    assert np.abs(out["S"] - out["S"].T).max() == 0.0


@pytest.fixture(scope="module")
def lib():
    from lasercalib_b200 import build, _cabi
    build.build()
    return _cabi.load()


# ------------------------------------------------------------------------------- 1. default at depth
@pytest.mark.gpu
@pytest.mark.parametrize("rig,P,pvis,weighted", DEPTH_CASES)
def test_default_int8_path_at_depth_equals_dmma(monkeypatch, rig, P, pvis, weighted):
    """The int8 path as it runs by default (no override) at depth against the same problem on the DMMA path
    (LCBA_SCHUR_I8=0): max|dS| <= 1e-14 max|S|, Jacobi-scaled <= 5e-14, rhs <= 1e-13 max|rhs|, cost rtol
    1e-13, S symmetric to the bit, two linearize calls bit-identical; ring64 also against the oracle
    (1e-11 / 1e-10).  Measured on a B200 (1000 W), S / Jacobi / rhs: ring24 x 150 k 8.5e-17 / 2.2e-16 /
    5.4e-16; ring64 x 40 k 3.0e-16 / 5.1e-16 / 5.1e-15; ring8 x 600 k 2.5e-16 / 3.8e-16 / 7.6e-16; cost
    identical; ring64 against the oracle 8.6e-15 / 1.8e-13.  Dropping the d = 6 anti-diagonal in the epilogue
    fails all three (S 10x to 75x its bound), as does ending each tile's last K range one block early."""
    ask = int(P / pvis * 1.08) + 1000
    pb = _subset(make_rig(rig, ask, seed=31, variant="volume", p_vis=pvis), P)
    C = pb["n_cams"]
    nfl = _flushes(C, P)
    print("%s x %d: %d TMEM flushes in the longest K range" % (rig, P, nfl))
    assert nfl >= 3
    w = np.random.default_rng(P).uniform(0.5, 2.0, pb["n_obs"]) if weighted else None
    i8, k_i8 = _run(monkeypatch, pb, LAM, w, repeat=True)
    assert "i8_rowmax" in k_i8 and i8["fell_back"] == 0, (sorted(k_i8), i8["fell_back"])
    dm, k_dm = _run(monkeypatch, pb, LAM, w, {"LCBA_SCHUR_I8": "0"})
    assert "i8_rowmax" not in k_dm, sorted(k_dm)
    np.testing.assert_array_equal(i8["S"], i8["again"]["S"])
    np.testing.assert_array_equal(i8["rhs"], i8["again"]["rhs"])
    _assert_symmetric(i8)
    _check("%s x %d int8 vs DMMA" % (rig, P), i8, dm, S=1e-14, jacobi=5e-14, rhs=1e-13, cost=1e-13)
    if rig == "ring64":
        _check("%s x %d int8 vs oracle" % (rig, P), i8, _oracle(pb, LAM, w), S=1e-11, rhs=1e-10)


# ----------------------------------------------------------------------------------- 2. the switch
@pytest.mark.gpu
def test_dispatch_switches_to_int8_at_32768_points(monkeypatch):
    """32767 points per shard run on DMMA by default, 32768 on int8; each against the forced other path
    with the bounds of the at-depth test.  Measured on a B200 at both sizes: S 1.2e-16, Jacobi 2.2e-16, rhs
    1.5e-15."""
    base = _subset(make_rig("ring24", I8_SWITCH + 2000, seed=33, variant="volume", p_vis=1.0), I8_SWITCH)
    for P, default_i8 in ((I8_SWITCH - 1, False), (I8_SWITCH, True)):
        pb = _subset(base, P)
        d, k_d = _run(monkeypatch, pb, LAM)
        assert ("i8_rowmax" in k_d) == default_i8, (P, sorted(k_d))
        o, k_o = _run(monkeypatch, pb, LAM, env={"LCBA_SCHUR_I8": "0" if default_i8 else "1"})
        assert ("i8_rowmax" in k_o) == (not default_i8), (P, sorted(k_o))
        i8, dm = (d, o) if default_i8 else (o, d)
        assert i8["fell_back"] == 0
        _assert_symmetric(i8)
        _check("ring24 x %d int8 vs DMMA (default %s)" % (P, "int8" if default_i8 else "DMMA"), i8, dm,
               S=1e-14, jacobi=5e-14, rhs=1e-13, cost=1e-13)


# ------------------------------------------------------------------------------- 3. ragged / tiny K
@pytest.mark.gpu
@pytest.mark.parametrize("P", [1, 5, 20, 21, 22, 41, 42, 43])
def test_int8_path_ragged_and_tiny_k(monkeypatch, P):
    """Forced int8 at one partial K block (21 points each), exactly one or two, and one point more, on ring24
    with weights: cameras that see none of the points leave rows without data (exponent 0).  Against DMMA
    (1e-13 / 1e-12, Jacobi-scaled 1e-12, as test_int8_tensor_core_schur_equals_fp64_paths) and the oracle
    (1e-11 / 1e-10).  The resolution guard is off (LCBA_I8_GUARD=0), so S is the int8 kernels' own result.
    Measured on a B200 against DMMA: S <= 3.9e-15, Jacobi <= 4.3e-15, rhs <= 5.6e-14;
    against the oracle S <= 4.1e-15, rhs <= 1.4e-13.  A plan that ends each tile's last K range one block
    early fails every size; dropping the d = 6 anti-diagonal fails P = 22, 41 and 42 (S up to 3x its bound)."""
    pb = _subset(make_rig("ring24", 80, seed=35, variant="volume", p_vis=1.0), P)
    w = np.random.default_rng(P).uniform(0.5, 2.0, pb["n_obs"])
    i8, k_i8 = _run(monkeypatch, pb, 1e-3, w, {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "1", "LCBA_I8_GUARD": "0"})
    dm, k_dm = _run(monkeypatch, pb, 1e-3, w, {"LCBA_SCHUR_MMA": "1", "LCBA_SCHUR_I8": "0"})
    assert "i8_rowmax" in k_i8 and "i8_rowmax" not in k_dm
    _assert_symmetric(i8)
    _check("ring24 x %d int8 vs DMMA" % P, i8, dm, S=1e-13, jacobi=1e-12, rhs=1e-12)
    _check("ring24 x %d int8 vs oracle" % P, i8, _oracle(pb, 1e-3, w), S=1e-11, rhs=1e-10)


# ---------------------------------------------------------------------------- 4. hard dynamic range
def _hard_problem(rig, kinds, P=33_000, seed=41):
    """A rig of P points (plus the near-camera ones) with the inputs that stress the row exponents of the int8
    path (an FP32 estimate of each row maximum, 1e-3 of slack and 2 bits of headroom):
      weights  - log-uniform in [1e-3, 1e3], 1 % exact zeros (on points with >= 4 views) and one point whose
                 weights are all zero
      outliers - 0.1 % of the observations moved by 500 px (large z = L^-1 g_p)
      twoview  - 1 % of the points kept in only two adjacent cameras of one ring (ill-conditioned point
                 factors, where the FP32 Q = Jp L^-T cancels)
      near     - 4 points about 100 mm in front of camera 14, observed (O.project) by every camera whose image
                 they fall in (rows whose maximum comes from one point)
      nocam    - camera 5 with all its observations removed (rows without data)
    Returns (problem, weights or None)."""
    if "combined" in kinds:
        kinds = set(HARD_KINDS) - {"combined"}
    rng = np.random.default_rng(seed)
    pb = _subset(make_rig(rig, int(P * 1.1), seed=seed, variant="volume", p_vis=1.0), P)
    cams_gt, C = pb["cams_gt"], pb["n_cams"]
    ci, pi, uv = pb["camera_ind"], pb["point_ind"], pb["points_2d"]
    pts0 = pb["pts0"]
    if "nocam" in kinds:
        keep = ci != 5
        ci, pi, uv = ci[keep], pi[keep], uv[keep]
    two = np.zeros(P, dtype=bool)
    if "twoview" in kinds:
        ring = np.repeat(np.arange(len(RIGS[rig]["rings"])), [r["n"] for r in RIGS[rig]["rings"]])
        starts = np.searchsorted(pi, np.arange(P + 1))
        drop = np.zeros(ci.size, dtype=bool)
        for p in rng.choice(P, P // 100, replace=False):
            cs = ci[starts[p]:starts[p + 1]]
            pairs = [j for j in range(cs.size - 1) if cs[j + 1] == cs[j] + 1 and ring[cs[j]] == ring[cs[j + 1]]]
            if not pairs:
                continue
            j = pairs[rng.integers(len(pairs))]
            m = np.ones(cs.size, dtype=bool)
            m[j:j + 2] = False
            drop[starts[p]:starts[p + 1]] = m
            two[p] = True
        assert two.sum() >= 0.8 * (P // 100), two.sum()
        ci, pi, uv = ci[~drop], pi[~drop], uv[~drop]
    if "near" in kinds:
        R = rotvec_to_rotmat(cams_gt[14, :3])
        centre = -R.T @ cams_gt[14, 3:6]
        new_pts, new_ci, new_pi = [], [], []
        while len(new_pts) < 4:
            X = centre + 100.0 * R[2] + rng.normal(0.0, 10.0, 3)
            views = []
            for c in range(C):
                if "nocam" in kinds and c == 5:
                    continue
                q, z = project_one_camera(X[None], cams_gt[c])
                if z[0] > 0 and 0 <= q[0, 0] < pb["images"][c, 0] and 0 <= q[0, 1] < pb["images"][c, 1]:
                    views.append(c)
            if 14 not in views or len(views) < 3:
                continue
            new_ci += views
            new_pi += [P + len(new_pts)] * len(views)
            new_pts.append(X)
        new_pts = np.array(new_pts)
        new_ci, new_pi = np.array(new_ci, dtype=np.int64), np.array(new_pi, dtype=np.int64)
        new_uv = O.project(new_pts[new_pi - P], cams_gt[new_ci]) + rng.normal(0.0, 0.3, (new_ci.size, 2))
        ci, pi, uv = np.concatenate([ci, new_ci]), np.concatenate([pi, new_pi]), np.concatenate([uv, new_uv])
        pts0 = np.vstack([pts0, new_pts + rng.normal(0.0, 0.5, new_pts.shape)])
        two = np.concatenate([two, np.zeros(len(new_pts), dtype=bool)])
    Pn = pts0.shape[0]
    if "outliers" in kinds:
        uv = uv.copy()
        idx = rng.choice(ci.size, ci.size // 1000, replace=False)
        uv[idx, rng.integers(0, 2, idx.size)] += 500.0 * rng.choice([-1.0, 1.0], idx.size)
    w = None
    if "weights" in kinds:
        w = 10.0 ** rng.uniform(-3.0, 3.0, ci.size)
        views = np.bincount(pi, minlength=Pn)
        cand = np.flatnonzero(views[pi] >= 4)
        w[rng.choice(cand, ci.size // 100, replace=False)] = 0.0
        w[pi == 7] = 0.0                                   # one point without any weight
        # a two-view point takes one weight for both views: with weights 1e5 apart it would in effect be a
        # one-view point (out of scope), its point block conditioned ~5e10 at lam = 1e-10, and any two FP64
        # evaluations of its Schur contribution differ by ~1e-7 of it (7e-10 of max|S| between the oracle
        # and both GPU paths on ring24, which agreed with each other to 1.4e-14)
        tw = np.flatnonzero(two[pi])                       # point-major: the two views are adjacent
        w[tw] = np.repeat(w[tw[::2]], 2)
    out = dict(pb)
    out.update(n_points=Pn, n_obs=int(ci.size), pts0=np.ascontiguousarray(pts0), points_2d=np.ascontiguousarray(uv),
               camera_ind=ci.astype(np.int64), point_ind=pi.astype(np.int64))
    assert Pn >= I8_SWITCH and np.all(np.bincount(pi, minlength=Pn) >= 2)
    return out, w


# Inputs on which one point sets a camera row's largest |Y| entry far above the square root of the row's Schur
# diagonal (m_r^2 / S_rr, FP64 numpy at x0: example18 near 64, combined 1.4e3; every other input <= 0.82):
# finer than the 48-bit digits resolve (error ~ 2^-47 m_r m_c), so the resolution guard (k_i8_check, threshold
# 16) must hand these to DMMA and no other.
GUARDED = {("example18", "near"), ("example18", "combined")}


@pytest.mark.gpu
@pytest.mark.parametrize("rig,kind", [(r, k) for r in ("ring24", "example18") for k in HARD_KINDS])
def test_default_int8_path_on_hard_inputs(monkeypatch, rig, kind):
    """Default dispatch (int8) at 33 k points on inputs with a hard dynamic range (_hard_problem), one kind at
    a time and all together, against the oracle (1e-11 / 1e-10, column scales rtol 1e-12) and DMMA
    (Jacobi-scaled <= 1e-12, S symmetric); the combined input also through a full solve(ftol=1e-4) on both
    paths: equal nfev and status, cost rtol 1e-10.  The resolution guard must fall back exactly on GUARDED.
    Measured on a B200 (1000 W), Jacobi-scaled against DMMA, before the guard existed: ring24 weights
    1.3e-14, outliers 2.9e-16, twoview 2.1e-16, near 3.1e-15, nocam 2.4e-16, combined 2.8e-14; example18
    weights 1.9e-14, outliers 5.0e-16, twoview 3.1e-16, nocam 2.6e-16, and the two GUARDED inputs 4.3e-13
    and 3.3e-11 (over the bound; the model 2^-47 m_r^2 / S_rr gives 4.6e-13 and 1.0e-11).  Against the
    oracle at most 1.9e-13 of max|S| and 4.6e-13 of max|rhs|.  With the guard the two GUARDED inputs fall back
    and measure 1.2e-15 and 3.1e-15; the others keep int8 and measure as before.  Combined solves: nfev 12 / 12
    and 11 / 11, status 2, cost 6.7e-13 and 4.5e-14 apart.  The two-view points of adjacent ring cameras have point blocks
    conditioned <= 1e2, so they do not make the FP32 row-maximum estimate cancel."""
    pb, w = _hard_problem(rig, {kind})
    lam = 1e-10 if kind in ("twoview", "combined") else LAM
    i8, k_i8 = _run(monkeypatch, pb, lam, w)
    assert "i8_rowmax" in k_i8, sorted(k_i8)
    dm, k_dm = _run(monkeypatch, pb, lam, w, {"LCBA_SCHUR_I8": "0"})
    assert "i8_rowmax" not in k_dm, sorted(k_dm)
    _assert_symmetric(i8)
    label = "%s x %d %s" % (rig, pb["n_points"], kind)
    print("%s: resolution guard %s" % (label, "fell back to DMMA" if i8["fell_back"] == 1 else "kept int8"))
    assert i8["fell_back"] == (1 if (rig, kind) in GUARDED else 0)
    ora = _oracle(pb, lam, w)
    np.testing.assert_allclose(i8["scale_inv"], ora["scale_inv"], rtol=1e-12)
    _check(label + " int8 vs oracle", i8, ora, S=1e-11, rhs=1e-10)
    if kind == "combined":
        from lasercalib_b200._cabi import Engine
        res = {}
        for name, env in (("i8", {}), ("dmma", {"LCBA_SCHUR_I8": "0"})):
            for k, v in env.items():
                monkeypatch.setenv(k, v)
            eng = Engine()
            try:
                eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], w)
                res[name], _ = eng.solve(ftol=1e-4)
            finally:
                eng.close()
                for k in env:
                    monkeypatch.delenv(k)
        a, b = res["i8"], res["dmma"]
        print("%s solve: nfev %d / %d, status %d / %d, cost rel diff %.2e (bound 1e-10)"
              % (label, a.nfev, b.nfev, a.status, b.status, abs(a.cost - b.cost) / b.cost))
        assert a.nfev == b.nfev and a.status == b.status
        np.testing.assert_allclose(a.cost, b.cost, rtol=1e-10)
    _check(label + " int8 vs DMMA", i8, dm, jacobi=1e-12)


# ------------------------------------------------------------------------------------------ 5. sharded
@pytest.mark.gpu
def test_point_sharded_int8_path_matches_single_gpu():
    """Two shards of 40 k points (ring24), each on the int8 path, against the single-GPU run of the same
    80 k points: S 1e-12, rhs 1e-11, cost rtol 1e-13 (tests/_gpu_dist_i8_worker.py).  Not yet measured: it
    has only run on one-GPU machines, where it skips."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(port),
           os.path.join(REPO, "tests", "_gpu_dist_i8_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(out.stdout[-2000:])
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    for r in range(2):
        assert "rank %d ok" % r in out.stdout


# ----------------------------------------------------------------------------------- 6. CPU: the plans
def test_int8_plans_of_the_scale_tests(lib):
    """Host logic only (make_i8_plan through lcba_debug_i8_plan, 148 SMs as on a B200): the sizes the GPU
    tests above use give the flush counts they rely on, and the two sizes around the dispatch switch plan."""
    for rig, P, _, _ in DEPTH_CASES:
        C = sum(r["n"] for r in RIGS[rig]["rings"])
        assert _flushes(C, P, sm_count=148) >= 3, (rig, P)
    for P in (I8_SWITCH - 1, I8_SWITCH):
        tiles, work, nkb = _plan(lib, 24, P, 148)
        assert nkb == -(-P // 21) and work.shape[0] == 148
        for m0, mn, n0, nn, n20, n2n, w0, nw in tiles:
            ranges = work[w0:w0 + nw]
            assert ranges[0, 1] == 0 and ranges[-1, 2] == nkb and np.all(ranges[1:, 1] == ranges[:-1, 2])
