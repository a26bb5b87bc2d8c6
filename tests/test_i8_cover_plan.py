"""The cover plan of the int8 tensor-core Schur kernel (schur_i8.cuh make_i8_cover_plan): full 128 x 64 tiles
with a two-range A operand instead of row strips with square diagonal blocks.

Host logic (no GPU): the tiles take every lower-triangle entry exactly once under k_i8_gather's rule, the
shapes fit the kernel, the K ranges form one wave, and the plan that runs is never slower in the cost model
than the strip plan.  On the GPU: the cover plan against the strip plan, the FP64 DMMA path and itself (two
calls), at depth."""
import math
import os

import numpy as np
import pytest

from lasercalib_b200.synth import make_rig

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAMS = list(range(8, 33)) + [40, 48, 56, 64]
POINTS = (1000, 125_000, 1_000_000)
SMS = 148                 # B200
I8_FLUSH = 224            # K blocks between TMEM flushes in k_i8_syrk (schur_i8.cuh I8_FLUSH)
LAM = 1e-5

# (rig, points, visibility, weighted): with the cover plan forced, the longest K range on a 148-SM B200 needs
# >= 3 TMEM flushes (the cover plan has fewer tiles than the strip plan, so each tile gets more CTAs and
# shorter ranges: ring24 x 150 k, a depth case of test_gpu_i8_scale, flushes only twice under it)
DEPTH_CASES = [("ring24", 200_000, 1.0, False), ("ring64", 60_000, 0.5, True), ("ring8", 600_000, 1.0, True)]


def _plan(C, P, which, sms=SMS):
    from lasercalib_b200._cabi import Engine
    return Engine.i8_plan(C, P, sms, which)


def _taken(pl, C):
    """How often k_i8_gather writes each entry (rho, sig), rho >= sig, of the (11 C + 1)-row matrix: the
    rule of the kernel, restated."""
    n = 11 * C
    cnt = np.zeros((n + 1, n + 1), dtype=np.int64)
    for m0, mn, m20, m2n, n0, nn, n20, n2n, _, _ in pl["tiles"]:
        rows = np.concatenate((np.arange(8 * m0, 8 * (m0 + mn)), np.arange(8 * m20, 8 * (m20 + m2n))))
        cols = np.concatenate((np.arange(8 * n0, 8 * (n0 + nn)), np.arange(8 * n20, 8 * (n20 + n2n))))
        row_rg = np.zeros(pl["nrg"], dtype=bool)
        row_rg[rows // 8] = True
        rho, sig = (a.ravel() for a in np.meshgrid(rows, cols, indexing="ij"))
        upper = rho < sig
        drop = upper & row_rg[sig // 8]
        if pl["cover"]:
            drop &= (rho // 8 >= n0) & (rho // 8 < n0 + nn)
        keep = ~drop
        rho, sig = np.where(upper, sig, rho)[keep], np.where(upper, rho, sig)[keep]
        ok = (rho <= n) & (sig < n)
        np.add.at(cnt, (rho[ok], sig[ok]), 1)
    return cnt


def _map_shapes(pl):
    """The tensor-map shapes (box height in row groups, distance of A's second row range or 0) that i8_deal
    makes for a plan's tiles, restated: A, column block 1 and column block 2; a height of 0 needs no map."""
    shapes = set()
    for m0, mn, m20, m2n, n0, nn, n20, n2n, _, _ in pl["tiles"]:
        shapes |= {(int(mn), int(m20 - m0) if m2n else 0), (int(nn), 0), (int(n2n), 0)}
    return {s for s in shapes if s[0] > 0}


def test_cover_plan_takes_each_lower_entry_once():
    """For every camera count and size, every lower-triangle entry of the (11 C + 1)-row matrix (the z row
    included, its diagonal excluded) is written exactly once and nothing above the diagonal; the strip plan
    under the same gather rule too."""
    for C in CAMS:
        n = 11 * C
        want = np.tril(np.ones((n + 1, n + 1), dtype=np.int64))
        want[n, n] = 0
        for P in POINTS:
            for which in (1, 2):
                pl = _plan(C, P, which)
                assert pl["cover"] == (which == 2)
                np.testing.assert_array_equal(_taken(pl, C), want, err_msg="C %d P %d plan %d" % (C, P, which))


def test_cover_plan_shapes_k_ranges_and_choice():
    """Column blocks are multiples of 16 columns, at most 64 in all; A has at most 16 row groups, and two
    ranges only of 8 row groups each in increasing order (the 5-D tensor-map box); every tile's K ranges
    partition [0, nkb) and the grid is one wave; the plan that runs (no LCBA_I8_PLAN) costs no more in the
    model than the strip plan and reports the executed ops of its tiles; both plans need at most 16 tensor-map
    shapes (I8_MAX_MAPS in schur_i8.cuh: i8_encode_maps fails beyond that).  24 cameras: 8 tiles, the model's
    slowest CTA 17 % below the strip plan's, 7.47e12 executed int8 ops per launch at 1 M points (strip
    8.76e12)."""
    for C in CAMS:
        for P in POINTS:
            pl = _plan(C, P, 2)
            nkb = -(-P // 21)
            assert pl["nkb"] == nkb and 1 <= len(pl["work"]) <= SMS
            cols = 0
            for ti, (m0, mn, m20, m2n, n0, nn, n20, n2n, w0, nw) in enumerate(pl["tiles"]):
                assert nn >= 2 and nn % 2 == 0 and n2n % 2 == 0 and nn + n2n <= 8, (C, ti)
                assert 1 <= mn + m2n <= 16 and m0 + mn <= pl["nrg"] and n0 + nn <= pl["nrg"]
                if m2n:
                    assert mn == m2n == 8 and m20 > m0 + mn and m20 + m2n <= pl["nrg"], (C, ti)
                w = pl["work"][w0:w0 + nw]
                assert nw >= 1 and (w[:, 0] == ti).all()
                assert w[0, 1] == 0 and w[-1, 2] == nkb and (w[1:, 1] == w[:-1, 2]).all() and (w[:, 2] > w[:, 1]).all()
                cols += 8 * int(nn + n2n)
            assert pl["executed_ops"] == 26 * 2 * 128 * cols * 64 * nkb
            for which, p in ((1, _plan(C, P, 1)), (2, pl)):
                assert len(_map_shapes(p)) <= 16, (C, P, which, sorted(_map_shapes(p)))
            chosen = _plan(C, P, 0)
            assert chosen["cycles"] <= chosen["strip_cycles"], (C, P)
            assert chosen["cover"] == (chosen["cover_cycles"] < chosen["strip_cycles"])
    pl = _plan(24, 1_000_000, 0)
    assert pl["cover"] and len(pl["tiles"]) == 8
    assert pl["cycles"] <= 0.84 * pl["strip_cycles"]
    assert abs(pl["executed_ops"] - 7.465e12) < 1e9 and abs(_plan(24, 1_000_000, 1)["executed_ops"] - 8.763e12) < 1e9


# ------------------------------------------------------------------------------------------------ GPU
def _subset(pb, P):
    keep = pb["point_ind"] < P
    out = dict(pb)
    out.update(n_points=P, n_obs=int(keep.sum()), pts0=pb["pts0"][:P].copy(), pts_gt=pb["pts_gt"][:P].copy(),
               points_2d=np.ascontiguousarray(pb["points_2d"][keep]), camera_ind=pb["camera_ind"][keep].copy(),
               point_ind=pb["point_ind"][keep].copy())
    return out


def _run(monkeypatch, pb, w, env, repeat=False):
    """linearize(LAM) at x0 under `env`; out["kernels"]: the kernels of one solver iteration, out["fell_back"]
    as in test_gpu_i8_scale."""
    from lasercalib_b200._cabi import Engine
    for k in ("LCBA_SCHUR_I8", "LCBA_SCHUR_MMA", "LCBA_I8_GUARD", "LCBA_I8_PLAN"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], w)
        eng.solve(max_iterations=1, profile=True)
        kernels = set(eng.profile())
        eng.set_params(pb["cams0"], pb["pts0"])
        out = eng.linearize(LAM)
        out["fell_back"] = eng.i8_fell_back()
        out["kernels"] = kernels
        if repeat:
            out["again"] = eng.linearize(LAM)
    finally:
        eng.close()
        for k in env:
            monkeypatch.delenv(k)
    return out


def _err(a, ref):
    Sr = ref["S"]
    d = np.sqrt(np.abs(np.diag(Sr)))
    dS = np.abs(a["S"] - Sr)
    return dict(S=dS.max() / np.abs(Sr).max(), jacobi=(dS / np.outer(d, d)).max(),
                rhs=np.abs(a["rhs"] - ref["rhs"]).max() / np.abs(ref["rhs"]).max())


def _check(label, a, ref, bounds):
    e = _err(a, ref)
    print("%s: %s" % (label, "; ".join("%s %.2e (bound %.0e)" % (k, e[k], bounds[k]) for k in bounds)))
    for k, b in bounds.items():
        assert e[k] <= b, (label, k, e[k], b)


# cover against strip: the same exact integer products, summed in FP64 in another grouping (K ranges, flushes)
COVER_VS_STRIP = dict(S=1e-15, jacobi=2e-15, rhs=1e-15)
I8_VS_DMMA = dict(S=1e-14, jacobi=5e-14, rhs=1e-13)


@pytest.mark.gpu
@pytest.mark.parametrize("rig,P,pvis,weighted", DEPTH_CASES + [("ring24", 1_000_000, 1.0, False)])
def test_cover_plan_equals_strip_plan_and_dmma(monkeypatch, rig, P, pvis, weighted):
    """The cover plan (forced) against the strip plan (forced) and the DMMA path on the same problem, with the
    longest K range of the cover plan >= 3 TMEM flushes at the depth cases; S symmetric and two calls
    bit-identical; the resolution guard stays off; ring24 x 1 M is the headline workload, where the cover plan
    is also the default."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    ask = int(P / pvis * 1.08) + 1000
    pb = _subset(make_rig(rig, ask, seed=41, variant="volume", p_vis=pvis), P)
    C = pb["n_cams"]
    pl = _plan(C, P, 2, sms)
    nfl = math.ceil(int((pl["work"][:, 2] - pl["work"][:, 1]).max()) / I8_FLUSH)
    print("%s x %d: cover plan %d tiles, %d TMEM flushes in the longest K range" % (rig, P, len(pl["tiles"]), nfl))
    if (rig, P) != ("ring24", 1_000_000):
        assert nfl >= 3
    w = np.random.default_rng(P).uniform(0.5, 2.0, pb["n_obs"]) if weighted else None
    cv = _run(monkeypatch, pb, w, {"LCBA_I8_PLAN": "cover"}, repeat=True)
    st = _run(monkeypatch, pb, w, {"LCBA_I8_PLAN": "strip"})
    dm = _run(monkeypatch, pb, w, {"LCBA_SCHUR_I8": "0"})
    assert "i8_rowmax" in cv["kernels"] and "i8_rowmax" in st["kernels"] and "i8_rowmax" not in dm["kernels"]
    assert cv["fell_back"] == 0 and st["fell_back"] == 0
    assert np.abs(cv["S"] - cv["S"].T).max() == 0.0
    np.testing.assert_array_equal(cv["S"], cv["again"]["S"])
    np.testing.assert_array_equal(cv["rhs"], cv["again"]["rhs"])
    _check("%s x %d cover vs strip" % (rig, P), cv, st, COVER_VS_STRIP)
    _check("%s x %d cover vs DMMA" % (rig, P), cv, dm, I8_VS_DMMA)
    _check("%s x %d strip vs DMMA" % (rig, P), st, dm, I8_VS_DMMA)
    assert abs(cv["cost"] - dm["cost"]) <= 1e-13 * abs(dm["cost"])
    if (rig, P) == ("ring24", 1_000_000):
        dflt = _run(monkeypatch, pb, w, {})
        np.testing.assert_array_equal(dflt["S"], cv["S"])
