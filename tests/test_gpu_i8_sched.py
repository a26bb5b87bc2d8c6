"""The K-major schedule of the int8 tensor-core Schur kernel (schur_i8.cuh i8_deal, k_i8_syrk): CTA q of a tile
with n CTAs takes the chunks j = q mod n of kc K blocks, so that all tiles sweep K together and read each K block
while it is in L2; a progress window bounds the drift.  LCBA_I8_SCHED=range keeps one contiguous K range per CTA.

Host logic (no GPU): under both schedules every (tile, K block) is read by exactly one CTA of the tile.  On the
GPU: S and rhs on the K-major schedule against the range schedule (the same exact integer products, summed in
FP64 in another grouping), two calls and two solves bit-identical, both tile plans."""
import numpy as np
import pytest

from lasercalib_b200.synth import make_rig

CAMS = list(range(8, 33)) + [40, 48, 56, 64]
POINTS = (1000, 125_000, 1_000_000)
SMS = 148                 # B200
LAM = 1e-5
K_VS_RANGE = dict(S=1e-15, rhs=1e-15)


def _schedule(C, P, which, kmajor, sms=SMS):
    from lasercalib_b200._cabi import Engine
    return Engine.i8_schedule(C, P, sms, which, kmajor)


def _kblocks(row):
    _, kb0, kb1, kfirst, kc, kstride = (int(x) for x in row)
    i = np.arange(kb1 - kb0)
    return kfirst + (i // kc) * kstride + i % kc


def test_schedules_read_each_k_block_once_per_tile():
    """For 8..64 cameras, three sizes and both tile plans: the CTAs of every tile read every K block exactly once
    under both schedules, each CTA at least one; the positions [kb0, kb1) partition the tile's K order; the range
    schedule is the contiguous deal (K block = position) without a window; the K-major one has chunks of <= 8 K
    blocks, n chunks apart for a tile of n CTAs, every CTA's count within one chunk of the others', and a window
    of at least twice the widest tile's chunk stride."""
    from lasercalib_b200._cabi import Engine
    for C in CAMS:
        for P in POINTS:
            nkb = -(-P // 21)
            for which in (1, 2):
                tiles = Engine.i8_plan(C, P, SMS, which)["tiles"]
                for kmajor in (False, True):
                    s = _schedule(C, P, which, kmajor)
                    work = s["work"]
                    assert work.shape[0] == int(tiles[:, 9].sum())
                    for ti, t in enumerate(tiles):
                        w = work[t[8]:t[8] + t[9]]
                        assert (w[:, 0] == ti).all()
                        assert w[0, 1] == 0 and w[-1, 2] == nkb and (w[1:, 1] == w[:-1, 2]).all()
                        assert (w[:, 2] > w[:, 1]).all(), (C, P, which, kmajor, ti)
                        seen = np.bincount(np.concatenate([_kblocks(r) for r in w]), minlength=nkb)
                        assert seen.shape[0] == nkb and (seen == 1).all(), (C, P, which, kmajor, ti)
                        cnt = w[:, 2] - w[:, 1]
                        if kmajor:
                            kc = int(w[0, 4])
                            assert 1 <= kc <= 8 and (w[:, 4] == kc).all() and (w[:, 5] == kc * t[9]).all()
                            assert (w[:, 3] == kc * np.arange(t[9])).all()
                            assert cnt.max() - cnt.min() <= kc
                        else:
                            assert (w[:, 3] == w[:, 1]).all() and (w[:, 5] == 0).all()
                    if kmajor:
                        assert s["window"] >= min(nkb, 2 * int(work[:, 5].max())), (C, P, which)
                    else:
                        assert s["window"] == 0


# ------------------------------------------------------------------------------------------------ GPU
def _problem(rig, C, P, pvis, seed):
    """P points of `rig` seen by at least 3 of its first C cameras."""
    pb = make_rig(rig, int(P / pvis * 1.3) + 1000, seed=seed, variant="volume", p_vis=pvis)
    keep = pb["camera_ind"] < C
    ci, pi, uv = pb["camera_ind"][keep], pb["point_ind"][keep], pb["points_2d"][keep]
    good = np.bincount(pi, minlength=pb["pts0"].shape[0]) >= 3
    good &= np.cumsum(good) <= P
    assert good.sum() == P
    sel = good[pi]
    remap = np.cumsum(good) - 1
    return dict(cams0=pb["cams0"][:C].copy(), pts0=pb["pts0"][good].copy(), points_2d=uv[sel].copy(),
                camera_ind=ci[sel].copy(), point_ind=remap[pi[sel]].copy(), n_cams=C, n_points=P)


def _run(monkeypatch, pb, w, env, repeat=False):
    """linearize(LAM) at x0 under `env`, after one profiled solver iteration (its kernels in out["kernels"])."""
    from lasercalib_b200._cabi import Engine
    for k in ("LCBA_SCHUR_I8", "LCBA_SCHUR_MMA", "LCBA_I8_GUARD", "LCBA_I8_PLAN", "LCBA_I8_SCHED"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], w)
        eng.solve(max_iterations=1, profile=True)
        out = dict(kernels=set(eng.profile()))
        eng.set_params(pb["cams0"], pb["pts0"])
        out.update(eng.linearize(LAM))
        out["fell_back"] = eng.i8_fell_back()
        if repeat:
            out["again"] = eng.linearize(LAM)
    finally:
        eng.close()
        for k in env:
            monkeypatch.delenv(k)
    return out


def _check(label, a, ref, bounds):
    e = dict(S=np.abs(a["S"] - ref["S"]).max() / np.abs(ref["S"]).max(),
             rhs=np.abs(a["rhs"] - ref["rhs"]).max() / np.abs(ref["rhs"]).max())
    print("%s: %s" % (label, "; ".join("%s %.2e (bound %.0e)" % (k, e[k], bounds[k]) for k in bounds)))
    for k, b in bounds.items():
        assert e[k] <= b, (label, k, e[k], b)


# (rig, cameras, points, visibility, weighted): the headline rig at a depth case and at full size, and 8, 48 and
# 64 cameras (one tile of many CTAs; many tiles of few)
CASES = [("ring24", 24, 150_000, 1.0, False), ("ring24", 24, 1_000_000, 1.0, False), ("ring8", 8, 400_000, 1.0, True),
         ("ring64", 48, 80_000, 0.5, True), ("ring64", 64, 60_000, 0.5, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("rig,C,P,pvis,weighted", CASES)
def test_kmajor_schedule_equals_range_schedule(monkeypatch, rig, C, P, pvis, weighted):
    """S and rhs on the K-major schedule (the default) within 1e-15 of max|S| / max|rhs| of the range schedule,
    two calls bit-identical, S symmetric, the int8 path ran and its result stood."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pb = _problem(rig, C, P, pvis, seed=51)
    s = _schedule(C, P, 0, True, sms)
    assert s["window"] < -(-P // 21), "the window must bind at this size"
    w = np.random.default_rng(P).uniform(0.5, 2.0, pb["camera_ind"].size) if weighted else None
    km = _run(monkeypatch, pb, w, {"LCBA_SCHUR_I8": "1"}, repeat=True)
    rg = _run(monkeypatch, pb, w, {"LCBA_SCHUR_I8": "1", "LCBA_I8_SCHED": "range"})
    assert "i8_rowmax" in km["kernels"] and "i8_rowmax" in rg["kernels"]
    assert km["fell_back"] == 0 and rg["fell_back"] == 0
    assert np.abs(km["S"] - km["S"].T).max() == 0.0
    np.testing.assert_array_equal(km["S"], km["again"]["S"])
    np.testing.assert_array_equal(km["rhs"], km["again"]["rhs"])
    _check("%s[%d] x %d K-major vs range" % (rig, C, P), km, rg, K_VS_RANGE)


@pytest.mark.gpu
def test_kmajor_schedule_both_plans(monkeypatch):
    """Both tile plans on both schedules, ring24 x 200 000: K-major within 1e-15 of range for each plan."""
    pb = _problem("ring24", 24, 200_000, 1.0, seed=53)
    out = {}
    for plan in ("strip", "cover"):
        for sched in ("kmajor", "range"):
            env = {"LCBA_SCHUR_I8": "1", "LCBA_I8_PLAN": plan}
            if sched == "range":
                env["LCBA_I8_SCHED"] = "range"
            r = _run(monkeypatch, pb, None, env)
            assert r["fell_back"] == 0
            out[plan, sched] = r
        _check("ring24 x 200000 %s: K-major vs range" % plan, out[plan, "kmajor"], out[plan, "range"], K_VS_RANGE)


@pytest.mark.gpu
def test_kmajor_schedule_two_solves_bit_identical():
    """Two solves from the same start on one handle (the second replays the captured graph, so the window's
    launch epochs advance without a reset): the same iterates, cost and trace, bit for bit."""
    from lasercalib_b200._cabi import Engine
    pb = _problem("ring24", 24, 150_000, 1.0, seed=55)
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
        runs = []
        for _ in range(2):
            eng.set_params(pb["cams0"], pb["pts0"])
            res, trace = eng.solve(max_iterations=4)
            cams, pts = eng.get_params()
            runs.append((cams, pts, res.cost, [(r["cost"], r["step_norm"]) for r in trace]))
        assert eng.i8_fell_back() == 0
    finally:
        eng.close()
    np.testing.assert_array_equal(runs[0][0], runs[1][0])
    np.testing.assert_array_equal(runs[0][1], runs[1][1])
    assert runs[0][2] == runs[1][2]
    np.testing.assert_array_equal(np.array(runs[0][3]), np.array(runs[1][3]))     # NaN where a row has no step
