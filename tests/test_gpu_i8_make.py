"""k_i8_make (schur_i8.cuh: the digit planes of the int8 tensor-core Schur path) against its reference
k_i8_make_ref, byte for byte, through lcba_debug_i8_make: camera counts with one camera group, a ragged last
group and the 13-row-group last group at 64 cameras; a ragged last K block and fewer points than one K block;
weights over six decades with exact zeros, partial visibility and a point without observations; two
damping values; one size at depth.  Every run starts from a plane buffer filled with a poison byte, two
different ones per kernel, so that bytes a kernel does not write cannot pass as the other kernel's."""
import numpy as np
import pytest

from lasercalib_b200.synth import make_rig

I8_PTS = 21               # points per K block (schur_i8.cuh)


def _problem(C, P, seed, p_vis=0.9, weighted=True):
    """Cameras 0..C-1 of ring24 / ring64 and exactly P points (each seen by >= 2 of them) plus one point
    without observations; weights log-uniform over [1e-3, 1e3] with 5 % exact zeros, or None."""
    base = make_rig("ring64" if C > 24 else "ring24", int(P * 1.6) + 64, seed=seed, variant="volume", p_vis=p_vis)
    keep = base["camera_ind"] < C
    ci, pi, uv = base["camera_ind"][keep], base["point_ind"][keep], base["points_2d"][keep]
    good = np.bincount(pi, minlength=base["pts0"].shape[0]) >= 2
    idx = np.flatnonzero(good)[:P]
    assert idx.size == P, (C, P, idx.size)
    remap = np.full(base["pts0"].shape[0], -1)
    remap[idx] = np.arange(P)
    sel = remap[pi] >= 0
    ci, pi, uv = ci[sel], remap[pi[sel]], uv[sel]
    pts = np.vstack([base["pts0"][idx], base["pts0"][idx[:1]] + 10.0])      # point P: no observation
    w = None
    if weighted:
        rng = np.random.default_rng(seed)
        w = 10.0 ** rng.uniform(-3.0, 3.0, ci.size)
        w[rng.random(ci.size) < 0.05] = 0.0
    return base["cams0"][:C].copy(), pts, uv, ci, pi, w


POISONS = (0xA5, 0x5A)    # the tap fills the plane buffer with one of these before the kernel runs


def _check_planes(eng, lam):
    """Reference planes over both poison bytes are equal (the reference writes every byte, the same bytes on
    every run), and k_i8_make's over both poison bytes equal them: a byte it left unwritten would show."""
    ref = None
    for poison in POISONS:
        _, r = eng.debug_i8_make(lam, ref=True, poison=poison)
        if ref is None:
            ref = r
            assert ref.size > 0 and np.count_nonzero(ref) > 0
        else:
            assert np.array_equal(r, ref), (lam, poison, np.flatnonzero(r != ref)[:8])
        del r
    for poison in POISONS:
        _, new = eng.debug_i8_make(lam, ref=False, poison=poison)
        bad = np.flatnonzero(new != ref)
        assert bad.size == 0, (lam, poison, bad.size, bad[:8], new[bad[:8]], ref[bad[:8]])
        del new


def _run(monkeypatch, prob, lams):
    from lasercalib_b200._cabi import Engine
    monkeypatch.setenv("LCBA_SCHUR_I8", "1")
    cams, pts, uv, ci, pi, w = prob
    eng = Engine()
    try:
        eng.set_problem(cams, pts, uv, ci, pi, w)
        for lam in lams:
            _check_planes(eng, lam)
    finally:
        eng.close()


def test_i8_plane_bytes_match_the_plan():
    """The host's plane size (_cabi.i8_plane_bytes, which sizes the tap's buffer) against the library's plan."""
    import ctypes
    from lasercalib_b200 import _cabi
    lib = _cabi.load()
    tiles = np.zeros((256, 10), dtype=np.int32)
    for C in (1, 7, 8, 9, 13, 16, 24, 29, 63, 64):
        for P in (1, 20, 21, 22, 1000, 150_000):
            nrg, nkb = ctypes.c_int32(), ctypes.c_int64()
            nt = lib.lcba_debug_i8_cover_plan(C, P, 148, 0, tiles.ctypes.data_as(ctypes.c_void_p), 256, None, 0, None,
                                              ctypes.byref(nrg), ctypes.byref(nkb), None, None)
            assert nt >= 1, (C, P, nt)
            assert _cabi.i8_plane_bytes(C, P) == nkb.value * 6 * nrg.value * 512, (C, P)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [8, 9, 13, 16, 24, 29, 64])
def test_i8_make_planes_equal_reference(monkeypatch, C):
    """P = 21 k + 10 (a ragged last K block, plus the point without observations), p_vis 0.9, weights over
    six decades with exact zeros, lam 1e-3 and 1e-6: the planes of k_i8_make equal k_i8_make_ref's."""
    P = I8_PTS * (40 if C > 24 else 90) + 10
    _run(monkeypatch, _problem(C, P, seed=C), (1e-3, 1e-6))


@pytest.mark.gpu
@pytest.mark.parametrize("C,P", [(24, 15), (64, 1)])
def test_i8_make_fewer_points_than_a_k_block(monkeypatch, C, P):
    """One K block, partly (P < 21) or almost entirely zero padding."""
    _run(monkeypatch, _problem(C, P, seed=100 + C, p_vis=1.0), (1e-4,))


@pytest.mark.gpu
def test_i8_make_at_depth_and_reference_deterministic(monkeypatch):
    """ring24 x 150 000 points (7143 K blocks: ~73 per CTA of k_i8_make, 98 CTAs per camera group on 148 SMs), unweighted, full
    visibility: two reference runs give the same bytes, and k_i8_make's planes equal them over both poisons."""
    from lasercalib_b200._cabi import Engine
    monkeypatch.setenv("LCBA_SCHUR_I8", "1")
    pb = make_rig("ring24", 150_000, seed=3, variant="volume", p_vis=1.0)
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
        _check_planes(eng, 1e-5)
    finally:
        eng.close()
