"""Held parameters of bundleAdjust without a GPU: the argument normalisation of
PySBA.bundleAdjust(fixed_camera_params=..., fixed_points=...) and the CPU oracle of the masked solve
(tests/_fixed_oracle.py)."""
import numpy as np
import pytest

from oracle import pysba_oracle as O
from lasercalib_b200.pySBA import normalize_fixed

from _fixed_oracle import trf_exact_fixed


def test_camera_mask_broadcasts_and_keeps_its_entries():
    m = np.zeros(11, bool)
    m[:6] = True
    cam, pt = normalize_fixed(m, None, 4, 10)
    assert pt is None and cam.shape == (4, 11) and cam.dtype == np.bool_
    assert np.array_equal(cam, np.tile(m, (4, 1)))
    full = np.zeros((4, 11), bool)
    full[2, 9:] = True
    cam, _ = normalize_fixed(full, None, 4, 10)
    assert np.array_equal(cam, full)


def test_point_mask_from_bool_or_indices():
    b = np.zeros(10, bool)
    b[[1, 7]] = True
    _, pt = normalize_fixed(None, b, 3, 10)
    assert np.array_equal(pt, b)
    for idx in (np.array([7, 1]), np.array([1, 7, 7], dtype=np.int32), np.array([1, 7], dtype=np.uint16)):
        _, pt = normalize_fixed(None, idx, 3, 10)
        assert np.array_equal(pt, b), idx


def test_empty_masks_mean_nothing_held():
    """All-false masks and an empty index array leave the solve unmasked (None)."""
    assert normalize_fixed(None, None, 3, 10) == (None, None)
    assert normalize_fixed(np.zeros(11, bool), np.zeros(10, bool), 3, 10) == (None, None)
    assert normalize_fixed(np.zeros((3, 11), bool), np.array([], dtype=np.int64), 3, 10) == (None, None)


@pytest.mark.parametrize("cam,pt", [
    (np.zeros(10, bool), None),                       # neither (11,) nor (C, 11)
    (np.zeros((2, 11), bool), None),                  # wrong camera count
    (np.zeros((3, 11, 1), bool), None),
    (np.zeros(11, dtype=np.int64), None),             # not bool
    (np.zeros(11, dtype=np.float64), None),
    (None, np.zeros(9, bool)),                        # wrong point count
    (None, np.zeros((10, 1), bool)),
    (None, np.array([0, 10])),                        # index out of range
    (None, np.array([-1])),
    (None, np.array([[0, 1]])),                       # indices not 1-D
    (None, np.array([0.0, 1.0])),                     # neither bool nor integer
])
def test_bad_masks_raise_value_error(cam, pt):
    with pytest.raises(ValueError):
        normalize_fixed(cam, pt, 3, 10)


@pytest.mark.parametrize("name", ["ba_ring8_volume1500", "ba_ring4_planar2000", "ba_example18_vis60_800"])
def test_oracle_without_mask_reproduces_trf_exact(golden, name):
    """trf_exact_fixed with nothing held is trf_exact through trf_exact_generic (sparse LU of the full
    normal equations instead of the Schur complement): same decisions; costs to round-off amplified by
    the gauge modes (measured 1.5e-7 along the trajectory, 6.1e-9 at the end)."""
    g = golden(name)
    a = O.trf_exact(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"], ftol=1e-4)
    b = trf_exact_fixed(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"], ftol=1e-4)
    assert (a.nfev, a.njev, a.status) == (b.nfev, b.njev, b.status)
    np.testing.assert_allclose(b.trace, [r["cost"] for r in a.trace] + [a.cost], rtol=3e-7)
    np.testing.assert_allclose(b.cost, a.cost, rtol=1e-8)
    assert b.x.shape == a.x.shape and b.grad.shape == a.grad.shape


def test_oracle_holds_masked_entries(golden):
    """Held entries of x are the input's, bit for bit, and their gradient entries are 0."""
    g = golden("ba_example18_vis60_800")
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cm = np.zeros((C, 11), bool)
    cm[0, :6] = True
    cm[:, 9:] = True
    pm = np.zeros(P, bool)
    pm[[0, P // 3, 2 * P // 3]] = True
    r = trf_exact_fixed(g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"],
                        cam_fixed=cm, pt_fixed=pm, ftol=1e-4)
    x0 = np.hstack((g["cams0"].ravel(), g["pts0"].ravel()))
    held = np.concatenate([cm.ravel(), np.repeat(pm, 3)])
    assert np.array_equal(r.x[held], x0[held])
    assert np.all(r.grad[held] == 0.0)
    assert r.x_free.size == (~held).sum()
    assert r.cost < 0.5 * np.sum(O.fun(x0, C, P, g["camera_ind"], g["point_ind"], g["points_2d"],
                                       O.default_weights(g["point_ind"])) ** 2)
