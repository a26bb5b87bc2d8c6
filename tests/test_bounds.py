"""Box bounds of bundleAdjust without a GPU: the argument normalisation of PySBA.bundleAdjust(bounds=...) with
least_squares' error messages, and the CPU oracle of trf_bounds (tests/_bounds_oracle.py) against trf_exact and
against scipy's own least_squares(bounds=...)."""
import numpy as np
import pytest
from scipy.optimize import Bounds, least_squares
from scipy.optimize._lsq.common import make_strictly_feasible

from oracle import pysba_oracle as O
from lasercalib_b200.pySBA import normalize_bounds
from lasercalib_b200.synth import make_rig

from _bounds_oracle import trf_bounds_exact_generic, trf_bounds_fixed
from _fixed_oracle import _restricted, trf_exact_fixed

X0 = np.array([0.0, 1.0, 2.0, 3.0])


def test_bounds_forms_normalise_like_least_squares():
    lb, ub = normalize_bounds((0.0, 5.0), X0)
    assert lb.shape == ub.shape == X0.shape and np.all(lb == 0.0) and np.all(ub == 5.0)
    lb2, ub2 = normalize_bounds(Bounds(np.zeros(4), np.full(4, 5.0)), X0)
    assert np.array_equal(lb, lb2) and np.array_equal(ub, ub2)
    lb3, ub3 = normalize_bounds(([-1, 0, 0, 0], np.inf), X0)
    assert lb3.dtype == np.float64 and np.all(np.isposinf(ub3))
    # every bound infinite: the unbounded solve (scipy dispatches to trf_no_bounds)
    assert normalize_bounds(None, X0) is None
    assert normalize_bounds((-np.inf, np.inf), X0) is None


@pytest.mark.parametrize("bounds,msg", [
    ((0.0, 1.0, 2.0), "`bounds` must contain 2 elements."),
    ((np.zeros(3), 5.0), "Inconsistent shapes between bounds and `x0`."),
    ((0.0, np.full(5, 5.0)), "Inconsistent shapes between bounds and `x0`."),
    ((1.0, 1.0), "Each lower bound must be strictly less than each upper bound."),
    ((np.array([0.0, 0, 3, 0]), np.array([1.0, 2, 2, 4])), "Each lower bound must be strictly less than each"),
    ((0.5, 5.0), "Initial guess is outside of provided bounds"),
    ((-1.0, 2.5), "Initial guess is outside of provided bounds"),
])
def test_bad_bounds_raise_least_squares_messages(bounds, msg):
    with pytest.raises(ValueError, match=msg.replace("`", ".").replace("(", ".").replace(")", ".")):
        normalize_bounds(bounds, X0)
    # least_squares itself says the same
    with pytest.raises(ValueError, match=msg.replace("`", ".")):
        least_squares(lambda x: x - 1.0, X0, bounds=bounds)


def test_held_entries_are_not_checked():
    """With a mask, only free entries must satisfy lb < ub and lie in the box; all-infinite free bounds -> None."""
    held = np.array([True, False, False, False])
    lb = np.array([0.5, 0.0, 0.0, 0.0])
    ub = np.array([0.5, 5.0, 5.0, 5.0])
    out = normalize_bounds((lb, ub), X0, held)
    assert out is not None and np.array_equal(out[0], lb)
    assert normalize_bounds(([7.0, -np.inf, -np.inf, -np.inf], np.inf), X0, held) is None
    with pytest.raises(ValueError, match="Initial guess is outside"):
        normalize_bounds((0.5, 5.0), X0, ~held)


@pytest.mark.parametrize("name", ["ba_ring8_volume1500", "ba_ring4_planar2000", "ba_example18_vis60_800"])
def test_oracle_with_infinite_bounds_is_the_unbounded_oracle(golden, name):
    """+-inf bounds: trf_bounds reduces to trf_no_bounds (v = 1, diag_h = 0, every step inside).  Against
    trf_exact_fixed (the same sparse solve) with the gauge held: same nfev, njev, status and trace; x to 1e-12 of
    its scale (measured here: 0 to 4e-15)."""
    g = golden(name)
    C, P = g["cams0"].shape[0], g["pts0"].shape[0]
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    pt = np.zeros(P, bool)
    pt[[0, P // 3, 2 * P // 3]] = True
    args = (g["cams0"], g["pts0"], g["points_2d"], g["camera_ind"], g["point_ind"])
    a = trf_exact_fixed(*args, cam_fixed=cam, pt_fixed=pt, ftol=1e-4)
    b = trf_bounds_fixed(*args, -np.inf, np.inf, cam_fixed=cam, pt_fixed=pt, ftol=1e-4)
    assert (a.nfev, a.njev, a.status) == (b.nfev, b.njev, b.status)
    np.testing.assert_allclose([r["cost"] for r in b.rows], a.trace, rtol=1e-12)
    assert np.abs(a.x - b.x).max() <= 1e-12 * np.abs(a.x).max()
    assert set(b.choices) == {"p"} and not b.active_mask.any()


def _small_rig(seed):
    """A 60-point ring4 rig with camera 0's extrinsics and three points held (no gauge freedom, so that LSMR and
    the exact solve reach the same steps): x0, fun and jac over the free entries, and their indices."""
    pb = make_rig("ring4", 60, seed=seed, variant="volume")
    C, P = pb["cams0"].shape[0], pb["pts0"].shape[0]
    ci, pi, p2 = pb["camera_ind"], pb["point_ind"], pb["points_2d"]
    w = O.default_weights(pi).reshape(-1, 1)
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))

    def fun(x):
        return O.fun(x, C, P, ci, pi, p2, w)

    def jac(x, *_):
        _, Jc, Jp = O.jacobian_blocks(x[:11 * C].reshape(C, 11), x[11 * C:].reshape(P, 3), ci, pi, w)
        return O.jacobian_csr(Jc, Jp, C, P, ci, pi)

    held = np.zeros(x0.size, dtype=bool)
    held[:6] = True
    held[11 * C + np.repeat(3 * np.array([0, P // 3, 2 * P // 3]), 3) + np.tile(np.arange(3), 3)] = True
    free = np.flatnonzero(~held)
    fun_x, jac_x = _restricted(fun, jac, x0, free)
    return pb, C, P, x0[free], fun_x, lambda x, *_: jac_x(x), free


def _binding_box(pb, C, P, kind):
    n = 11 * C + 3 * P
    lb, ub = np.full(n, -np.inf), np.full(n, np.inf)
    c0 = pb["cams0"]
    lc, uc = lb[:11 * C].reshape(C, 11), ub[:11 * C].reshape(C, 11)
    if "k" in kind:
        lc[:, 7], uc[:, 7] = c0[:, 7] - 2e-4, c0[:, 7] + 2e-4
        lc[:, 8], uc[:, 8] = c0[:, 8] - 1e-3, c0[:, 8] + 1e-3
    if "f" in kind:
        uc[:, 6] = c0[:, 6] + 0.5
    if "z" in kind:
        lb[11 * C + 2::3] = pb["pts0"][:, 2].min()
    return lb, ub


RIGS = [(0, "k"), (1, "kf"), (2, "kz"), (3, "kfz"), (4, "k")]


# cost of the oracle against scipy's LSMR-based trf_bounds with tight LSMR tolerances, measured on a CPU: <= 8.6e-14
SCIPY_COST_RTOL = 1e-11


@pytest.mark.parametrize("seed,kind", RIGS)
def test_oracle_matches_scipy_trf_bounds(seed, kind):
    """The oracle (exact augmented solve) against least_squares(bounds=..., x_scale='jac', tr_solver='lsmr') with an
    analytic CSR Jacobian and tight LSMR tolerances on small rigs with binding k1/k2, f and z bounds: same status, nfev
    and njev; cost to SCIPY_COST_RTOL."""
    pb, C, P, x0, fun, jac, free = _small_rig(seed)
    lb, ub = (b[free] for b in _binding_box(pb, C, P, kind))
    ref = least_squares(fun, x0, jac=jac, bounds=(lb, ub), x_scale="jac", method="trf", tr_solver="lsmr",
                        tr_options=dict(atol=1e-15, btol=1e-15, maxiter=10000), ftol=1e-4)
    ora = trf_bounds_exact_generic(fun, jac, x0, lb, ub, 1e-4)
    assert (ora.status, ora.nfev, ora.njev) == (ref.status, ref.nfev, ref.njev)
    np.testing.assert_allclose(ora.cost, ref.cost, rtol=SCIPY_COST_RTOL)
    assert np.array_equal(ora.active_mask, ref.active_mask)


def test_rig_set_reaches_every_branch_and_binds():
    """Over the rigs above, select_step chooses the subspace step, the reflection and the anti-gradient, and the
    solves end with entries on their bounds."""
    seen, active = set(), 0
    for seed, kind in RIGS:
        pb, C, P, x0, fun, jac, free = _small_rig(seed)
        lb, ub = (b[free] for b in _binding_box(pb, C, P, kind))
        ora = trf_bounds_exact_generic(fun, jac, x0, lb, ub, 1e-4)
        seen |= set(ora.choices)
        active += np.count_nonzero(ora.active_mask)
    assert seen == {"p", "r", "ag"}, seen
    assert active > 0


def test_x0_on_a_bound_is_moved_strictly_inside():
    """An x0 exactly on a bound starts from make_strictly_feasible(x0, lb, ub) (rstep = 1e-10)."""
    pb, C, P, x0, fun, jac, free = _small_rig(0)
    lb, ub = (b[free] for b in _binding_box(pb, C, P, "z"))
    i = int(np.flatnonzero(free == 11 * C + 2 + 3 * int(np.argmin(pb["pts0"][:, 2])))[0])
    assert x0[i] == lb[i]
    seen = []

    def fun_rec(x):
        seen.append(x.copy())
        return fun(x)

    trf_bounds_exact_generic(fun_rec, jac, x0, lb, ub, 1e-4, max_nfev=1)
    moved = make_strictly_feasible(x0, lb, ub)
    assert seen[0][i] == lb[i] + 1e-10 * max(1.0, abs(lb[i])) == moved[i]
    assert np.array_equal(np.delete(seen[0], i), np.delete(x0, i))
