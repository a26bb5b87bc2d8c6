"""Worker of tests/test_gpu_bounds.py (launched by torchrun, one rank per GPU): a point-sharded bounded solve must
reproduce the single-GPU bounded solve, with bounded points on both sides of the shard cut; ranks that hold
different camera bounds must all fail; a rank without bounds joins the bounded loop of a rank that has some."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from lasercalib_b200 import dist as D  # noqa: E402
from lasercalib_b200._cabi import Engine, LcbaError  # noqa: E402
from lasercalib_b200.pySBA import PySBA  # noqa: E402
from lasercalib_b200.synth import make_rig  # noqa: E402


def main():
    rank, ws, local = D.init_from_env()
    assert ws == 2
    torch.cuda.set_device(local)
    pb = make_rig("ring24", 20000, seed=3, variant="volume", p_vis=0.95)
    C, P = pb["n_cams"], pb["n_points"]
    nc = 11 * C
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    pt = np.zeros(P, bool)
    pt[[0, P // 3, 2 * P // 3]] = True
    sh = D.shard_problem(pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], None, rank, ws)
    cut = sh["hi"] if rank == 0 else sh["lo"]
    t = torch.tensor([cut], dtype=torch.int64, device="cuda")
    torch.distributed.broadcast(t, 0)
    cut = int(t.item())
    # k1, k2 of every camera within 1e-6 of x0; points within 1e-3 below their initial z around the cut and
    # every 13th point elsewhere
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    lb, ub = np.full(x0.size, -np.inf), np.full(x0.size, np.inf)
    for a in (7, 8):
        lb[a:nc:11], ub[a:nc:11] = x0[a:nc:11] - 1e-6, x0[a:nc:11] + 1e-6
    bp = np.zeros(P, bool)
    bp[max(0, cut - 200):cut + 200] = True
    bp[::13] = True
    lb[nc + 2 + 3 * np.flatnonzero(bp)] = pb["pts0"][bp, 2] - 1e-3
    # one GPU, bounded, on every rank's own device
    eng = Engine(local)
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    eng.set_fixed(cam, pt)
    eng.set_bounds(lb[:nc].reshape(C, 11), ub[:nc].reshape(C, 11), lb[nc:].reshape(P, 3), ub[nc:].reshape(P, 3))
    res1, _ = eng.solve(ftol=1e-4)
    x1 = np.hstack([a.ravel() for a in eng.get_params()])
    eng.close()
    # sharded through the drop-in API (bundleAdjust slices the point bounds per rank)
    sba = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    res2 = sba.bundleAdjust(1e-4, verbose=0, fixed_camera_params=cam, fixed_points=pt, bounds=(lb, ub))
    assert res2.nfev == res1.nfev and res2.status == res1.status, (res2.nfev, res1.nfev)
    np.testing.assert_allclose(res2.cost, res1.cost, rtol=1e-12)
    assert np.abs(res2.x - x1).max() <= 1e-9 * np.abs(x1).max()
    assert np.all((res2.x >= lb) & (res2.x <= ub))
    assert res2.active_mask.shape == x0.shape
    # different camera bounds over the ranks: every rank fails
    e2 = Engine(local)
    e2.set_problem(pb["cams0"], sh["pts"], sh["points_2d"], sh["camera_ind"], sh["point_ind"], pt_offset=sh["pt_offset"])
    D.connect_engine(e2)
    lo, hi = sh["lo"], sh["hi"]
    bad = ub[:nc].copy()
    if rank == 1:
        bad[11 + 7] += 1e-6
    e2.set_bounds(lb[:nc].reshape(C, 11), bad.reshape(C, 11), lb[nc:].reshape(P, 3)[lo:hi], ub[nc:].reshape(P, 3)[lo:hi])
    try:
        e2.solve(ftol=1e-4)
        raise AssertionError("rank %d: mismatched camera bounds were accepted" % rank)
    except LcbaError as e:
        assert e.code == -1, e
    # point bounds on rank 0 only, none on rank 1: both ranks run the bounded loop and agree
    e2.set_params(pb["cams0"], sh["pts"])
    if rank == 0:
        e2.set_bounds(None, None, lb[nc:].reshape(P, 3)[lo:hi], None)
    else:
        e2.set_bounds()
    r3, _ = e2.solve(ftol=1e-4)
    assert r3.status > 0
    v = torch.tensor([r3.cost, float(r3.nfev)], dtype=torch.float64, device="cuda")
    w = v.clone()
    torch.distributed.broadcast(w, 0)
    assert torch.equal(v, w), (v, w)
    pts3 = e2.get_params()[1]
    if rank == 0:
        assert np.all(pts3[:, 2] >= lb[nc:].reshape(P, 3)[lo:hi, 2])
    e2.close()
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    print("rank %d ok" % rank)


if __name__ == "__main__":
    main()
