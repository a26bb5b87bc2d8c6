"""Worker of tests/test_gpu_fixed_params.py (launched by torchrun, one rank per GPU): a point-sharded solve
with held parameters must reproduce the single-GPU masked solve, and ranks that hold different camera
entries must all fail."""
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
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    # held points at both ends of both shards and on each side of the cut
    sh = D.shard_problem(pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], None, rank, ws)
    cut = sh["hi"] if rank == 0 else sh["lo"]
    t = torch.tensor([cut], dtype=torch.int64, device="cuda")
    torch.distributed.broadcast(t, 0)
    cut = int(t.item())
    held = [0, 1, 2, cut - 3, cut - 2, cut - 1, cut, cut + 1, cut + 2, P - 1] + list(range(10, P, 97))
    pt = np.zeros(P, bool)
    pt[held] = True
    # one GPU, masked, on every rank's own device
    eng = Engine(local)
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    eng.set_fixed(cam, pt)
    res1, _ = eng.solve(ftol=1e-4)
    eng.close()
    # sharded through the drop-in API
    sba = PySBA(pb["cams0"].copy(), pb["pts0"].copy(), pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    res2 = sba.bundleAdjust(1e-4, verbose=0, fixed_camera_params=cam, fixed_points=pt)
    assert res2.nfev == res1.nfev and res2.status == res1.status, (res2.nfev, res1.nfev)
    np.testing.assert_allclose(res2.cost, res1.cost, rtol=1e-12)
    assert np.array_equal(sba.points3D[pt], pb["pts0"][pt])
    assert np.array_equal(sba.cameraArray[cam], pb["cams0"][cam])
    # different camera masks over the ranks: every rank fails
    e2 = Engine(local)
    e2.set_problem(pb["cams0"], sh["pts"], sh["points_2d"], sh["camera_ind"], sh["point_ind"], pt_offset=sh["pt_offset"])
    D.connect_engine(e2)
    bad = cam.copy()
    if rank == 1:
        bad[1, 6] = True
    e2.set_fixed(bad, pt[sh["lo"]:sh["hi"]])
    try:
        e2.solve(ftol=1e-4)
        raise AssertionError("rank %d: mismatched camera masks were accepted" % rank)
    except LcbaError as e:
        assert e.code == -1, e
    e2.close()
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    print("rank %d ok" % rank)


if __name__ == "__main__":
    main()
