"""Worker of tests/test_gpu_covariance.py (launched by torchrun, one rank per GPU): the point-sharded covariance
must equal the single-GPU one, and a gauge-free sharded call must fail on every rank."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from lasercalib_b200 import dist as D  # noqa: E402
from lasercalib_b200._cabi import Engine  # noqa: E402
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
    pt = np.zeros(P, bool)
    pt[[0, P // 3, 2 * P // 3, P // 2, P // 2 + 1]] = True
    # one GPU on every rank's own device
    eng = Engine(local)
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    eng.set_fixed(cam, pt)
    eng.solve(ftol=1e-4)
    cams1, pts1 = eng.get_params()
    cam_cov1, pt6, cost1, piv1 = eng.covariance()
    eng.close()
    # sharded through the drop-in API at the same x
    sba = PySBA(cams1.copy(), pts1.copy(), pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    r = sba.covariance(fixed_camera_params=cam, fixed_points=pt, absolute_sigma=True)
    s = np.sqrt(np.diag(cam_cov1))
    s[s == 0] = 1.0
    e_cam = np.abs((r.camera_cov - cam_cov1) / np.outer(s, s)).max()
    iu = np.array([[0, 1, 2], [1, 3, 4], [2, 4, 5]])
    ref_pt = pt6[:, iu]
    d = np.sqrt(np.einsum("paa->pa", ref_pt))
    d[d == 0] = 1.0
    e_pt = np.abs((r.point_cov - ref_pt) / (d[:, :, None] * d[:, None, :])).max()
    assert e_cam <= 1e-10 and e_pt <= 1e-10, (e_cam, e_pt)
    np.testing.assert_allclose(r.cost, cost1, rtol=1e-12)
    # the ranks sum S from their shards' partials in another order than one GPU does: equal up to rounding
    np.testing.assert_allclose(r.min_pivot, piv1, rtol=1e-10)
    assert np.all(r.point_cov[pt] == 0.0)
    # gauge free: every rank refuses
    try:
        sba.covariance()
        raise AssertionError("rank %d: a gauge-free covariance was accepted" % rank)
    except np.linalg.LinAlgError as e:
        assert "singular" in str(e), e
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    print("rank %d ok e_cam %.2e e_pt %.2e" % (rank, e_cam, e_pt))


if __name__ == "__main__":
    main()
