"""Worker of tests/test_gpu_i8_scale.py::test_point_sharded_int8_path_matches_single_gpu (launched by
torchrun, one rank per GPU): two shards of ~40 k points, each large enough for the int8 tensor-core Schur
path, must reproduce the reduced camera system of the single-GPU run."""
import os
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

import torch  # noqa: E402

from lasercalib_b200 import dist as D  # noqa: E402
from lasercalib_b200._cabi import Engine  # noqa: E402
from lasercalib_b200.synth import make_rig  # noqa: E402

P = 80_000
LAM = 1e-5


def main():
    rank, ws, local = D.init_from_env()
    assert ws == 2
    torch.cuda.set_device(local)
    pb = make_rig("ring24", P + 2000, seed=43, variant="volume", p_vis=1.0)
    keep = pb["point_ind"] < P
    pts0, uv = pb["pts0"][:P].copy(), np.ascontiguousarray(pb["points_2d"][keep])
    ci, pi = pb["camera_ind"][keep].copy(), pb["point_ind"][keep].copy()
    # single-GPU reference on every rank's own device
    eng = Engine(local)
    eng.set_problem(pb["cams0"], pts0, uv, ci, pi)
    lin1 = eng.linearize(LAM)
    eng.close()
    # sharded: one solver iteration to read which kernels ran, then S at x0
    sh = D.shard_problem(pts0, uv, ci, pi, None, rank, ws)
    assert sh["pts"].shape[0] >= 32768, sh["pts"].shape
    e2 = Engine(local)
    e2.set_problem(pb["cams0"], sh["pts"], sh["points_2d"], sh["camera_ind"], sh["point_ind"], pt_offset=sh["pt_offset"])
    D.connect_engine(e2)
    e2.solve(max_iterations=1, profile=True)
    kernels = set(e2.profile())
    assert "i8_rowmax" in kernels, sorted(kernels)
    e2.set_params(pb["cams0"], sh["pts"])
    lin2 = e2.linearize(LAM)
    e2.close()
    eS = np.abs(lin2["S"] - lin1["S"]).max() / np.abs(lin1["S"]).max()
    er = np.abs(lin2["rhs"] - lin1["rhs"]).max() / np.abs(lin1["rhs"]).max()
    ec = abs(lin2["cost"] - lin1["cost"]) / abs(lin1["cost"])
    print("rank %d: %d points; S %.2e = %.3f of 1e-12, rhs %.2e = %.3f of 1e-11, cost %.2e = %.3f of 1e-13"
          % (rank, sh["pts"].shape[0], eS, eS / 1e-12, er, er / 1e-11, ec, ec / 1e-13))
    assert eS <= 1e-12 and er <= 1e-11 and ec <= 1e-13
    torch.distributed.barrier()
    torch.distributed.destroy_process_group()
    print("rank %d ok" % rank)


if __name__ == "__main__":
    main()
