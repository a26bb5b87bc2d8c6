"""Time lcba_covariance on ring24 x 1 M points (gauge held: camera 0's extrinsics and three points).

Everything is timed with CUDA events.  The whole call: two events on an otherwise idle stream, recorded right
before the call and right after it returns (it ends with a synchronise of the library's stream, so the pair
brackets the call, the copies of S^-1 and of the P x 6 point blocks to pageable host memory included).  The kernels:
a separate run with LCBA_COV_PROFILE=1, where the library brackets every launch of the call with CUDA events on its
own stream (lcba_get_profile): k_point_cov, with its rate on the triangular flop count 2 * n (n + 1) / 2 * 3 P
against the FP64 DMMA peak of 37.1 TFLOP/s (profiles/r01_fp64_peak.txt), k_chol_inverse and k_chol_inverse_gram.

usage: python tools/cov_time.py [--points 1000000] [--reps 5] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)

DMMA_PEAK = 37.1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rig", default="ring24")
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from lasercalib_b200._cabi import Engine
    from lasercalib_b200.synth import make_rig
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say("# card: " + q.stdout.strip().splitlines()[0] if q.returncode == 0 else "# card: unknown")
    pb = make_rig(a.rig, a.points, seed=0, variant="volume", p_vis=0.95)
    C, P = pb["n_cams"], pb["n_points"]
    n = 11 * C
    cam = np.zeros((C, 11), bool)
    cam[0, :6] = True
    pt = np.zeros(P, bool)
    pt[[0, P // 3, 2 * P // 3]] = True
    e = Engine()
    e.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    e.set_fixed(cam, pt)
    e.solve(ftol=1e-4)
    say("# %s x %d points, %d observations, %d cameras; Schur route: %s" %
        (a.rig, P, pb["camera_ind"].size, C, "int8" if e.i8_fell_back() != -1 else "DMMA/DFMA"))
    e.covariance()                                  # warm-up: buffers, modules
    ts = []
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(a.reps):
        torch.cuda.synchronize()
        t0.record()
        e.covariance()
        t1.record()
        t1.synchronize()
        ts.append(t0.elapsed_time(t1))
    say("lcba_covariance whole call (CUDA events around the call): median %.3f ms (min %.3f, max %.3f) over %d calls"
        % (np.median(ts), min(ts), max(ts), a.reps))
    os.environ["LCBA_COV_PROFILE"] = "1"
    k = {}
    for _ in range(a.reps):
        e.covariance()
        for name, st in e.profile().items():
            k.setdefault(name, []).append(st["total_ms"] / st["launches"])
    del os.environ["LCBA_COV_PROFILE"]
    e.close()
    flop = 2.0 * n * (n + 1) / 2 * 3 * P
    for name, kern in (("point_cov", "k_point_cov"), ("chol_inverse", "k_chol_inverse"),
                       ("chol_inverse_gram", "k_chol_inverse_gram")):
        v = k.get(name, [])
        if not v:
            say("%s: no record" % kern)
            continue
        ms = float(np.median(v))
        extra = ""
        if name == "point_cov":
            extra = ", %.2e flop (triangular), %.1f TFLOP/s = %.1f %% of %.1f" % (
                flop, flop / ms / 1e9, 100 * flop / ms / 1e9 / (DMMA_PEAK / 1e12), DMMA_PEAK / 1e12)
        say("%s (CUDA events, LCBA_COV_PROFILE=1): median %.3f ms over %d calls%s" % (kern, ms, len(v), extra))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
