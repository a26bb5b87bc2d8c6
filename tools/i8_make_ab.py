"""A/B of the digit-plane kernels of the int8 Schur path (schur_i8.cuh: k_i8_make and its reference
k_i8_make_ref) on one GPU, alternating inside one process through lcba_debug_i8_make: per round and kernel,
the CUDA-event time per launch over `reps` back-to-back launches (after one warm-up launch), plus the card's
name, power limit and maximum SM clock.  Only times the kernels: the planes (4.97 GB at ring24 x 1 M) are
not copied.

    python tools/i8_make_ab.py OUT_DIR [rig] [points] [rounds] [reps]

Writes OUT_DIR/i8_make_ab.json and prints a summary (median and range per kernel, and the plane write rate)."""
import json
import os
import subprocess
import sys

import numpy as np

sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return q.stdout.strip()
    except Exception as e:            # the numbers stay valid; only the label is missing
        return "unknown (%s)" % type(e).__name__


def main():
    out_dir = sys.argv[1]
    rig = sys.argv[2] if len(sys.argv) > 2 else "ring24"
    points = int(sys.argv[3]) if len(sys.argv) > 3 else 1_000_000
    rounds = int(sys.argv[4]) if len(sys.argv) > 4 else 4
    reps = int(sys.argv[5]) if len(sys.argv) > 5 else 20
    os.makedirs(out_dir, exist_ok=True)
    from lasercalib_b200._cabi import Engine, i8_plane_bytes
    from lasercalib_b200.synth import make_rig
    pb = make_rig(rig, points, seed=0, variant="volume", p_vis=1.0)
    C, P = pb["n_cams"], pb["n_points"]
    plane_bytes = i8_plane_bytes(C, P)
    os.environ["LCBA_SCHUR_I8"] = "1"
    res = dict(card=card(), rig=rig, points=P, n_obs=int(pb["n_obs"]), reps=reps, plane_bytes=plane_bytes, runs=[])
    eng = Engine()
    try:
        eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
        for ref in (False, True):
            eng.debug_i8_make(1e-5, ref=ref, reps=1, planes=False, poison=None)          # warm-up
        for rnd in range(rounds):
            for ref in ((False, True) if rnd % 2 == 0 else (True, False)):
                name = "k_i8_make_ref" if ref else "k_i8_make"
                ms, _ = eng.debug_i8_make(1e-5, ref=ref, reps=reps, planes=False, poison=None)
                res["runs"].append(dict(round=rnd, kernel=name, ms=ms, tb_s=plane_bytes / ms * 1e-9))
                print("round %d %-13s: %.3f ms / launch, %.2f TB/s" % (rnd, name, ms, plane_bytes / ms * 1e-9), flush=True)
    finally:
        eng.close()
    res["card_after"] = card()
    summary = {}
    for name in ("k_i8_make", "k_i8_make_ref"):
        t = np.array([r["ms"] for r in res["runs"] if r["kernel"] == name])
        summary[name] = dict(ms_median=float(np.median(t)), ms_min=float(t.min()), ms_max=float(t.max()),
                             tb_s_median=plane_bytes / float(np.median(t)) * 1e-9)
        print("%-13s: %.3f ms (%.3f - %.3f), %.2f TB/s" % (name, summary[name]["ms_median"], t.min(), t.max(),
                                                          summary[name]["tb_s_median"]))
    res["summary"] = summary
    print("card:", res["card"])
    with open(os.path.join(out_dir, "i8_make_ab.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
