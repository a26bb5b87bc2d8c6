"""A/B of held parameters (lcba_set_fixed) on the bench rig, one GPU, one process: per round, the same
K outer iterations of bundleAdjust(1e-4) from x0 with no mask, with the gauge mask (camera 0's extrinsics
and three points) and with the gauge mask plus 1 % of the points held, in alternation.  Device time per
iteration from lcba_result.solve_ms, the card's name, power limit and maximum SM clock read in the same run.

    python tools/fixed_ab.py OUT_FILE [rig] [points] [rounds] [steps]

Writes OUT_FILE (text) and prints it."""
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
    out = sys.argv[1]
    rig = sys.argv[2] if len(sys.argv) > 2 else "ring24"
    points = int(sys.argv[3]) if len(sys.argv) > 3 else 1_000_000
    rounds = int(sys.argv[4]) if len(sys.argv) > 4 else 5
    steps = int(sys.argv[5]) if len(sys.argv) > 5 else 20
    from lasercalib_b200._cabi import Engine
    from lasercalib_b200.synth import make_rig
    pb = make_rig(rig, points, seed=0, variant="volume", p_vis=1.0)
    C, P = pb["n_cams"], pb["n_points"]
    gauge = np.zeros((C, 11), bool)
    gauge[0, :6] = True
    pts3 = np.zeros(P, bool)
    pts3[[0, P // 3, 2 * P // 3]] = True
    pts1 = pts3 | (np.random.default_rng(0).random(P) < 0.01)
    modes = {"none": (None, None), "gauge": (gauge, pts3), "gauge+1%pts": (gauge, pts1)}
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])

    def run(mode, k):
        eng.set_fixed(*modes[mode])
        done, ms = 0, 0.0
        while done < k:
            eng.set_params(pb["cams0"], pb["pts0"])
            r, _ = eng.solve(ftol=1e-4, max_nfev=200, max_iterations=k - done)
            if r.iterations <= 0:
                raise RuntimeError("solver made no iteration")
            done += int(r.iterations)
            ms += r.solve_ms
        return ms / done

    for m in modes:
        run(m, 3)                      # warm-up: modules, graphs of every mode
    times = {m: [] for m in modes}
    for _ in range(rounds):
        for m in modes:
            times[m].append(run(m, steps))
    eng.close()
    base = np.median(times["none"])
    lines = ["# tools/fixed_ab.py %s x %d points, %d rounds x %d iterations per mode, alternating in one process"
             % (rig, points, rounds, steps),
             "# card (name, power limit, max SM clock): %s" % card(),
             "# device ms per outer iteration (lcba_result.solve_ms / iterations): median [min, max], vs no mask"]
    for m, t in times.items():
        med = np.median(t)
        lines.append("%-12s %.4f [%.4f, %.4f]  %+.2f %%" % (m, med, min(t), max(t), 100.0 * (med / base - 1.0)))
    lines.append("# per round: " + "; ".join("%s %s" % (m, " ".join("%.4f" % v for v in t)) for m, t in times.items()))
    text = "\n".join(lines) + "\n"
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(text)
    print(text, end="")


if __name__ == "__main__":
    main()
