"""A/B of box bounds (lcba_set_bounds) on the bench rig, one GPU, one process: per round, the same K outer
iterations of the solve (ftol 1e-4) from x0 unbounded, with finite bounds that never bind (x0 -+ 1e6 max(1, |x0|):
the bounded loop, whose reflection pass finds every step inside the box and returns at once) and with binding
bounds (k1 and k2 within 1e-6 of x0, every point at most 1e-3 below its initial z), in alternation.  Device
time per iteration from lcba_result.solve_ms, trials per iteration (nfev / iterations), entries on a bound at
the end, and the card's name, power limit and maximum SM clock read in the same run.

    python tools/bounds_ab.py OUT_FILE [rig] [points] [rounds] [steps]

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
    x0 = np.hstack((pb["cams0"].ravel(), pb["pts0"].ravel()))
    nc = 11 * C
    loose = (x0 - 1e6 * np.maximum(1.0, np.abs(x0)), x0 + 1e6 * np.maximum(1.0, np.abs(x0)))
    lb, ub = np.full(x0.size, -np.inf), np.full(x0.size, np.inf)
    for a in (7, 8):                   # k1, k2 of every camera
        lb[a:nc:11], ub[a:nc:11] = x0[a:nc:11] - 1e-6, x0[a:nc:11] + 1e-6
    lb[nc + 2::3] = x0[nc + 2::3] - 1e-3
    modes = {"unbounded": None, "never-binding": loose, "binding": (lb, ub)}
    eng = Engine()
    eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
    trials = {m: [0, 0] for m in modes}
    active = {}

    def run(mode, k):
        b = modes[mode]
        if b is None:
            eng.set_bounds()
        else:
            eng.set_bounds(b[0][:nc].reshape(C, 11), b[1][:nc].reshape(C, 11), b[0][nc:].reshape(P, 3),
                           b[1][nc:].reshape(P, 3))
        done, ms = 0, 0.0
        while done < k:
            eng.set_params(pb["cams0"], pb["pts0"])
            r, _ = eng.solve(ftol=1e-4, max_nfev=200, max_iterations=k - done)
            if r.iterations <= 0:
                raise RuntimeError("solver made no iteration")
            done += int(r.iterations)
            ms += r.solve_ms
            trials[mode][0] += int(r.nfev) - 1
            trials[mode][1] += int(r.iterations)
        active[mode] = int(np.count_nonzero(eng.active_mask(1e-8)))
        return ms / done

    for m in modes:
        run(m, 3)                      # warm-up: modules, graphs of every mode
    times = {m: [] for m in modes}
    for _ in range(rounds):
        for m in modes:
            times[m].append(run(m, steps))
    eng.close()
    base = np.median(times["unbounded"])
    lines = ["# tools/bounds_ab.py %s x %d points, %d rounds x %d iterations per mode, alternating in one process"
             % (rig, points, rounds, steps),
             "# card (name, power limit, max SM clock): %s" % card(),
             "# device ms per outer iteration (lcba_result.solve_ms / iterations): median [min, max], vs unbounded;"
             " trials per iteration; entries on a bound after the last run"]
    for m, t in times.items():
        med = np.median(t)
        lines.append("%-14s %.4f [%.4f, %.4f]  %+.2f %%  %.3f trials/it  %d active"
                     % (m, med, min(t), max(t), 100.0 * (med / base - 1.0), trials[m][0] / max(1, trials[m][1]),
                        active[m]))
    lines.append("# per round: " + "; ".join("%s %s" % (m, " ".join("%.4f" % v for v in t)) for m, t in times.items()))
    text = "\n".join(lines) + "\n"
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        f.write(text)
    print(text, end="")


if __name__ == "__main__":
    main()
