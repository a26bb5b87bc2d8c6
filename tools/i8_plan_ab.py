"""A/B of two settings of the int8 Schur SYRK on one GPU, alternating inside one process: by default its two tile
plans (LCBA_I8_PLAN=strip,cover), or any other switch such as its two schedules (LCBA_I8_SCHED=range,kmajor).
Per round and setting, the device time of K solver iterations and the CUDA-event time of k_i8_syrk per launch
(the "schur" entry of the solver's profile), plus the card's name and power limit.

    python tools/i8_plan_ab.py OUT_DIR [rig] [points] [rounds] [steps] [VAR=a,b]

Writes OUT_DIR/i8_plan_ab.json (OUT_DIR/<var>_ab.json for another switch) and prints a summary (median and
range per setting)."""
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
    steps = int(sys.argv[5]) if len(sys.argv) > 5 else 20
    var, vals = (sys.argv[6] if len(sys.argv) > 6 else "LCBA_I8_PLAN=strip,cover").split("=")
    vals = tuple(vals.split(","))
    os.makedirs(out_dir, exist_ok=True)
    from lasercalib_b200._cabi import Engine
    from lasercalib_b200.synth import make_rig
    pb = make_rig(rig, points, seed=0, variant="volume", p_vis=1.0)
    tol = dict(ftol=1e-4, xtol=1e-8, gtol=1e-8, max_nfev=200)   # as bench.py

    def steps_ms(eng, k, profile):
        done, ms, prof = 0, 0.0, {}
        while done < k:
            eng.set_params(pb["cams0"], pb["pts0"])
            r, _ = eng.solve(max_iterations=k - done, profile=profile, **tol)
            done += int(r.iterations)
            ms += r.solve_ms
            if profile:
                for name, v in eng.profile().items():
                    a = prof.setdefault(name, [0, 0.0])
                    a[0] += v["launches"]
                    a[1] += v["total_ms"]
        return ms / done, prof

    res = dict(card=card(), rig=rig, points=points, n_obs=int(pb["n_obs"]), steps=steps, switch=var, runs=[])
    for rnd in range(rounds):
        for plan in (vals if rnd % 2 == 0 else vals[::-1]):
            os.environ[var] = plan
            eng = Engine()
            try:
                eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
                steps_ms(eng, 3, False)                              # warm-up
                ms_step, _ = steps_ms(eng, steps, False)
                _, prof = steps_ms(eng, steps, True)
            finally:
                eng.close()
            syrk = prof["schur"][1] / prof["schur"][0]
            res["runs"].append(dict(round=rnd, plan=plan, ms_per_step=ms_step, ms_k_i8_syrk=syrk,
                                    prof={k: v[1] / v[0] for k, v in prof.items()}))
            print("round %d %-5s: %.3f ms / step, k_i8_syrk %.3f ms / launch" % (rnd, plan, ms_step, syrk), flush=True)
    os.environ.pop(var)
    res["card_after"] = card()
    summary = {}
    for plan in vals:
        s = np.array([r["ms_per_step"] for r in res["runs"] if r["plan"] == plan])
        k = np.array([r["ms_k_i8_syrk"] for r in res["runs"] if r["plan"] == plan])
        summary[plan] = dict(ms_per_step_median=float(np.median(s)), ms_per_step_min=float(s.min()), ms_per_step_max=float(s.max()),
                             syrk_median=float(np.median(k)), syrk_min=float(k.min()), syrk_max=float(k.max()))
        print("%-5s: step %.3f ms (%.3f - %.3f), k_i8_syrk %.3f ms (%.3f - %.3f)" % (
            plan, summary[plan]["ms_per_step_median"], s.min(), s.max(), summary[plan]["syrk_median"], k.min(), k.max()))
    res["summary"] = summary
    print("card:", res["card"])
    name = "i8_plan_ab.json" if var == "LCBA_I8_PLAN" else var.lower() + "_ab.json"
    with open(os.path.join(out_dir, name), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
