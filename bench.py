#!/usr/bin/env python
"""Benchmark of the bundle-adjustment hot path (BASELINE.json metric: LM iterations/s and
residual+Jacobian observations/s on the 24-camera x 1 M-point rig, 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W            # this engine (default: config 3)
    python bench.py --config {1,2,3,4,5} ...                 # BASELINE.json configs[config-1]
    python bench.py --impl reference --steps K --warmup W    # CPU path (scipy least_squares)
    python bench.py ... --dump-outputs DIR                   # also save the last timed step's results

A step is ONE trust-region (LM) outer iteration over the whole observation set:
linearise -> reduced camera system -> Cholesky -> back-substitution -> trial cost ->
on-device accept/reject (reference equivalent: one pass of scipy trf.py:465-578).
N > 1 shards the SAME problem by point (strong scaling, NCCL all-reduce of the reduced
camera system); launch with torchrun (RANK/LOCAL_RANK/WORLD_SIZE in the env).
Prints one JSON line on rank 0.

--dump-outputs DIR writes, after the timed steps of the headline workload, what the last of them
handed back to its caller, as float64 .npy files: cameras.npy (C x 11), points3d.npy (P x 3),
cost.npy and optimality.npy.  The inputs depend on the arguments only (seeded), so two builds run
with the same arguments can be compared file for file.  The files stay under DUMP_MAX_BYTES: above
that, points3d.npy holds a fixed seeded sample of the rows, listed in points3d_rows.npy.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

# the bench may run from a read-only checkout and must leave the tree as it found it
sys.dont_write_bytecode = True
REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

METRIC = "LM_iters_per_sec"
UNIT = "iter/s"
FP64_PEAK_FALLBACK_TFLOPS = 37.1   # highest FP64 rate measured on this pool (profiles/r01_fp64_peak.txt)
HBM_FALLBACK_GBS = 6650.0          # B200_PROFILING.md fallback
BF16_FALLBACK_TFLOPS = 1590.0      # B200_PROFILING.md fallback

# BASELINE.json configs (1-based like the verdict): rig, points, visibility, variant
CONFIGS = {
    1: dict(rig="ring4", points=10_000, pvis=1.0, what="4-camera rig, 10k laser points (the reference's own CPU-runnable case)"),
    2: dict(rig="example18", points=200_000, pvis=1.0, what="18-camera rig in the example/config.json layout, 200k laser points"),
    3: dict(rig="ring24", points=1_000_000, pvis=1.0, what="24-camera rig, 1M laser points"),
    4: dict(rig="wide8", points=2_000_000, pvis=1.0, what="8-camera 65MP wide-angle rig (scripts/65MP.py geometry), 2M points"),
    5: dict(rig="ring64", points=10_000_000, pvis=0.5, what="64-camera rig, 10M points, p_vis 0.5 (8 GPUs)"),
}
N_CAMS = {"ring4": 4, "example18": 18, "ring24": 24, "wide8": 8, "ring64": 64, "ring8": 8}
DUMP_MAX_BYTES = 64_000_000


def load_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": HBM_FALLBACK_GBS, "bf16_tflops": BF16_FALLBACK_TFLOPS}, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU with NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.01)
        except Exception as e:  # NVML missing: report that, never fail the bench
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def pinned(a):
    """Copy a numpy array into page-locked host memory (returns a numpy view of it)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t.numpy(), t


def dump_outputs(directory, cams, pts, cost, optimality):
    """Write the solver's results as float64 .npy files (see the module docstring)."""
    os.makedirs(directory, exist_ok=True)
    out = {"cameras": np.asarray(cams, dtype=np.float64), "cost": np.array([cost], dtype=np.float64),
           "optimality": np.array([optimality], dtype=np.float64)}
    pts = np.asarray(pts, dtype=np.float64)
    room = DUMP_MAX_BYTES - 5 * 128 - sum(a.nbytes for a in out.values())     # 128-byte .npy headers
    if pts.nbytes > room:
        # each sampled row costs 3 coordinates + its row number
        rows = np.sort(np.random.default_rng(0).choice(pts.shape[0], room // (4 * 8), replace=False))
        out["points3d_rows"] = rows.astype(np.float64)
        pts = pts[rows]
    out["points3d"] = pts
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def workload_string(cfg_id, rig, points, pvis):
    return "%s: %d cameras x %d laser points, p_vis=%.2f, volume variant, seed 0 (BASELINE.json configs[%d])" \
        % (rig, N_CAMS.get(rig, 0), points, pvis, cfg_id - 1)


def schur_flops(k_hist_counts, n_obs):
    """Algorithmic FP64 flop of one Schur launch (SURVEY.md 8d): per point with k views
    2*363*k(k+1)/2 (S update, lower triangle) + 2*99*k (W V^-1) + 2*33*k (rhs), plus
    ~300 flop/observation of model + Jacobian."""
    k = np.arange(k_hist_counts.size, dtype=np.float64)
    per_point = 726.0 * k * (k + 1) / 2 + 198.0 * k + 66.0 * k
    return float(np.sum(per_point * k_hist_counts) + 300.0 * n_obs)


def _sha16(path):
    import hashlib
    with open(path, "rb") as f:
        return hashlib.sha256(f.read()).hexdigest()[:16]


def i8_ops(C, P):
    """int8 tensor work of one k_i8_syrk launch (schur_i8.cuh): (algorithmic, executed) in ops (1 MAC = 2).
    Algorithmic: the 26 digit products (i + j <= 6) of the lower triangle of the (11C+1)-row SYRK over
    K = 3 P.  Executed: what the tile plan issues (128-row tiles, upper parts of diagonal tiles, padding
    rows, 64 kappa per 21 points), restated from make_i8_plan."""
    R = 11 * C + 1
    alg = 26 * 2.0 * 3.0 * P * R * (R + 1) / 2
    nrg = (R + 7) // 8
    nrg += nrg & 1
    nmt = (nrg + 15) // 16
    last_m = nrg - 16 * (nmt - 1)
    fold = nmt > 1 and last_m <= 4
    nfull = nmt - 1 if fold else nmt
    cols = 0
    for mt in range(nfull):
        m0, mn = 16 * mt, min(16, nrg - 16 * mt)
        cols += 8 * (m0 + mn)                      # all column tiles of this row tile (block 1)
        if fold:
            cols += 8 * last_m                     # + the folded left-over rows as column block 2
    if fold:
        cols += 8 * last_m                         # corner tile
    kpad = -(-P // 21) * 64
    return alg, 26 * 2.0 * 128 * cols * kpad


def cpu_reference_run(rig, n_points, p_vis, n_full):
    """The reference CPU path (oracle.bundle_adjust == PySBA.bundleAdjust through scipy
    least_squares: TRF + 3-point FD Jacobian + LSMR, pySBA.py:141-142) with the reference's OWN
    tolerances, bundleAdjust(1e-4), run to termination on a bounded sample of the workload.
    iterations = nfev - 1; cores = measured cpu time / wall time of the call."""
    from lasercalib_b200.synth import make_rig
    from oracle import pysba_oracle as O
    pb = make_rig(rig, n_points, seed=0, variant="volume", p_vis=p_vis)
    t0, c0 = time.perf_counter(), time.process_time()
    res = O.bundle_adjust(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], ftol=1e-4)[0]
    dt, cpu = time.perf_counter() - t0, time.process_time() - c0
    iters = max(1, int(res.nfev) - 1)
    it_s_sample = iters / dt
    n_sample = pb["n_obs"]
    return dict(value=it_s_sample * n_sample / n_full, unit=UNIT, cores=round(cpu / dt, 2), kind="port",
                sample="%s rig, %d points (%d obs): bundleAdjust(1e-4) = %d outer iterations (nfev %d, status %d) in "
                       "%.1f s = %.4f iter/s; scaled linearly in observations to %d obs%s" %
                       (rig, pb["n_points"], n_sample, iters, int(res.nfev), int(res.status), dt, it_s_sample, n_full,
                        "" if n_sample < n_full else " (the full workload: no extrapolation)"),
                host_cpus=os.cpu_count(), sample_iters_per_s=it_s_sample, sample_obs=n_sample,
                sample_seconds=dt, extrapolated=bool(n_sample < n_full))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=sorted(CONFIGS))
    ap.add_argument("--rig", default=None)
    ap.add_argument("--points", type=int, default=None)
    ap.add_argument("--pvis", type=float, default=None)
    ap.add_argument("--cpu-points", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs saves the results of this engine's timed steps; --impl reference has none")
    K, W = args.steps, max(args.warmup, 0)
    cfg = dict(CONFIGS[args.config])
    rig = args.rig or cfg["rig"]
    points = args.points or cfg["points"]
    pvis = cfg["pvis"] if args.pvis is None else args.pvis

    rank = int(os.environ.get("RANK", "0"))
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    workload = workload_string(args.config, rig, points, pvis)

    from lasercalib_b200.synth import make_rig

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        full = make_rig(rig, points, seed=0, variant="volume", p_vis=pvis)
        C, P, n_full = full["n_cams"], full["n_points"], full["n_obs"]
        del full
        cpu_pts = args.cpu_points or (points if points <= 20_000 else 20_000)
        cb = cpu_reference_run(rig, cpu_pts, pvis, n_full)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT,
                "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": 1e3 / cb["value"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload, "n_cams": C, "n_points": P, "n_obs": n_full,
                           "mean_views_per_point": n_full / P, "parallelism": "host cores (scipy least_squares)",
                           "solver": "scipy TRF + 3-point FD Jacobian + LSMR, bundleAdjust(1e-4) to termination"},
                "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ this engine
    import torch
    from lasercalib_b200 import dist as D
    from lasercalib_b200._cabi import Engine
    from lasercalib_b200.pySBA import PySBA
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback; use --impl reference)")
    rank, ws, local = D.init_from_env()
    if ws == 1:
        local = 0
    torch.cuda.set_device(local)
    import torch.distributed as tdist

    def barrier():
        torch.cuda.synchronize()
        if ws > 1:
            tdist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if ws == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        return float(t.item())

    peaks, peak_src = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", HBM_FALLBACK_GBS))
    bf16_peak = float(peaks.get("bf16_tflops", BF16_FALLBACK_TFLOPS))
    fp64_peak = FP64_PEAK_FALLBACK_TFLOPS
    tol = dict(ftol=1e-4, xtol=1e-8, gtol=1e-8, max_nfev=200)

    def device_run(pb, k_steps, w_steps, sample_clocks=False, per_kernel=True, keep_params=False):
        """Device-resident rate of `k_steps` real outer iterations (bundleAdjust(1e-4) from the standard
        perturbed x0, repeated from x0 until k_steps are done), plus per-kernel CUDA-event times.
        keep_params: also return the parameters the last timed step left (this rank's points)."""
        sh = D.shard_problem(pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"], None, rank, ws)
        eng = Engine(local)
        eng.set_problem(pb["cams0"], sh["pts"], sh["points_2d"], sh["camera_ind"], sh["point_ind"],
                        pt_offset=sh["pt_offset"])
        if ws > 1:
            D.connect_engine(eng)

        def run_steps(k, profile=False):
            done, ms, launches, last = 0, 0.0, 0, None
            prof = {}
            while done < k:
                eng.set_params(pb["cams0"], sh["pts"])
                r, _ = eng.solve(max_iterations=k - done, profile=profile, **tol)
                if r.iterations <= 0:
                    raise RuntimeError("solver made no iteration")
                done += int(r.iterations)
                ms += r.solve_ms
                launches += int(r.gpu_launches)
                last = r
                if profile:
                    for kname, v in eng.profile().items():
                        a = prof.setdefault(kname, dict(launches=0, total_ms=0.0))
                        a["launches"] += v["launches"]
                        a["total_ms"] += v["total_ms"]
            return done, ms, launches, last, prof

        if w_steps > 0:
            run_steps(w_steps)
        sampler = ClockSampler(local) if (rank == 0 and sample_clocks) else None
        barrier()
        if sampler:
            sampler.start()
        steps_done, dev_ms, launches, res, _ = run_steps(k_steps)
        barrier()
        clocks = sampler.stop() if sampler else None
        total_ms = max_over_ranks(dev_ms)
        out = dict(steps=steps_done, ms_per_step=total_ms / max(1, steps_done), launches=launches,
                   final_cost=res.cost, optimality=res.optimality, nfev=int(res.nfev), clocks=clocks, shard=sh,
                   engine=eng, prof={})
        if keep_params:     # before the profiled pass below restarts from x0
            out["params"] = eng.get_params()
        if per_kernel:
            barrier()
            out["prof"] = run_steps(k_steps, profile=True)[4]
            barrier()
        return out

    def rooflines(pb, sh, run, eng):
        """roofline of the dominant kernel (the Schur step) and of the HBM-bound M1 kernel."""
        prof = run["prof"]
        C, N = pb["n_cams"], pb["n_obs"]
        n_loc, p_loc = sh["point_ind"].size, sh["pts"].shape[0]
        k_loc = np.bincount(np.bincount(sh["point_ind"] - sh["pt_offset"], minlength=p_loc))
        ms_jac = max_over_ranks(eng.time_device(1, 10))
        ms_res = max_over_ranks(eng.time_device(0, 10))
        roof = None
        if "schur" in prof:
            per = lambda name: prof[name]["total_ms"] / prof[name]["launches"] if name in prof else 0.0  # noqa: E731
            ms_schur, ms_y, ms_u = per("schur"), per("make_Y"), per("cam_normal")
            ms_rm = 2.0 * per("i8_rowmax")                       # k_i8_rowmax + k_i8_rowexp per Schur pass
            fl = schur_flops(k_loc, n_loc)
            kern_total = sum(v["total_ms"] for v in prof.values())
            helpers = ms_y + ms_u + ms_rm
            share = sum(prof[n]["total_ms"] for n in ("schur", "make_Y", "cam_normal", "i8_rowmax") if n in prof) / kern_total
            if "i8_rowmax" in prof:
                alg, exe = i8_ops(C, p_loc)
                peak = 2.0 * bf16_peak
                roof = {"kernel": "k_i8_syrk (tcgen05.mma kind::i8; helpers k_i8_make + k_i8_rowmax)",
                        "bound": "tensor", "precision": "int8 digit planes, exact int32 accumulation, FP64 recombination",
                        "achieved": alg / ms_schur * 1e-9, "peak": peak, "unit": "TFLOP/s",
                        "frac": alg / ms_schur * 1e-9 / peak, "traffic": None,
                        "ops": "int8 tensor ops (1 multiply-add = 2): 26 digit products x lower triangle x 3 P",
                        "ops_per_launch": alg, "executed_ops_per_launch": exe,
                        "executed_frac": exe / ms_schur * 1e-9 / peak, "ms_per_launch": ms_schur,
                        "ms_k_schur": ms_schur, "ms_helpers": helpers, "ms_k_make_Y": ms_y, "ms_k_rowmax": ms_rm,
                        "fp64_flop_per_launch": fl,
                        "fp64_equivalent_tflops_kernel": fl / ms_schur * 1e-9,
                        "fp64_equivalent_tflops_step": fl / (ms_schur + helpers) * 1e-9,
                        "fp64_equivalent_frac_of_fp64_peak": fl / (ms_schur + helpers) * 1e-9 / fp64_peak,
                        "share_of_step": share,
                        "peak_source": "%s (MEASURED_PEAKS.json bf16_tflops %.1f) x 2: dense int8 runs at twice the "
                                       "bf16 tensor rate (nominal 4500 vs 2250 TFLOP/s)" % (peak_src, bf16_peak)}
            else:
                mma = "make_Y" in prof
                roof = {"kernel": "k_schur_mma (+ k_make_Y)" if mma else "k_schur",
                        "bound": "tensor" if mma else "fp64", "precision": "fp64",
                        "achieved": fl / (ms_schur + helpers) * 1e-9, "peak": fp64_peak, "unit": "TFLOP/s",
                        "frac": fl / (ms_schur + helpers) * 1e-9 / fp64_peak, "traffic": None,
                        "flop_per_launch": fl, "ms_per_launch": ms_schur + helpers, "ms_k_schur": ms_schur,
                        "ms_helpers": helpers, "ms_k_make_Y": ms_y,
                        "frac_k_schur_alone": fl / ms_schur * 1e-9 / fp64_peak, "share_of_step": share,
                        "peak_source": "FP64 DMMA (mma.sync m8n8k4) / DFMA microbenchmarks on this pool "
                                       "(tools/fp64_peak.cu, profiles/r01_fp64_peak.txt): 37.1 TFLOP/s"}
        jac_bytes = 264.0 * n_loc + 24.0 * p_loc
        roof_m1 = {"kernel": "k_jacobian_blocks", "bound": "hbm", "achieved": jac_bytes / ms_jac * 1e-6,
                   "peak": hbm_peak, "unit": "GB/s", "frac": jac_bytes / ms_jac * 1e-6 / hbm_peak,
                   "traffic": None, "bytes_per_launch": jac_bytes, "ms_per_launch": ms_jac,
                   "obs_per_s": N / ms_jac * 1e3, "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs)"}
        try:   # dram bytes per launch from the committed `ncu --set full` capture of THIS kernel set and workload
            with open(os.path.join(REPO, "profiles", "r02_traffic.json")) as f:
                tr = json.load(f)
            # the capture is only valid for the kernel sources it was taken with: kernels_sha16 maps each kernel
            # to the hash of its source file at capture time (tools/ncu_summary.py stamp)
            def fresh(kernel):
                rec = tr.get("kernels_sha16", {}).get(kernel)
                return rec is not None and rec[1] == _sha16(os.path.join(REPO, "lasercalib_b200", "csrc", rec[0]))
            if ws == 1 and tr.get("n_obs") == N:
                t = {k: v for k, v in tr["dram_bytes_per_launch"].items() if fresh(k)}
                if roof is not None and "i8_rowmax" in prof:
                    roof["traffic"] = t.get("k_i8_syrk")
                    roof["traffic_helpers"] = (t.get("k_i8_make", 0) + t.get("k_i8_rowmax", 0)) or None
                roof_m1["traffic"] = t.get("k_jacobian_blocks")
        except Exception:
            pass
        return roof, roof_m1, ms_jac, ms_res

    # ---- headline: device-resident run ----
    pb = make_rig(rig, points, seed=0, variant="volume", p_vis=pvis)
    C, P, N = pb["n_cams"], pb["n_points"], pb["n_obs"]
    run = device_run(pb, K, W, sample_clocks=True, keep_params=args.dump_outputs is not None)
    eng, sh = run["engine"], run["shard"]
    if args.dump_outputs is not None:
        cams_out, pts_out = run.pop("params")
        pts_out = D.allgather_rows(pts_out, sh["bounds"])         # collective: every rank takes part
        if rank == 0:
            dump_outputs(args.dump_outputs, cams_out, pts_out, run["final_cost"], run["optimality"])
        del cams_out, pts_out
    roof, roof_m1, ms_jac, ms_res = rooflines(pb, sh, run, eng)
    eng.close()
    n_loc = sh["point_ind"].size

    # ---- end to end through the public API with host buffers (e2e) ----
    cams_h, _k0 = pinned(pb["cams0"])
    pts_h, _k1 = pinned(pb["pts0"])
    p2_h, _k2 = pinned(pb["points_2d"])
    ci_h, _k3 = pinned(pb["camera_ind"])
    pi_h, _k4 = pinned(pb["point_ind"])
    sba = PySBA(cams_h.copy(), pts_h.copy(), p2_h, ci_h, pi_h)
    sba.bundleAdjust(1e-4, verbose=0, max_iterations=1, max_nfev=200)     # warm the path
    barrier()
    e2e_iters, e2e_calls = 0, 0
    split = dict(ingest_ms=0.0, solve_wall_ms=0.0, solve_device_ms=0.0, d2h_ms=0.0)
    t0 = time.perf_counter()
    while e2e_iters < K:
        sba = PySBA(cams_h, pts_h, p2_h, ci_h, pi_h)          # fresh object: full ingest per call
        r2 = sba.bundleAdjust(1e-4, verbose=0, max_iterations=K - e2e_iters, max_nfev=200)
        _ = float(r2.cost) + float(sba.cameraArray[0, 0])
        e2e_iters += int(r2["nit"])
        e2e_calls += 1
        for kk in split:
            split[kk] += sba.last_timing[kk]
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    h2d = (C * 11 + sh["pts"].size) * 8 + n_loc * (16 + 8 + 8)
    d2h = (C * 11 + sh["pts"].size) * 8
    e2e = {"value": e2e_iters / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": h2d * e2e_calls / max(1, e2e_iters),
           "d2h_bytes_per_step": d2h * e2e_calls / max(1, e2e_iters), "seconds_total": e2e_s,
           "steps": e2e_iters, "calls": e2e_calls,
           "ms_per_call": {kk: v / max(1, e2e_calls) for kk, v in split.items()},
           "note": "PySBA(...).bundleAdjust(1e-4) on pinned host numpy arrays, repeated from x0 until K "
                   "iterations: every call = ingest (H2D, validate, narrow, CSR/masks, plans) + its "
                   "iterations + parameters D2H; wall clock, max over ranks; ms_per_call splits rank 0's calls"}

    # ---- secondary workloads (N = 1, default config only): the other BASELINE configs ----
    secondary = []
    if ws == 1 and args.config == 3 and not args.no_secondary and args.rig is None and args.points is None:
        k2 = max(4, K // 2)
        extra = [(3, "ring24", 1_000_000, 0.5), (1, "ring4", 10_000, 1.0), (2, "example18", 200_000, 1.0),
                 (4, "wide8", 2_000_000, 1.0)]
        for cid, rg, npts, pv in extra:
            pb2 = make_rig(rg, npts, seed=0, variant="volume", p_vis=pv)
            r2 = device_run(pb2, k2, 2)
            rf2, rm2, _, _ = rooflines(pb2, r2["shard"], r2, r2["engine"])
            r2["engine"].close()
            entry = {"workload": workload_string(cid, rg, npts, pv), "n_cams": pb2["n_cams"], "n_points": pb2["n_points"],
                     "n_obs": pb2["n_obs"], "mean_views_per_point": pb2["n_obs"] / pb2["n_points"],
                     "value": 1e3 / r2["ms_per_step"], "unit": UNIT, "ms_per_step": r2["ms_per_step"],
                     "steps": r2["steps"], "nfev": r2["nfev"], "final_cost": r2["final_cost"],
                     "resjac_obs_per_s": rm2["obs_per_s"], "roofline": rf2, "roofline_m1": rm2,
                     "kernels_ms_per_step": {k: v["total_ms"] / max(1, r2["steps"]) for k, v in r2["prof"].items()}}
            if cid == 1 and not args.no_cpu_baseline:
                # config 1 is the case the reference runs directly: the CPU arm in full, side by side
                cb1 = cpu_reference_run(rg, npts, pv, pb2["n_obs"])
                sba1 = PySBA(pb2["cams0"].copy(), pb2["pts0"].copy(), pb2["points_2d"], pb2["camera_ind"], pb2["point_ind"])
                t1 = time.perf_counter()
                res1 = sba1.bundleAdjust(1e-4, verbose=0)
                entry["bundleAdjust_call_s"] = time.perf_counter() - t1
                entry["bundleAdjust_nfev"] = int(res1.nfev)
                entry["cpu_baseline"] = cb1
            secondary.append(entry)
            del pb2

    if rank != 0:
        return 0
    cpu_baseline = None
    if ws == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_reference_run(rig, args.cpu_points or min(points, 6000), pvis, N)
    steps_done, ms_per_step = run["steps"], run["ms_per_step"]
    line = {"metric": METRIC, "value": 1e3 / ms_per_step, "unit": UNIT, "n_gpus": ws, "steps": steps_done,
            "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "n_cams": C, "n_points": P, "n_obs": N,
                       "mean_views_per_point": N / P, "parallelism": "point-shard x%d" % ws,
                       "l2": "inputs (%.0f MB of observations) exceed the 126 MB L2; no explicit flush"
                             % (N * 28 / 1e6),
                       "solver": "scipy-TRF semantics, exact Schur/Cholesky Gauss-Newton direction"},
            "resjac_obs_per_s": N / ms_jac * 1e3, "residual_obs_per_s": N / ms_res * 1e3,
            "roofline": roof, "roofline_m1": roof_m1,
            "hbm_frac_iteration": None, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": run["launches"], "clocks": run["clocks"],
            "kernels_ms_per_step": {k: v["total_ms"] / max(1, steps_done) for k, v in run["prof"].items()},
            "final_cost": run["final_cost"], "nfev": run["nfev"], "secondary": secondary or None}
    # algorithmic HBM bytes of one iteration (SURVEY 8d B_M2, 4 streaming passes + Schur)
    b_m2 = 4 * 24.0 * N + (4 * 24 + 24) * P
    line["hbm_frac_iteration"] = b_m2 / (ms_per_step * 1e-3) / 1e9 / hbm_peak
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
