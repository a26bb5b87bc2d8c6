"""Per-CTA cycle counters of k_i8_syrk (LCBA_SCHUR_STATS=1): which tile kinds set the kernel's time.
Usage: [LCBA_I8_PLAN=strip|cover] [LCBA_I8_SCHED=range] python tools/i8_stats.py [rig] [points]"""
import ctypes as C, os, sys
os.environ["LCBA_SCHUR_STATS"] = "1"
os.environ.setdefault("LCBA_SCHUR_I8", "1")
sys.path.insert(0, ".")
import numpy as np
from lasercalib_b200._cabi import Engine
from lasercalib_b200.synth import make_rig
rig = sys.argv[1] if len(sys.argv) > 1 else "ring24"
pb = make_rig(rig, int(sys.argv[2]) if len(sys.argv) > 2 else 1000000, seed=0, variant="volume", p_vis=1.0)
eng = Engine()
eng.set_problem(pb["cams0"], pb["pts0"], pb["points_2d"], pb["camera_ind"], pb["point_ind"])
eng.linearize(1e-6); eng.linearize(1e-6)
buf = np.zeros((1024, 4), dtype=np.int64)
nk, ns = C.c_int(), C.c_int()
eng.lib.lcba_debug_schur_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
rc = eng.lib.lcba_debug_schur_stats(eng.h, buf.ctypes.data_as(C.c_void_p), 1024, C.byref(nk), C.byref(ns))
assert rc == 0, rc
import torch
sms = torch.cuda.get_device_properties(0).multi_processor_count
plan = os.environ.get("LCBA_I8_PLAN")
pl = Engine.i8_plan(pb["n_cams"], pb["n_points"], sms, {"strip": 1, "cover": 2}.get(plan, 0))
sched = "range" if os.environ.get("LCBA_I8_SCHED") == "range" else "K-major"
print("%s plan, %s schedule: tiles %d, CTAs %d, K blocks %d" % ("cover" if pl["cover"] else "strip", sched, len(pl["tiles"]),
                                                                len(pl["work"]), pl["nkb"]))
for m0, mn, m20, m2n, n0, nn, n20, n2n, w0, nw in pl["tiles"]:
    st = buf[w0:w0 + nw].astype(float)
    kb = (pl["work"][w0:w0 + nw, 2] - pl["work"][w0:w0 + nw, 1]).astype(float)
    print("tile rows rg %2d+%2d (+%2d+%d) cols %2d+%d (+%d): %2d CTAs x %5.0f K blocks: MMA warp %.2f Mcyc (max %.2f) = %4.0f cyc / K block, waiting at FULL %4.1f %%, producer in the window %4.1f %%"
          % (m0, mn, m20, m2n, n0, nn, n2n, nw, kb.mean(), st[:, 1].mean() / 1e6, st[:, 1].max() / 1e6, (st[:, 1] / kb).mean(),
             100 * st[:, 0].sum() / st[:, 1].sum(), 100 * st[:, 2].sum() / max(st[:, 3].sum(), 1.0)))
