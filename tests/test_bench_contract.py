"""bench.py host side (no GPU): the reference arm's JSON line carries the contract's keys, and the op / traffic
bookkeeping of the GPU arm is consistent with BASELINE.json and the committed profiles; --dump-outputs (writer on
the host, and once through the GPU arm)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(REPO, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_line_has_the_contract_keys():
    """`bench.py --impl reference` on a tiny bounded sample (400 points): ONE JSON line, the GPU arm's metric /
    unit / config keys, `impl`, a `cpu_baseline` describing this very run and an `e2e` object without copies."""
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-points", "400"], capture_output=True, text=True, timeout=600,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(REPO, "BASELINE.json")))
    # BASELINE.json's metric: "LM iters/sec & residual+Jacobian obs/sec, 24 cams x 1M pts, ..." -> the headline half
    assert "LM iters/sec" in base["metric"]
    assert d["impl"] == "reference" and d["metric"] == "LM_iters_per_sec" and d["unit"] == "iter/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f64" and d["n_gpus"] == 1
    for k in ("value", "steps", "warmup", "ms_per_step", "scaling", "data"):
        assert k in d
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["unit"] == d["unit"] and cb["value"] == d["value"]
    assert cb["cores"] > 0 and "bundleAdjust(1e-4)" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3


def test_configs_follow_baseline_json_and_traffic_stamps_are_wellformed():
    b = _bench()
    base = json.load(open(os.path.join(REPO, "BASELINE.json")))
    assert sorted(b.CONFIGS) == list(range(1, len(base["configs"]) + 1))
    # algorithmic <= executed int8 ops, both grow linearly in the points
    a1, e1 = b.i8_ops(24, 1_000_000)
    a2, e2 = b.i8_ops(24, 2_000_000)
    assert 0 < a1 <= e1 and abs(a2 / a1 - 2.0) < 1e-3 and abs(e2 / e1 - 2.0) < 1e-3
    tr = json.load(open(os.path.join(REPO, "profiles", "r02_traffic.json")))
    for kernel, (fn, sha) in tr["kernels_sha16"].items():
        assert kernel in tr["dram_bytes_per_launch"] and len(sha) == 16
        assert os.path.exists(os.path.join(REPO, "lasercalib_b200", "csrc", fn))
    assert b._sha16(os.path.join(REPO, "bench.py")) == b._sha16(os.path.join(REPO, "bench.py"))


def _load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f), allow_pickle=False) for f in os.listdir(d)}


def test_dump_outputs_writes_float64_under_the_size_limit(tmp_path, monkeypatch):
    """dump_outputs: every file float64; all of it when it fits, otherwise the same seeded sample of point rows
    on every call, with the row numbers beside it, and the files together within DUMP_MAX_BYTES."""
    b = _bench()
    rng = np.random.default_rng(1)
    cams, pts = rng.normal(size=(4, 11)), rng.normal(size=(5000, 3))
    b.dump_outputs(str(tmp_path / "all"), cams, pts, 1.5, 2.5)
    d = _load_dump(tmp_path / "all")
    assert sorted(d) == ["cameras", "cost", "optimality", "points3d"]
    assert all(a.dtype == np.float64 for a in d.values())
    assert np.array_equal(d["cameras"], cams) and np.array_equal(d["points3d"], pts)
    assert d["cost"].tolist() == [1.5] and d["optimality"].tolist() == [2.5]

    monkeypatch.setattr(b, "DUMP_MAX_BYTES", 40_000)
    for name in ("s1", "s2"):
        b.dump_outputs(str(tmp_path / name), cams, pts, 1.5, 2.5)
    s1, s2 = _load_dump(tmp_path / "s1"), _load_dump(tmp_path / "s2")
    assert sum(os.path.getsize(tmp_path / "s1" / (k + ".npy")) for k in s1) <= 40_000
    assert all(a.dtype == np.float64 for a in s1.values())
    rows = s1["points3d_rows"].astype(np.int64)
    assert 0 < rows.size < pts.shape[0] and np.all(np.diff(rows) > 0) and rows[-1] < pts.shape[0]
    assert np.array_equal(s1["points3d"], pts[rows])
    assert all(np.array_equal(s1[k], s2[k]) for k in s1)


@pytest.mark.gpu
def test_dump_outputs_of_the_gpu_arm(tmp_path):
    """`bench.py --dump-outputs DIR` on config 1: --steps timed steps, and the files hold the final state of the
    last one (its cost is the JSON line's final_cost, its cameras and points are finite and moved from x0)."""
    from lasercalib_b200.synth import make_rig
    out = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--config", "1", "--steps", "3",
                          "--warmup", "1", "--no-secondary", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3
    d = _load_dump(tmp_path)
    pb = make_rig("ring4", 10_000, seed=0, variant="volume", p_vis=1.0)
    assert d["cameras"].shape == pb["cams0"].shape and d["points3d"].shape == pb["pts0"].shape
    assert all(a.dtype == np.float64 and np.all(np.isfinite(a)) for a in d.values())
    assert d["cost"][0] == line["final_cost"]
    assert not np.array_equal(d["points3d"], pb["pts0"])
