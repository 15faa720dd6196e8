"""bench.py contract: one JSON line with the keys the driver reads.  The reference arm (CPU, oracle port) runs anywhere; the
GPU arm is checked on the GPU box with a handful of steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "cpu_baseline"}


def _run(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                       timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_split_blocks_covers_exactly_the_requested_steps():
    import bench
    for K in (1, 6, 49, 50, 51, 200, 1001):
        b = bench.split_blocks(K)
        assert sum(b) == K and max(b) <= bench.BLOCK_STEPS and max(b) - min(b) <= 1, (K, b)


def _dumped(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_reference_arm_prints_the_contract_line(tmp_path):
    j = _run("--impl", "reference", "--steps", "4", "--warmup", "1", "--dump-outputs", str(tmp_path / "a"))
    assert BASE_KEYS <= set(j) and j["impl"] == "reference" and j["metric"] == "env-steps/sec" and j["unit"] == "env-steps/s"
    assert j["value"] > 0 and j["higher_is_better"] is True and j["vs_baseline"] is None and j["dtype"] == "f64"
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1 and j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in j["config"]
    _run("--impl", "reference", "--steps", "4", "--warmup", "1", "--dump-outputs", str(tmp_path / "b"))
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    assert sorted(a) == ["done", "observ", "reward"] and all(x.dtype.name == "float32" for x in a.values())
    n = a["reward"].shape[0]
    assert a["observ"].shape == (n, 4) and a["done"].shape == (n,)
    for k in a:                                 # same arguments, same inputs: the same outputs
        assert (a[k] == b[k]).all(), k


@pytest.mark.gpu
def test_gpu_arm_prints_the_contract_line(tmp_path):
    j = _run("--steps", "6", "--warmup", "3", "--dump-outputs", str(tmp_path))
    assert BASE_KEYS | {"clocks", "gpu_launches", "roofline", "timing"} <= set(j)
    assert j["n_gpus"] == 1 and j["steps"] == 6 and j["warmup"] == 3 and j["dtype"] == "f32" and j["scaling"] == "weak"
    assert j["gpu_launches"] == 6               # one step kernel per step (4096 envs fit one wave: no warp re-grouping launches)
    assert j["value"] > 1e6 and abs(j["ms_per_step"] * 1e-3 * j["value"] - j["config"]["envs_per_gpu"]) < 1e-3 * j["config"]["envs_per_gpu"]
    t = j["timing"]                             # exactly --steps timed steps: ms_per_step = their total time / --steps
    assert t["steps_timed"] == 6 and sum(t["block_steps"]) == 6 and len(t["block_ms"]) == len(t["block_steps"]) == t["blocks"]
    assert len(t["per_rank_ms_per_step"]) == 1 and abs(sum(t["block_ms"]) / 6 - j["ms_per_step"]) < 1e-3 * j["ms_per_step"]
    rf = j["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert j["e2e"]["value"] > 1e6 and j["e2e"]["h2d_bytes_per_step"] == 4096 * 2 * 4 and j["e2e"]["d2h_bytes_per_step"] > 0
    assert j["e2e"]["value"] < j["value"]
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["value"] > 1e3
    c = j["config"]
    assert c["error_flags_or"] == 0 and 0.0 <= c["resets_per_step"] < 0.02
    x = c["extras"]
    for name in ("walk_ik_demo_clock_x4", "north_star_size", "north_star_size_demo_clock_x4", "C3_gallop_ol_rand_gains",
                 "C4_turn_ik_heightfield", "C5_standup_arm_18dof"):
        assert "error" not in x[name], (name, x[name])
        assert x[name]["value"] > 1e6 and (x[name]["error_flags_or"] & 1) == 0, (name, x[name])
    assert x["north_star_size"]["envs_per_gpu"] == 65536 and x["north_star_size"]["value"] > 1e7
    assert x["walk_ik_demo_clock_x4"]["resets_per_step"] < c["resets_per_step"] + 1e-9      # walking robots do not fall
    assert "error" not in x["rollout_with_policy"]
    d = _dumped(tmp_path)                       # the last timed step's outputs: what BatchedRexEnv.step returned
    assert sorted(d) == ["done", "motor_command", "observ", "reward"] and all(a.dtype.name == "float32" for a in d.values())
    assert d["observ"].shape == (4096, 4) and d["reward"].shape == d["done"].shape == (4096,) and d["motor_command"].shape == (4096, 12)
    assert np.isfinite(d["observ"]).all() and set(np.unique(d["done"])) <= {0.0, 1.0} and np.abs(d["observ"]).max() > 0
