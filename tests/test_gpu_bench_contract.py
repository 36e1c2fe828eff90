"""bench.py's JSON line against the measurement contract (run on the GPU box)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.helpers import ROOT

pytestmark = pytest.mark.gpu


def _run(*flags):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True,
                       cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_bench_line_has_every_contract_key():
    d = _run("--steps", "30", "--warmup", "3", "--cpu-seconds", "1.5")
    assert d["metric"] == "env-steps/sec" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 30 and d["warmup"] >= 3 and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"
    assert "workload" in d["config"] and d["config"]["envs_per_gpu"] == 4096 and "model" not in d["config"]
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == json.loads(json.dumps(bench.workload_config(4096, 1)))    # the same dict in both arms
    assert d["run"]["reset_mode"] == "cached" and d["run"]["step_kernel_build"] == "latency"
    assert abs(d["value"] - 4096 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["gpu_launches"] == 30                                   # one launch of step_kernel per step
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    e = d["e2e"]
    assert e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 4096 * 12 * 4 and e["d2h_bytes_per_step"] == 4096 * 78 * 4
    assert 0 < e["value"] < d["value"] * 1.05                        # host round trip cannot beat the resident step
    r = d["roofline"]
    assert r["bound"] in ("fp32", "hbm", "tensor") and r["unit"] == "TFLOP/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
    assert r["traffic"] is None or (r["traffic"] > 0 and r["traffic_source"])   # ncu record for this batch/build, or none
    assert r["hbm"]["peak"] > 1000 and 0 < r["hbm"]["frac"] < 1
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["unit"] == d["unit"] and c["sample"]
    assert d["value"] > 20 * c["value"]
    assert d["policy_rollout"]["value"] > 0 and d["saturated"]["value"] > d["value"]
    # the legs that put the rest of north_star under the driver's clock
    assert d["ppo_train"]["value"] > 0 and d["ppo_train"]["grad_allreduce"]["pack_unpack_kernels"] == 0
    ps = d["ppo_stand"]
    assert ps["seconds_to_target"] is not None and ps["seconds_to_target"] < 300 and ps["final_return"] >= ps["target_return"]
    assert d["body_contacts"]["value"] > 0 and d["gae"]["frac"] > 0.1 and d["reset_mode_simulate"]["value"] > 0


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs writes obs / reward / done of the last of exactly --steps timed steps; the same arguments give
    the same inputs, hence the same outputs, run after run."""
    quick = ("--warmup", "3", "--no-cpu-baseline", "--no-policy-rollout", "--no-ppo-train", "--no-saturated")
    dumps = {}
    for tag, steps in (("a", 7), ("b", 7), ("c", 8)):
        d = _run("--steps", str(steps), *quick, "--dump-outputs", str(tmp_path / tag))
        assert d["steps"] == steps and d["gpu_launches"] == steps
        dumps[tag] = {k: np.load(tmp_path / tag / (k + ".npy")) for k in ("obs", "reward", "done")}
    a = dumps["a"]
    assert a["obs"].shape == (4096, 76) and a["reward"].shape == (4096,) and a["done"].shape == (4096,)
    assert all(x.dtype == np.float32 for x in a.values()) and np.isfinite(a["obs"]).all()
    for k in a:
        assert np.array_equal(a[k], dumps["b"][k]), k
    assert not np.array_equal(a["obs"], dumps["c"]["obs"])


def test_reference_arm_line():
    d = _run("--impl", "reference", "--steps", "5", "--warmup", "1")
    assert d["impl"] == "reference" and d["metric"] == "env-steps/sec" and d["unit"] == "env-steps/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == json.loads(json.dumps(bench.workload_config(4096, 1)))
    assert d["run"]["reset_mode"] == "simulate"
