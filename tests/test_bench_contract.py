"""bench.py prints one JSON line with the contract's keys (reference arm on CPU here; our arm on the GPU box)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
             "config", "cpu_baseline", "e2e"}


def _run(args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-seconds", "1"])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    have_live = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "Deep-Q-learning_TRON", "tron"))
    assert d["value"] > 100 and d["cpu_baseline"]["kind"] == ("reference" if have_live else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["cpu_c_port"]["value"] > d["value"]  # the C port is reported next to the Python loop
    r = d["port_over_reference_cost"]
    assert r["port_steps_per_s_per_core"] > 100 and (not have_live or 0.3 < r["port_over_reference"] < 3.0)


@pytest.mark.gpu
def test_our_arm_line():
    d = _run(["--steps", "3", "--warmup", "3", "--envs-per-gpu", "262144", "--ticks-per-step", "8", "--e2e-steps", "3", "--cpu-seconds", "1", "--no-configs"])
    assert BASE_KEYS | {"roofline", "clocks", "gpu_launches", "parity_in_run", "eps_greedy_streams"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["gpu_launches"] == 24 and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["parity_in_run"] is True
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.05 < r["frac"] < 1.2
    assert abs(d["value"] - 262144 * 8 * 3 / (d["ms_per_step"] * 3e-3)) / d["value"] < 1e-6
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 2 * 262144 and e["d2h_bytes_per_step"] == 262144 * (288 + 10) and 0 < e["value"] < d["value"]
    assert e["roofline"]["bound"] == "pcie" and 0 < e["roofline"]["frac"] < 1.3 and e["blocking_api"]["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert len(d["eps_greedy_streams"]) == 4 and all(x["value"] > 0 for x in d["eps_greedy_streams"])


@pytest.mark.gpu
def test_dump_outputs_follow_the_ticks_played(tmp_path):
    """--dump-outputs writes the last timed step's outputs; warmup 2 + steps 2 and warmup 1 + steps 3 play the same ticks from the
    same inputs, so two processes must dump identical arrays while reporting the steps they timed."""
    import numpy as np
    small = ["--envs-per-gpu", "65536", "--ticks-per-step", "4", "--no-e2e", "--no-cpu-baseline", "--no-configs", "--no-streams"]
    runs = {}
    for steps, warmup in ((2, 2), (3, 1)):
        out = tmp_path / ("s%d" % steps)
        d = _run(small + ["--steps", str(steps), "--warmup", str(warmup), "--dump-outputs", str(out)])
        assert d["steps"] == steps and d["gpu_launches"] == 4 * steps and d["parity_in_run"] is True
        runs[steps] = {f.stem: np.load(f) for f in sorted(out.glob("*.npy"))}
        assert sum(f.stat().st_size for f in out.glob("*.npy")) <= 64 << 20
    a, b = runs[2], runs[3]
    assert set(a) == {"obs", "reward", "done", "winner"} and a["obs"].shape[1:] == (2, 1, 12, 12) and a["obs"].shape[0] == a["done"].shape[0]
    for k in a:
        assert a[k].dtype == np.float32 and np.array_equal(a[k], b[k]), k
    assert 0 < a["done"].sum() < a["done"].size and set(np.unique(a["winner"])) <= {0.0, 1.0, 2.0}


@pytest.mark.gpu
def test_our_arm_config_legs():
    """the BASELINE config #3 / #4 / #5 legs of the default invocation (small headline so the test stays short)"""
    d = _run(["--steps", "2", "--warmup", "3", "--envs-per-gpu", "65536", "--ticks-per-step", "4", "--no-e2e", "--no-cpu-baseline", "--no-streams"], timeout=900)
    c = d["configs"]
    assert set(c) == {"cfg3", "cfg4", "cfg5", "large_grid_fused_obs"}
    assert c["cfg5"]["value"] > 1e9 and c["cfg5"]["roofline"]["bound"] == "hbm" and 0 < c["cfg5"]["reset_fraction"] < 1
    assert c["cfg5"]["step_many_16_ticks_per_launch"]["value"] > c["cfg5"]["value"]
    assert [s["epsilon"] for s in c["cfg5"]["eps_greedy_streams"]] == [0.5, 0.1, 0.003]
    assert all(s["value"] > 1e9 and s["mean_episode_ticks"] > 3 for s in c["cfg5"]["eps_greedy_streams"])
    assert c["large_grid_fused_obs"]["value"] > 1e8 and 0.5 < c["large_grid_fused_obs"]["roofline"]["frac"] < 1.2
    for k in ("cfg3", "cfg4"):
        assert c[k]["value"] > 1e5 and set(c[k]["ms"]) >= {"q_forward", "env_replay", "learn"} and 0 < c[k]["env_replay_fraction_of_loop"] < 1
    assert "allreduce" in c["cfg4"]["ms"] and c["cfg4"]["learn_steps"] == 12
