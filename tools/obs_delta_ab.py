#!/usr/bin/env python
"""A/B of the observation delta store (tron_step_args.obs_prev) in one process: the same env and reused obs buffer, timed in
alternating blocks of 128 ticks with TRON_OPT_ENCODE_VARIANT 64 (full rows) and 0 (changed 32-byte units only), plus an untimed
pass that counts on the device which fraction of the buffer's 32-byte units really changes from one tick to the next.
usage: obs_delta_ab.py [--reps 6] [--caps 4,5,6,8] [--out FILE.jsonl]
  --caps   also time every config under these TRON_OPT_BITS_CTAS_PER_SM values (delta path)"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tron_b200  # noqa: E402
from tron_b200 import abi  # noqa: E402
from tron_b200.batch_env import BatchedTron  # noqa: E402

M = 1 << 20
BLOCK = 128
CONFIGS = [  # name, N, dtype, enc, layout, slide_mode, policy epsilon (None: random-action tape as in bench.py)
    ("headline bf16 lut1", 4 * M, "bf16", "lut1", "bits10", None, None),
    ("bf16 pop_up3", 2 * M, "bf16", "popup3", "bits10", None, None),
    ("f32 lut1", 2 * M, "f32", "lut1", "bits10", None, None),
    ("i8 lut1", 4 * M, "i8", "lut1", "bits10", None, None),
    ("temper bf16 lut1", 4 * M, "bf16", "lut1", "bits", "temper", None),
    ("eps 0.1 bf16 lut1", 4 * M, "bf16", "lut1", "bits10", None, 0.1),
]
TDT = {"bf16": torch.bfloat16, "f32": torch.float32, "i8": torch.int8}


def set_opt(opt, v):
    tron_b200.lib.check(tron_b200.lib.load().tron_set_option(opt, v), "tron_set_option")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def sm_clock():
    return subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                          capture_output=True, text=True).stdout.strip()


def make(N, dt, enc, layout, slide, eps):
    env = BatchedTron(N, 10, 10, obs_dtype=TDT[dt], obs_enc=enc, reward="ddqn", seed=0, layout=layout, slide_mode=slide,
                      policy="uniform" if eps is None else "free_eps", policy_epsilon=eps or 0.0)
    obs = env.reset()
    tape = [env.random_actions(1000 + i) for i in range(4)] if eps is None else [None] * 4
    out = dict(reward=torch.empty((N, 2), dtype=torch.float32, device="cuda"), done=torch.empty(N, dtype=torch.uint8, device="cuda"),
               winner=torch.empty(N, dtype=torch.uint8, device="cuda"), want_ep_len=False)
    tick = [0]

    def step(n):
        for _ in range(n):
            env.step(tape[tick[0] & 3], obs=obs, **out)
            tick[0] += 1
    return env, obs, step


def timed(step):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    step(BLOCK)
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / BLOCK


def dirty_fraction(obs, step, ticks=8):
    """fraction of the buffer's 32-byte units that differ between consecutive ticks (device-side compare)"""
    set_opt(abi.OPT_ENCODE_VARIANT, 64)
    u = obs.view(torch.uint8).view(-1, 32)
    changed = total = 0
    for _ in range(ticks):
        prev = u.clone()
        step(1)
        changed += int((prev != u).any(1).sum())
        total += u.shape[0]
        del prev
    return changed / total


def summary(xs):
    return {"median_ms": statistics.median(xs), "min_ms": min(xs), "max_ms": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--caps", default="")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n"); out.flush()
    emit(dict(card(), kind="card"))
    for name, N, dt, enc, layout, slide, eps in CONFIGS:
        env, obs, step = make(N, dt, enc, layout, slide, eps)
        step(64)
        torch.cuda.synchronize()
        t = {64: [], 0: []}
        clocks = []
        for _ in range(a.reps):
            for v in (64, 0):
                set_opt(abi.OPT_ENCODE_VARIANT, v)
                t[v].append(timed(step))
            clocks.append(sm_clock())
        set_opt(abi.OPT_ENCODE_VARIANT, 0)
        full, delta = summary(t[64]), summary(t[0])
        emit({"kind": "ab", "config": name, "envs": N, "block_ticks": BLOCK, "full_rows": full, "delta": delta,
              "speedup_median": full["median_ms"] / delta["median_ms"], "ranges_overlap": delta["max_ms"] >= full["min_ms"],
              "env_steps_per_s_delta": N / (delta["median_ms"] * 1e-3), "env_steps_per_s_full": N / (full["median_ms"] * 1e-3),
              "dirty_unit_fraction_32B": dirty_fraction(obs, step), "sm_clock_samples": clocks})
        set_opt(abi.OPT_ENCODE_VARIANT, 0)
        if a.caps:
            for cap in [int(c) for c in a.caps.split(",")]:
                set_opt(abi.OPT_BITS_CTAS_PER_SM, cap)
                step(8)
                xs = [timed(step) for _ in range(a.reps)]
                emit({"kind": "cta_cap", "config": name, "cap": cap, "delta": summary(xs)})
            set_opt(abi.OPT_BITS_CTAS_PER_SM, 0)
        del env, obs, step
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
