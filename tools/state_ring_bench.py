#!/usr/bin/env python
"""FrameRing vs StateRing in one process: device time per sample launch, device time per step(), bytes per game-tick of each ring
(from the allocated tensors) and DDQN.train's env_replay_ms per tick with replay="frames" / "states".  One JSON line per number,
each with the card's name, power limit and max SM clock read in the same run (default output: profiles/r4_state_ring.jsonl).

Device times per call are CUDA-graph replays of 50 calls (the device_us method of tools/latency_bench.py).  A captured step writes
full observation rows: BatchedTron.step does not pass obs_prev under capture, so the delta store that a reused `obs` buffer enables
shows only in the DDQN.train numbers."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tron_b200.batch_env import BatchedTron  # noqa: E402
from tron_b200.replay import FrameRing, StateRing  # noqa: E402

sys.path.insert(0, os.path.join(ROOT, "tools"))
from latency_bench import device_us  # noqa: E402

CASES = {  # name -> env dtype, encoding, sample out dtype
    "ddqn_bf16_popup3_to_f32": (torch.bfloat16, "popup3", torch.float32),
    "dqn_f32_lut1_to_f32": (torch.float32, "lut1", torch.float32),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def ring_bytes(ring):
    ts = [v for v in vars(ring).values() if torch.is_tensor(v)]
    return sum(t.numel() * t.element_size() for t in ts)


def rings(N, dt, enc, window):
    """a FrameRing and a StateRing with the same sample window, each on its own env, both played `window` ticks"""
    ea = BatchedTron(N, 10, 10, obs_dtype=dt, obs_enc=enc, seed=0, layout="bits10")
    eb = BatchedTron(N, 10, 10, obs_dtype=dt, obs_enc=enc, seed=0, layout="bits10")
    fr, sr = FrameRing(ea, window + 1, keep_terminal=True, seed=1), StateRing(eb, window, seed=1)
    fr.begin()
    sr.begin()
    for _ in range(window):
        a = ea.random_actions()
        fr.step(actions=a)
        sr.step(actions=a)
    torch.cuda.synchronize()
    return fr, sr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_state_ring.jsonl"))
    ap.add_argument("--sample-games", type=int, default=65536)
    ap.add_argument("--step-games", type=int, nargs="+", default=[131072, 4194304])
    ap.add_argument("--train-games", type=int, default=131072)
    ap.add_argument("--train-steps", type=int, default=40)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "state_ring_bench needs a GPU"
    info = card()
    lines = []

    def emit(**kw):
        o = dict(info, **kw)
        print(json.dumps(o), flush=True)
        lines.append(o)

    # ---- one sample launch, k = 64 / 1024 / 4096, 65,536 games, an 8-tick window
    for name, (dt, enc, odt) in CASES.items():
        fr, sr = rings(args.sample_games, dt, enc, 8)
        for k in (64, 1024, 4096):
            us = {}
            for label, ring in (("frames", fr), ("states", sr)):
                out = ring.sample(k, odt, counter=0)
                us[label] = device_us(lambda: ring.sample(k, odt, counter=7, out=out))
            emit(what="sample_device_us", case=name, games=args.sample_games, window_ticks=8, k=k, frames_us=round(us["frames"], 2),
                 states_us=round(us["states"], 2), states_over_frames=round(us["states"] / us["frames"], 3))
        del fr, sr
        torch.cuda.empty_cache()

    # ---- one step() of each ring and bytes per game-tick (DDQN configuration)
    dt, enc, _ = CASES["ddqn_bf16_popup3_to_f32"]
    for N in args.step_games:
        fr, sr = rings(N, dt, enc, 2)
        f_us = device_us(lambda: fr.step(), calls=10, replays=10)
        s_us = device_us(lambda: sr.step(), calls=10, replays=10)
        emit(what="step_device_us", case="ddqn_bf16_popup3", games=N, frames_us=round(f_us, 2), states_us=round(s_us, 2),
             frames_bytes_per_game_tick=round(ring_bytes(fr) / (fr.S * N), 2), states_bytes_per_game_tick=round(ring_bytes(sr) / (sr.S * N), 2))
        del fr, sr
        torch.cuda.empty_cache()
    for name, (dt, enc, _) in CASES.items():
        fr, sr = rings(4096, dt, enc, 2)
        emit(what="bytes_per_game_tick", case=name, frames=round(ring_bytes(fr) / (fr.S * 4096), 2), states=round(ring_bytes(sr) / (sr.S * 4096), 2))

    # ---- the DDQN loop: env_replay_ms per tick (select_actions + ring step), frames vs states
    from tron_b200 import dropin
    dropin.install()
    import DDQN
    for replay in ("frames", "states", "frames", "states"):
        tm = {}
        DDQN.train(n_envs=args.train_games, env_steps=args.train_steps, replay=replay, timings=tm, warmup_steps=8)
        emit(what="ddqn_env_replay_ms_per_tick", games=args.train_games, replay=replay, ticks=tm["ticks"],
             env_replay_ms_per_tick=round(tm["env_replay_ms"] / tm["ticks"], 4), q_forward_ms_per_tick=round(tm["q_forward_ms"] / tm["ticks"], 4),
             learn_ms_per_tick=round(tm["learn_ms"] / tm["ticks"], 4))
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        for o in lines:
            f.write(json.dumps(o) + "\n")


if __name__ == "__main__":
    main()
