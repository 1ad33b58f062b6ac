#!/usr/bin/env python
"""bench.py -- env-steps/s of the batched 2-player TRON tick (BASELINE.json metric) on N B200s of one node.

  python bench.py --gpus 1 --steps 20 --warmup 5                      # our arm (CUDA kernels through the C ABI)
  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference --gpus 1 --steps 3 --warmup 1      # reference arm: the reference's own Python loop on the host cores

A "step" is one pass of the hot path over one batch of synthetic input: --ticks-per-step (default 128) consecutive fused ticks (move,
collision, winner, trail write, auto-reset, reward, both players' observation planes; one tron_step launch per tick) of every env
on the GPU, driven by a pre-generated action tape resident in HBM.  With the driver's K = 20 steps the timed region is > 1 s.
Headline workload: BASELINE config #2 (10x10 grid, uniform random actions, 1-plane bf16 observations, auto-reset) scaled from 4096 to
--envs-per-gpu games so that state + observations are far larger than L2; envs shard across ranks with no collective (weak
scaling).  The same run also measures the other BASELINE configs (`configs`: #5 64x64 pure tick, #3 DQN loop, #4 DDQN loop with
the gradient all-reduce timed separately), epsilon-greedy action streams on every rank, the end-to-end host-buffer path against
the measured PCIe ceiling, and checks a slice of the timed state against the CPU oracle.  One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "env-steps/s (batched 2-player TRON)"
UNIT = "env-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=1 << 22)
    ap.add_argument("--ticks-per-step", type=int, default=128, help="consecutive ticks (one tron_step launch each) that make up one bench step")
    ap.add_argument("--width", type=int, default=10)
    ap.add_argument("--obs-dtype", default="bf16", choices=["bf16", "f32", "i8"])
    ap.add_argument("--enc", default="lut1", choices=["lut1", "popup3", "popup3_const", "none"])
    ap.add_argument("--layout", default="bits10", choices=["bits10", "bits", "tile8", "trail"],
                    help="state layout: 32-byte bit planes (10x10 only), 48-byte bit planes, int8 Tile.value grid, or trail lists (pure ticks)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU work budget for the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the BASELINE config #3/#4/#5 legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle check of the timed state")
    ap.add_argument("--no-streams", dest="streams", action="store_false", help="skip the epsilon-greedy action-stream lines")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (obs, reward, done, winner of a fixed seeded sample of rank 0's envs) "
                         "as DIR/<name>.npy in float32, about 32 MiB in all, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons, power = [], None, set(), []
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2]); power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power) if power else None}


# ----------------------------------------------------------------------------------------------- CPU legs
def _c_oracle_worker(args):
    from oracle import c_oracle as oc
    n_envs, W, ticks, dt, enc, seed = args
    steps, sec = oc.bench_random(n_envs, W, W, ticks, dt, enc, seed)
    return steps, sec


def _py_port_worker(args):
    from oracle import py_port
    seed, env_steps, W = args[:3]
    t0 = time.perf_counter()
    steps, _ = py_port.play_random(seed, env_steps, W, W, with_pop_up=len(args) > 3 and args[3])
    return steps, time.perf_counter() - t0


_LIVE = {}  # the live reference's modules (imported once in the parent, inherited by forked workers)


def live_reference():
    """Import the unmodified reference from baseline/_ref (a copy made by __graft_entry__.build() in the authoring container; it is
    git-ignored but travels to the GPU box).  -> (game module, util module, player module) or None when it is not there / not importable."""
    if "mods" in _LIVE:
        return _LIVE["mods"]
    mods = None
    ref = os.path.join(ROOT, "baseline", "_ref", "Deep-Q-learning_TRON")
    if os.path.isdir(os.path.join(ref, "tron")):
        saved_path, saved_mods = list(sys.path), {k: v for k, v in sys.modules.items() if k.split(".")[0] in ("tron", "config", "Net", "orderedset")}
        try:
            for k in saved_mods:
                del sys.modules[k]
            sys.path[:] = [p for p in sys.path if os.path.basename(os.path.normpath(p or ".")) != "deep-q-learning_tron_b200"]
            sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref", "shim"))  # `orderedset`: the one missing third-party import (dead code on this path)
            sys.path.insert(0, ref)
            try:
                import torchvision  # noqa: F401  (before the file-less namespace package `tron` exists, see tests/golden/make_golden.py)
            except Exception:
                pass
            import tron.game as game
            import tron.util as util
            import tron.player as player
            mods = (game, util, player)
        except Exception as e:  # missing dependency on this box -> the port stands in
            _LIVE["error"] = "%s: %s" % (type(e).__name__, e)
            mods = None
        finally:
            sys.path[:] = saved_path
    _LIVE["mods"] = mods
    return mods


def _live_ref_worker(args):
    """the reference's own loop: make_game(True, True) + Game.step(randrange(4), randrange(4)) (BASELINE.md section 4), optionally + pop_up"""
    import random
    seed, env_steps, with_pop_up = args
    game, util, player = _LIVE["mods"]
    random.seed(seed)
    steps = 0
    t0 = time.perf_counter()
    while steps < env_steps:
        g = util.make_game(True, True)
        done = False
        while not done:
            s1, s2, done = g.step(random.randrange(4), random.randrange(4))
            if with_pop_up:
                util.pop_up(s1); util.pop_up(s2)
            steps += 1
    return steps, time.perf_counter() - t0


def cpu_c_port(W, dt, enc, budget_s, cores):
    """The plain-C oracle (scalar port), one process per host core, same random-policy auto-reset workload."""
    import multiprocessing as mp
    from oracle import c_oracle as oc
    oc.build()
    n_envs = 4096
    _, sec = oc.bench_random(n_envs, W, W, 8, dt, enc, 1)  # calibrate
    ticks = max(8, int(budget_s / max(sec / 8, 1e-6)))
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        res = pool.map(_c_oracle_worker, [(n_envs, W, ticks, dt, enc, 100 + i) for i in range(cores)])
    wall = time.perf_counter() - t0
    steps = sum(r[0] for r in res)
    return steps / max(r[1] for r in res), "%d procs x %d envs x %d ticks, C oracle, wall %.1fs" % (cores, n_envs, ticks, wall)


def cpu_python_loop(W, env_steps_per_core, cores, with_pop_up=False, live=False):
    """-> (env-steps/s over all cores, env-steps played); time = the slowest worker's own loop time (pool start-up excluded)"""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        if live:
            res = pool.map(_live_ref_worker, [(i, env_steps_per_core, with_pop_up) for i in range(cores)])
        else:
            res = pool.map(_py_port_worker, [(i, env_steps_per_core, W, with_pop_up) for i in range(cores)])
    steps = sum(r[0] for r in res)
    return steps / max(r[1] for r in res), steps


def port_over_reference_cost():
    """single-core env-steps/s of the port and of the live reference on the same box (None when the reference is not importable here)"""
    from oracle import py_port
    t0 = time.perf_counter()
    s, _ = py_port.play_random(0, 1500, 10, 10)
    port = s / (time.perf_counter() - t0)
    if live_reference() is None:
        return {"port_steps_per_s_per_core": port, "reference_steps_per_s_per_core": None, "port_over_reference": None,
                "note": "live reference not importable on this box (%s); measured in the authoring container: see tests/golden/misc.json" % _LIVE.get("error", "baseline/_ref absent")}
    s, dt = _live_ref_worker((0, 1500, False))
    ref = s / dt
    return {"port_steps_per_s_per_core": port, "reference_steps_per_s_per_core": ref, "port_over_reference": port / ref}


def run_reference(a):
    """Reference arm: the reference's own Python Game.step loop -- the UNMODIFIED reference from baseline/_ref when it imports on this
    box (kind "reference"), else the pure-Python port oracle/py_port.py (kind "port", validated against the live reference for results
    and cost) -- multiprocess over all host cores, same workload, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    W = a.width
    live = live_reference() is not None and W == 10  # make_game reads the grid size from the reference's config.py (10x10)
    ratio = port_over_reference_cost()
    rate1 = ratio["reference_steps_per_s_per_core"] if live else ratio["port_steps_per_s_per_core"]
    per = max(200, int(min(2.5, 120.0 / max(a.steps, 1)) * rate1))  # ~2.5 s of work per core per step, whole run bounded to ~2 min
    for _ in range(a.warmup):
        cpu_python_loop(W, max(50, per // 8), cores, live=live)
    total, dt = 0, 0.0
    for _ in range(a.steps):
        rate, st = cpu_python_loop(W, per, cores, live=live)
        total += st
        dt += st / rate
    v = total / dt
    popup_rate, _ = cpu_python_loop(W, max(100, per // 4), cores, with_pop_up=True, live=live)  # BASELINE.md section 4 "variant B"
    other_rate, _ = cpu_python_loop(W, max(100, per // 2), cores, live=not live) if live_reference() is not None and W == 10 else (None, 0)
    c_v, c_sample = cpu_c_port(W, 3, 1, min(a.cpu_seconds, 6.0), cores)
    kind = "reference" if live else "port"
    what = ("the UNMODIFIED reference (baseline/_ref): make_game(True,True) + Game.step(randrange(4), randrange(4))" if live else
            "pure-Python port of Game.step (results and cost validated vs the live reference)")
    sample = "%d host procs x %d env-steps per bench step, %s" % (cores, per, what)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * dt / max(a.steps, 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i8",
        "data": "synthetic", "config": workload_config(a, None),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "other_python_arm": {"value": other_rate, "unit": UNIT, "cores": cores, "kind": "port" if live else "reference"},
        "port_over_reference_cost": ratio,
        "cpu_c_port": {"value": c_v, "unit": UNIT, "cores": cores, "kind": "port", "sample": c_sample},
        "python_loop_with_pop_up": {"value": popup_rate, "unit": UNIT, "cores": cores, "note": "same loop + pop_up on both observations (DDQN data path)"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ----------------------------------------------------------------------------------------------- ours
def workload_config(a, n_envs):
    return {"workload": "BASELINE config #2 scaled: %dx%d grid, uniform random actions (pre-generated u8 tape in HBM), auto-reset, "
                        "%s observations (%s), fused step+obs, state layout %s" % (a.width, a.width, a.obs_dtype, a.enc, a.layout),
            "envs_per_gpu": n_envs, "grid": [a.width, a.width], "obs_dtype": a.obs_dtype, "obs_enc": a.enc, "state_layout": a.layout,
            "ticks_per_step": a.ticks_per_step,
            "l2_policy": "inputs larger than L2 (state+obs per GPU >> 126 MB), no flush", "parallelism": "env-sharded, no collective"}


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_of(key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture of the same configuration
    (profiles/traffic.json: {key: {"bytes": dram__bytes_read.sum + dram__bytes_write.sum, "source": profile file}})"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(key)
        return (t["bytes"], t.get("source")) if isinstance(t, dict) else (t, None)
    except Exception:
        return None, None


DUMP_BYTES = 32 << 20


def dump_outputs(dirname, obs, reward, done, winner):
    """The tick's outputs for a fixed seeded sample of envs (the same ids for the same --envs-per-gpu), as float32 .npy files.
    All values are small integers or bf16 / f32 numbers, so float32 holds them exactly."""
    import numpy as np
    import torch
    n = reward.shape[0]
    per_env = 4 * (reward[0].numel() + 2 + (obs[0].numel() if obs is not None else 0))
    k = min(n, DUMP_BYTES // per_env)
    idx = torch.as_tensor(np.sort(np.random.default_rng(0).choice(n, size=k, replace=False)), device=reward.device)
    os.makedirs(dirname, exist_ok=True)
    for name, t in (("obs", obs), ("reward", reward), ("done", done), ("winner", winner)):
        if t is not None:
            np.save(os.path.join(dirname, name + ".npy"), t.index_select(0, idx).float().cpu().numpy())


def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    import tron_b200
    from tron_b200 import abi
    from tron_b200.batch_env import BatchedTron, HostTron, host_copy_bandwidth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()

    def reduce_(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return reduce_(x, dist.ReduceOp.MAX)

    def sum_over_ranks(x):
        return reduce_(x, dist.ReduceOp.SUM)

    peak, peak_src = hbm_peak()
    N, W, TPS = a.envs_per_gpu, a.width, max(1, a.ticks_per_step)
    tdt = {"bf16": torch.bfloat16, "f32": torch.float32, "i8": torch.int8}[a.obs_dtype]
    dt_code = {"bf16": abi.BF16, "f32": abi.F32, "i8": abi.I8}[a.obs_dtype]
    enc_code = {"lut1": abi.ENC_LUT1, "popup3": abi.ENC_POPUP3, "popup3_const": abi.ENC_POPUP3_CONST, "none": abi.ENC_NONE}[a.enc]
    if a.layout == "bits10" and W != 10:
        a.layout = "tile8"
    env = BatchedTron(N, W, W, device=dev, obs_dtype=tdt, obs_enc=a.enc, reward="ddqn", auto_reset=True, seed=0, env_id_base=rank * N, layout=a.layout)
    obs = env.reset()
    # synthetic random-policy action stream, resident in HBM before the timed region
    tape = [env.random_actions(1000 + i) for i in range(4)]
    reward = torch.empty((N, 2), dtype=torch.float32, device=dev)
    done = torch.empty(N, dtype=torch.uint8, device=dev)
    winner = torch.empty(N, dtype=torch.uint8, device=dev)
    ticks_played = 0

    def one_step():
        nonlocal ticks_played
        for _ in range(TPS):
            env.step(tape[ticks_played & 3], obs=obs, reward=reward, done=done, winner=winner, want_ep_len=False)
            ticks_played += 1

    for _ in range(a.warmup):
        one_step()
    torch.cuda.synchronize()
    st0 = env.stats_dict()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier(); torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    ev0.record()
    for _ in range(a.steps):
        one_step()
    ev1.record()
    torch.cuda.synchronize(); barrier()
    t_wall1 = time.perf_counter()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    st1 = env.stats_dict()
    env_steps = st1["env_steps"] - st0["env_steps"]
    assert env_steps == N * a.steps * TPS, (env_steps, N * a.steps * TPS)
    f_reset = (st1["episodes"] - st0["episodes"]) / env_steps
    value = sum_over_ranks(float(env_steps)) / (ms * 1e-3)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, obs, reward, done, winner)

    # ---- in-run parity: the timed state itself, on the first and last 2048 env ids of this rank, against the CPU oracle
    parity = None
    if not a.no_parity and a.layout != "trail":
        from oracle import c_oracle as oc
        K = min(2048, N)
        host_tape = [t.cpu().numpy() for t in tape]
        ex = env.export()
        ok = True
        for lo in sorted({0, N - K}):
            o = oc.OracleEnv(K, W, W, obs_dtype=dt_code, obs_enc=enc_code, reward="ddqn", seed=0, env_id_base=rank * N + lo)
            o.reset()
            planes, full_enc = o.P, o.obs_enc
            o.P, o.obs_enc = 0, abi.ENC_NONE  # intermediate ticks: state only
            last = None
            for t in range(ticks_played):
                if t == ticks_played - 1:
                    o.P, o.obs_enc = planes, full_enc
                last = o.step(host_tape[t & 3][lo:lo + K])
            oex = o.export()
            ok = ok and all(np.array_equal(ex[k][lo:lo + K].cpu().numpy(), oex[k]) for k in oex)
            if planes:
                got = obs[lo:lo + K]
                got = got.view(torch.int16).cpu().numpy().view(np.uint16) if got.dtype == torch.bfloat16 else got.cpu().numpy()
                ok = ok and np.array_equal(got, last[0])
            ok = ok and np.array_equal(reward[lo:lo + K].cpu().numpy(), last[1]) and np.array_equal(done[lo:lo + K].cpu().numpy(), last[2])
        parity = bool(sum_over_ranks(0.0 if ok else 1.0) == 0.0)
        if not parity:
            raise SystemExit("bench.py: the timed CUDA state differs from the oracle -- refusing to report a number")

    # ---- roofline of the one kernel in a tick: algorithmic bytes per env-step (SURVEY 8d) x envs per launch / launch time
    C, P = env.C, env.P
    b_o = {"bf16": 2, "f32": 4, "i8": 1}[a.obs_dtype]
    M = 30  # per-env metadata + I/O actually moved: meta 8 r + 8 w, actions 2, reward 8, done + winner 2 (SURVEY 8d rounds this up to 48)
    grid_bytes = {"bits10": 32, "bits": 48}.get(a.layout, C)  # state bytes per game as stored (SURVEY 8d: C * b_g)
    if a.layout == "trail":
        grid_bytes = 0
    if P:
        bytes_per_env_step = grid_bytes * (1 + f_reset) + 2 * P * C * b_o + M
    else:  # pure tick (SURVEY 8d): <=4 sectors read+written, one metadata sector each way, reset amortisation
        bytes_per_env_step = 320 + f_reset * grid_bytes
        if a.layout == "trail":
            bytes_per_env_step = 64 + 32 + M - 16
    launch_ms = ms / (a.steps * TPS)
    achieved = bytes_per_env_step * N / (launch_ms * 1e-3) / 1e9
    kernel = {"bits10": "step_bits_kernel<false,10,...>", "bits": "step_bits_kernel<true,...>", "trail": "step_trail_kernel"}.get(
        a.layout, "step_sparse_kernel" if (not P and C >= 1024) else "step_tile_kernel")
    traffic, traffic_src = traffic_of("%s_%s_%s_%d" % (a.layout, a.obs_dtype, a.enc, N))
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "kernel": kernel, "state_bytes_per_game": grid_bytes,
                "bytes_per_env_step": bytes_per_env_step, "reset_fraction": f_reset,
                "envs_per_launch": N, "launch_ms": launch_ms, "frac_of_8TBs_nominal": achieved / 8000.0}
    del obs
    torch.cuda.empty_cache()

    # ---- e2e: the same workload through the host-buffer C-ABI front end (pinned host arrays in, host arrays out), steps pipelined
    e2e = None
    if not a.no_e2e:
        host_tape = [t.cpu().numpy() for t in tape]

        def e2e_leg(dtc, pipelined):
            h = HostTron(N, W, W, obs_dtype=dtc, obs_enc=enc_code, reward="ddqn", seed=0, env_id_base=rank * N, n_chunks=16, layout=a.layout,
                         double_buffer=pipelined)
            h.reset()
            for i in range(2):
                h.step(host_tape[i & 3])
            barrier()
            t0 = time.perf_counter()
            if pipelined:
                h.step_begin(host_tape[0])
                for i in range(a.e2e_steps):
                    if i + 1 < a.e2e_steps:
                        h.step_begin(host_tape[(i + 1) & 3])
                    h.step_wait()
            else:
                for i in range(a.e2e_steps):
                    h.step(host_tape[i & 3])
            dt_ = max_over_ranks(time.perf_counter() - t0)
            barrier()
            chk = float(h.reward2[(a.e2e_steps - 1) % len(h.reward2)][:1024].sum())
            h.close()
            return sum_over_ranks(float(N * a.e2e_steps)) / dt_, dt_, chk

        es8 = 1
        d2h_bytes = N * (2 * P * C * es8 + 8 + 2)
        # measured PCIe ceiling of this box: every rank copies 1 GiB device -> NUMA-local pinned host memory at the same time
        # (buffers are allocated and touched BEFORE the barrier, so that the timed copies of the ranks really overlap: the
        # library's own tron_host_copy_bandwidth allocates inside the call, and the allocation skew between ranks is longer than its copies)
        def concurrent_copy_peak(direction, nbytes, repeats):
            import ctypes as C
            from tron_b200 import _lib
            lib = _lib.load()
            hp = C.c_void_p()
            _lib.check(lib.tron_host_alloc(C.byref(hp), nbytes), "tron_host_alloc")  # pinned, on the GPU's NUMA node
            try:
                hbuf = torch.frombuffer((C.c_uint8 * nbytes).from_address(hp.value), dtype=torch.uint8)
                hbuf.fill_(1)
                dbuf = torch.ones(nbytes, dtype=torch.uint8, device=dev)
                src, dst = (dbuf, hbuf) if direction == "d2h" else (hbuf, dbuf)
                dst.copy_(src, non_blocking=True)
                torch.cuda.synchronize()
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(repeats):
                    dst.copy_(src, non_blocking=True)
                e1.record(); torch.cuda.synchronize()
                gbps = nbytes * repeats / (e0.elapsed_time(e1) * 1e-3) / 1e9
                del hbuf, dbuf, src, dst
            finally:
                barrier()
                _lib.check(lib.tron_host_free(hp), "tron_host_free")
            return gbps
        pcie_d2h = concurrent_copy_peak("d2h", 1 << 30, 8 if world > 1 else 3)
        pcie_h2d = concurrent_copy_peak("h2d", 1 << 28, 8 if world > 1 else 3)
        pcie_sum = sum_over_ranks(pcie_d2h)
        v_pipe, dt_pipe, chk = e2e_leg(abi.I8, True)
        v_block, _, _ = e2e_leg(abi.I8, False)
        achieved_pcie = d2h_bytes * a.e2e_steps / dt_pipe / 1e9  # this rank's share; max-over-ranks time
        e2e = {"value": v_pipe, "unit": UNIT, "h2d_bytes_per_step": 2 * N, "d2h_bytes_per_step": d2h_bytes, "steps": a.e2e_steps,
               "obs_dtype": "i8 (the reference's Game.step returns integer arrays, tron/map.py:83-84)",
               "api": "tron_host_env_step_begin/_wait (pinned NUMA-local host buffers, 16 chunks, copy stream behind the tick kernels, two steps in flight)",
               "blocking_api": {"value": v_block, "unit": UNIT, "api": "tron_host_env_step (one step at a time)"},
               "roofline": {"bound": "pcie", "achieved": achieved_pcie, "peak": pcie_d2h, "unit": "GB/s", "frac": achieved_pcie / pcie_d2h,
                            "peak_source": "measured in this run: back-to-back 1 GiB cudaMemcpyAsync device -> pinned host per rank, all ranks started together behind a barrier",
                            "h2d_peak": pcie_h2d, "aggregate_d2h_peak_all_ranks": pcie_sum},
               "checksum": chk}
        if a.obs_dtype != "i8" and P:  # the same call with the headline's observation dtype (2x / 4x the PCIe bytes)
            v2, _, _ = e2e_leg(dt_code, True)
            e2e["%s_obs_variant" % a.obs_dtype] = {"value": v2, "unit": UNIT, "d2h_bytes_per_step": N * (2 * P * C * b_o + 10)}

    # ---- epsilon-greedy action streams (SURVEY 8d proxy computed in-kernel), every rank
    streams = None
    if a.streams:
        streams = []
        obs_e = torch.empty((N, 2, P, W + 2, W + 2), dtype=tdt, device=dev) if P else None
        for eps in (1.0, 0.5, 0.1, 0.003):
            env_e = BatchedTron(N, W, W, device=dev, obs_dtype=tdt, obs_enc=a.enc, reward="ddqn", seed=3, env_id_base=rank * N, layout=a.layout,
                                policy="free_eps", policy_epsilon=eps)
            env_e.reset()
            for i in range(40):  # let episode lengths reach their stationary mix
                env_e.step(obs=obs_e, reward=reward, done=done, winner=winner, want_ep_len=False)
            torch.cuda.synchronize()
            q0 = env_e.stats_dict()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n_t = 2 * TPS
            for i in range(n_t):
                env_e.step(obs=obs_e, reward=reward, done=done, winner=winner, want_ep_len=False)
            e1.record(); torch.cuda.synchronize()
            q1 = env_e.stats_dict()
            fe = sum_over_ranks(float(q1["episodes"] - q0["episodes"])) / sum_over_ranks(float(q1["env_steps"] - q0["env_steps"]))
            be = (grid_bytes * (1 + fe) + 2 * P * C * b_o + M - 2) if P else bytes_per_env_step
            ms_e = max_over_ranks(e0.elapsed_time(e1))
            rate = world * N * n_t / (ms_e * 1e-3)
            streams.append({"epsilon": eps, "value": rate, "unit": UNIT, "n_gpus": world, "reset_fraction": fe, "bytes_per_env_step": be,
                            "frac_of_peak": rate / world * be / 1e9 / peak})
            del env_e
        del obs_e
        torch.cuda.empty_cache()
    del env
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs
    configs = None
    if not a.no_configs:
        configs = {}
        # #5: 64x64, 2M envs per GPU, pure tick, on-device counter-based RNG for actions and spawns, trail-list state
        n5 = 1 << 21
        env5 = BatchedTron(n5, 64, 64, device=dev, obs_enc="none", reward="ddqn", seed=0, env_id_base=rank * n5, layout="trail")
        env5.reset()
        r5 = torch.empty((n5, 2), dtype=torch.float32, device=dev); d5 = torch.empty(n5, dtype=torch.uint8, device=dev); w5 = torch.empty(n5, dtype=torch.uint8, device=dev)
        for _ in range(40):
            env5.step(reward=r5, done=d5, winner=w5, want_ep_len=False)
        torch.cuda.synchronize()
        s0 = env5.stats_dict()
        smp = ClockSampler(local)
        if rank == 0:
            smp.start(); time.sleep(0.1)
        barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw0 = time.perf_counter()
        n_t = 8 * TPS
        e0.record()
        for _ in range(n_t):
            env5.step(reward=r5, done=d5, winner=w5, want_ep_len=False)
        e1.record(); torch.cuda.synchronize(); barrier()
        tw1 = time.perf_counter()
        ms5 = max_over_ranks(e0.elapsed_time(e1))
        s1 = env5.stats_dict()
        f5 = (s1["episodes"] - s0["episodes"]) / max(1, s1["env_steps"] - s0["env_steps"])
        b5 = 64 + 32 + 10  # 64 hot bytes read, header + the one changed list uint4 written, reward / done / winner
        v5 = world * n5 * n_t / (ms5 * 1e-3)
        tr5, tr5_src = traffic_of("trail_none_64_%d" % n5)
        configs["cfg5"] = {"workload": "BASELINE config #5: 64x64 grid, %d envs/GPU, pure tick (no observations), on-device Philox policy + spawns, trail-list state" % n5,
                           "value": v5, "unit": UNIT, "n_gpus": world, "ticks": n_t, "ms_per_tick": ms5 / n_t, "reset_fraction": f5,
                           "mean_episode_ticks": (s1["ep_ticks"] - s0["ep_ticks"]) / max(1, s1["episodes"] - s0["episodes"]),
                           "roofline": {"bound": "hbm", "achieved": v5 / world * b5 / 1e9, "peak": peak, "unit": "GB/s", "frac": v5 / world * b5 / 1e9 / peak,
                                        "bytes_per_env_step": b5, "traffic": tr5, "traffic_source": tr5_src, "kernel": "step_trail_kernel",
                                        "note": "latency / issue bound, not bandwidth bound: see DESIGN.md section 6 and profiles/r2_step_trail_64x64_2M.json"},
                           "clocks": smp.stop(tw0, tw1) if rank == 0 else None}
        # the same games advanced 16 ticks per launch (tron_step_many: state stays in registers between ticks, outputs [T,N] per tick)
        for _ in range(2):
            env5.step_many(16)
        torch.cuda.synchronize(); barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(TPS // 4):
            env5.step_many(16)
        e1.record(); torch.cuda.synchronize()
        ms5m = max_over_ranks(e0.elapsed_time(e1))
        configs["cfg5"]["step_many_16_ticks_per_launch"] = {"value": world * n5 * 16 * (TPS // 4) / (ms5m * 1e-3), "unit": UNIT, "n_gpus": world}
        del env5
        # the same pure tick under the epsilon-greedy proxy policy (SURVEY 8d): long episodes, the lists outgrow the 12 hot entries and
        # "is this cell free?" goes through the occupancy bitmap in the cold area
        st5 = []
        for eps in (0.5, 0.1, 0.003):
            env_e = BatchedTron(n5, 64, 64, device=dev, obs_enc="none", reward="ddqn", seed=3, env_id_base=rank * n5, layout="trail",
                                policy="free_eps", policy_epsilon=eps)
            env_e.reset()
            for _ in range(300):  # episode lengths reach their stationary mix (mean 31 ticks at epsilon 0.003)
                env_e.step(reward=r5, done=d5, winner=w5, want_ep_len=False)
            torch.cuda.synchronize()
            q0 = env_e.stats_dict()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(2 * TPS):
                env_e.step(reward=r5, done=d5, winner=w5, want_ep_len=False)
            e1.record(); torch.cuda.synchronize()
            q1 = env_e.stats_dict()
            ms_e = max_over_ranks(e0.elapsed_time(e1))
            st5.append({"epsilon": eps, "value": world * n5 * 2 * TPS / (ms_e * 1e-3), "unit": UNIT, "n_gpus": world,
                        "reset_fraction": sum_over_ranks(float(q1["episodes"] - q0["episodes"])) / sum_over_ranks(float(q1["env_steps"] - q0["env_steps"])),
                        "mean_episode_ticks": (q1["ep_ticks"] - q0["ep_ticks"]) / max(1, q1["episodes"] - q0["episodes"])})
            del env_e
        configs["cfg5"]["eps_greedy_streams"] = st5
        del r5, d5, w5
        torch.cuda.empty_cache()
        # beyond BASELINE: the 64x64 board WITH fused bf16 observations (SURVEY 8d's last table row), trail lists + bulk-stored template rows
        n6 = 1 << 17
        env6 = BatchedTron(n6, 64, 64, device=dev, obs_dtype=torch.bfloat16, obs_enc="lut1", reward="ddqn", seed=0, env_id_base=rank * n6, layout="auto")
        o6 = env6.reset()
        r6 = torch.empty((n6, 2), dtype=torch.float32, device=dev); d6 = torch.empty(n6, dtype=torch.uint8, device=dev); w6 = torch.empty(n6, dtype=torch.uint8, device=dev)
        for _ in range(10):
            env6.step(obs=o6, reward=r6, done=d6, winner=w6, want_ep_len=False)
        torch.cuda.synchronize(); barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(TPS):
            env6.step(obs=o6, reward=r6, done=d6, winner=w6, want_ep_len=False)
        e1.record(); torch.cuda.synchronize()
        ms6 = max_over_ranks(e0.elapsed_time(e1))
        v6 = world * n6 * TPS / (ms6 * 1e-3)
        b6 = 64 + 32 + 2 * 66 * 66 * 2 + 10  # hot state read, header + one list uint4 written, both observation planes, reward / done / winner
        tr6, tr6_src = traffic_of("trail_bf16_lut1_64_%d" % n6)
        configs["large_grid_fused_obs"] = {"workload": "64x64 grid, %d envs/GPU, fused bf16 1-plane observations, on-device Philox policy, state layout %s" % (n6, env6.layout),
                                           "value": v6, "unit": UNIT, "n_gpus": world, "ticks": TPS, "ms_per_tick": ms6 / TPS,
                                           "roofline": {"bound": "hbm", "achieved": v6 / world * b6 / 1e9, "peak": peak, "unit": "GB/s", "frac": v6 / world * b6 / 1e9 / peak,
                                                        "bytes_per_env_step": b6, "traffic": tr6, "traffic_source": tr6_src, "kernel": "step_trail_obs_bulk_kernel"}}
        del env6, o6, r6, d6, w6
        torch.cuda.empty_cache()

        from tron_b200 import dropin
        dropin.install()
        import DDQN
        import DQN
        # #3: DQN.py survivor loop, 65,536 self-play envs on each GPU (independent replicas), frame-sharing GPU replay
        tm3 = {}
        DQN.train(n_envs=65536, iterations=1, device=dev, seed=rank, amp=True)  # warm-up (cuDNN autotune, allocator)
        torch.cuda.synchronize(); barrier()
        DQN.train(n_envs=65536, iterations=2, device=dev, seed=rank, timings=tm3, amp=True)
        tot3 = max_over_ranks(tm3["q_forward_ms"] + tm3["env_replay_ms"] + tm3["learn_ms"])
        configs["cfg3"] = {"workload": "BASELINE config #3: DQN.py survivor loop, 65,536 batched self-play envs per GPU, 1-plane f32 observations, frame-sharing GPU replay",
                           "value": world * 65536 * tm3["ticks"] / (tot3 * 1e-3), "unit": UNIT, "n_gpus": world, "ticks": tm3["ticks"], "learn_steps": tm3["learn_steps"],
                           "ms": {"q_forward": max_over_ranks(tm3["q_forward_ms"]), "env_replay": max_over_ranks(tm3["env_replay_ms"]), "learn": max_over_ranks(tm3["learn_ms"])},
                           "env_replay_fraction_of_loop": tm3["env_replay_ms"] / (tm3["q_forward_ms"] + tm3["env_replay_ms"] + tm3["learn_ms"]),
                           "acting_forward": "bf16 autocast", "state_layout": tm3["layout"], "replay": tm3["replay"]}
        # #4: DDQN.py, 131,072 envs per GPU (1M over 8 GPUs), pop_up 3-plane bf16 observations, NCCL all-reduce of the Q-net gradient
        tm4 = {}
        DDQN.train(n_envs=131072, env_steps=8, device=dev, seed=0, amp=True)  # warm-up
        torch.cuda.synchronize(); barrier()
        DDQN.train(n_envs=131072, env_steps=48, device=dev, seed=0, amp=True, timings=tm4, warmup_steps=8)
        tot4 = max_over_ranks(tm4["q_forward_ms"] + tm4["env_replay_ms"] + tm4["learn_ms"])
        configs["cfg4"] = {"workload": "BASELINE config #4: DDQN.py loop, 131,072 envs per GPU, pop_up 3-plane bf16 observations, frame-sharing GPU replay, "
                                       "one learn step (batch 64) every 4 ticks, flat-bucket NCCL all-reduce overlapped with the next tick",
                           "value": world * 131072 * tm4["ticks"] / (tot4 * 1e-3), "unit": UNIT, "n_gpus": world, "ticks": tm4["ticks"], "learn_steps": tm4["learn_steps"],
                           "ms": {"q_forward": max_over_ranks(tm4["q_forward_ms"]), "env_replay": max_over_ranks(tm4["env_replay_ms"]),
                                  "learn": max_over_ranks(tm4["learn_ms"]), "allreduce": max_over_ranks(tm4["allreduce_ms"])},
                           "allreduce_us_per_call": {"min": max_over_ranks(tm4["allreduce_us_min"]), "median": max_over_ranks(tm4["allreduce_us_median"]),
                                                     "max": max_over_ranks(tm4["allreduce_us_max"]),
                                                     "note": "device time from 'backward finished' to 'reduced gradient ready' on the side stream; includes waiting "
                                                             "for the slowest rank; overlapped with the next tick's forward + env step"},
                           "allreduce_calls": tm4["allreduce_calls"],
                           "learn_ms_per_step": max_over_ranks(tm4["learn_ms"]) / max(1, tm4["learn_steps"]),
                           "env_replay_fraction_of_loop": tm4["env_replay_ms"] / (tm4["q_forward_ms"] + tm4["env_replay_ms"] + tm4["learn_ms"]),
                           "acting_forward": "bf16 autocast", "state_layout": tm4["layout"], "replay": tm4["replay"]}
        torch.cuda.empty_cache()

    # ---- launch-bound regime of the literal config #2 size: 4096 envs, T ticks per launch (tron_step_many)
    small = None
    if rank == 0:
        env_s = BatchedTron(4096, W, W, device=dev, obs_dtype=tdt, obs_enc=a.enc, seed=0, layout=a.layout)
        env_s.reset()
        env_s.step_many(64)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            env_s.step_many(64)
        e1.record(); torch.cuda.synchronize()
        small = {"envs": 4096, "ticks_per_launch": 64, "value": 4096 * 64 * 10 / (e0.elapsed_time(e1) * 1e-3), "unit": UNIT,
                 "note": "literal BASELINE config #2 size: L2-resident and launch-bound, obs written every tick"}
        from tron_b200.batch_env import GraphedStep
        gs = GraphedStep(BatchedTron(4096, W, W, device=dev, obs_dtype=tdt, obs_enc=a.enc, seed=1, layout=a.layout), policy="random", ticks_per_replay=16)
        gs.env.reset()
        gs.replay(); torch.cuda.synchronize()
        e0.record()
        for _ in range(40):
            gs.replay()
        e1.record(); torch.cuda.synchronize()
        small["cuda_graph_16_ticks_per_replay"] = {"value": 4096 * 16 * 40 / (e0.elapsed_time(e1) * 1e-3), "unit": UNIT,
                                                   "note": "one tron_step launch per tick, 16 ticks captured in a CUDA graph, device-side RNG counter"}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cores = os.cpu_count() or 1
        v, sample = cpu_c_port(W, dt_code, enc_code, a.cpu_seconds, cores)
        pv, psteps = cpu_python_loop(W, 1500, cores)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
               "python_loop_port": {"value": pv, "unit": UNIT, "cores": cores, "sample": "%d env-steps, pure-Python port of the reference's Game.step loop" % psteps}}

    if rank == 0:
        if e2e is not None and cpu is not None:  # the end-to-end number next to both CPU arms measured in this run
            e2e["vs_cpu_arms"] = {"c_oracle_port_all_cores": e2e["value"] / cpu["value"], "python_loop_port_all_cores": e2e["value"] / cpu["python_loop_port"]["value"],
                                  "cores": cpu["cores"], "note": "the driver's e2e_ratio uses the --impl reference line (the live reference's Python loop)"}
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i8", "data": "synthetic", "config": workload_config(a, N),
               "timed_region_s": ms * 1e-3, "ms_per_tick": launch_ms, "parity_in_run": parity,
               "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": a.steps * TPS, "clocks": clocks,
               "eps_greedy_streams": streams, "configs": configs, "small_n": small,
               "episode_stats": {"reset_fraction": f_reset, "mean_episode_ticks": (st1["ep_ticks"] - st0["ep_ticks"]) / max(1, st1["episodes"] - st0["episodes"])}}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)
