#!/usr/bin/env python
"""Randomised differential test: random (layout, size, encoding, dtype, slide mode, policy, spawn mode, tapes / RNG, step /
step_many / masked reset / terminal frames / replay ring / one obs buffer reused every tick) configurations, CUDA (through the C ABI) vs the CPU oracle, bit for bit.
usage: fuzz_gpu.py [seconds] [seed] [--seeds K] [--debug-checks] [--log FILE]
  --seeds K        run K seeds of 60 cases each instead of a time budget
  --debug-checks   (with TRON_B200_DEBUG=1: the range-checked library) print the device-side violation count at the end"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import c_oracle as oc  # noqa: E402
from tron_b200 import abi  # noqa: E402
from _gpu import TORCH_DT, assert_same_state, assert_same_step, make_pair, to_np  # noqa: E402


def replay_case(rng, case):
    """random pushes into the transition ring + one-launch sample/gather vs the oracle"""
    from tron_b200.replay import ReplayRing
    dt = int(rng.choice([abi.BF16, abi.F32, abi.I8]))
    F = int(rng.choice([16, 25, 144, 432]))
    cap = int(rng.choice([7, 64, 1000, 4097]))
    seed = int(rng.integers(0, 1 << 30))
    ring, oring = ReplayRing(cap, (F,), TORCH_DT[dt], seed=seed), oc.OracleRing(cap, F, dt)
    for _ in range(int(rng.integers(1, 5))):
        stride = int(rng.choice([1, 2]))
        n = int(rng.integers(1, 2 * cap)) * stride
        s = torch.as_tensor(rng.integers(-10, 11, size=(n, F))).to(TORCH_DT[dt]); s2 = torch.as_tensor(rng.integers(-10, 11, size=(n, F))).to(TORCH_DT[dt])
        a = rng.integers(0, 4, size=n).astype(np.uint8); r = rng.normal(size=n).astype(np.float32); d = rng.integers(0, 2, size=n // stride).astype(np.uint8)
        ring.push(s.cuda(), s2.cuda(), torch.as_tensor(a), torch.as_tensor(r), torch.as_tensor(d), done_stride=stride)
        off, chunk = 0, cap - cap % stride
        while off < n:  # the oracle ring takes at most `capacity` transitions per call, like the ABI
            m = min(chunk, n - off)
            oring.push(to_np(s)[off:off + m], to_np(s2)[off:off + m], a[off:off + m], r[off:off + m], d[off // stride:(off + m) // stride], done_stride=stride)
            off += m
        for name in ("state", "next_state", "action", "reward", "done"):
            assert np.array_equal(to_np(getattr(ring, name)), getattr(oring, name)), "replay case %d: %s" % (case, name)
    k = int(rng.integers(1, len(oring) + 1))
    c = int(rng.integers(0, 1000))
    got = ring.sample(k, counter=c, want_indices=True)
    idx = oc.sample_indices(len(oring), k, seed, c)
    assert np.array_equal(got[5].cpu().numpy(), idx) and len(set(idx.tolist())) == k, "replay case %d: indices" % case
    for gg, ww in zip(got[:5], oring.gather(idx, abi.F32)):
        assert np.array_equal(to_np(gg).reshape(ww.shape), ww), "replay case %d: gather" % case
    return "case %d: replay ring cap=%d F=%d dt=%d k=%d" % (case, cap, F, dt, k)


def one_case(rng, case):
    if rng.random() < 0.08:
        return replay_case(rng, case)
    layout = rng.choice(["tile8", "bits10", "trail", "bits", "bits"])
    if layout == "bits":
        W = int(rng.choice([2, 3, 5, 8, 10, 10, 11]))
        H = W if rng.random() < 0.7 else int(rng.integers(2, 128 // W + 1))
    else:
        W = 10 if layout == "bits10" else int(rng.choice([2, 3, 5, 8, 10, 12, 15, 21, 32, 47, 64]))
        H = W if (layout == "bits10" or rng.random() < 0.8) else int(rng.integers(2, 20))
    N = int(rng.choice([1, 7, 128, 129, 1000, 3000])) if W <= 32 else int(rng.choice([3, 40, 300]))
    enc = int(rng.choice([abi.ENC_NONE, abi.ENC_LUT1, abi.ENC_POPUP3, abi.ENC_POPUP3_CONST]))
    dt = int(rng.choice([abi.BF16, abi.F32, abi.I8]))
    slide = abi.SLIDE_NONE if layout == "bits10" else int(rng.choice([abi.SLIDE_NONE, abi.SLIDE_NONE, abi.SLIDE_ICE, abi.SLIDE_TEMPER, abi.SLIDE_TAPE]))
    policy = int(rng.choice([abi.POLICY_UNIFORM, abi.POLICY_FREE_EPS]))
    kw = dict(layout=layout, obs_dtype=dt, obs_enc=enc, const_plane=float(rng.integers(-3, 9)), seed=int(rng.integers(0, 1 << 30)),
              env_id_base=int(rng.integers(0, 1 << 20)), slide_mode=slide, slide_rate=float(rng.choice([0.0, 0.15, 0.7])),
              spawn_mode=int(rng.integers(0, 2)), policy=policy, policy_epsilon=float(rng.choice([0.0, 0.05, 0.5])),
              auto_reset=bool(rng.random() < 0.8), reward=str(rng.choice(["ddqn", "survivor", "acktr2"])))
    g, o = make_pair(N, W, H, **kw)
    a, b = g.reset(), o.reset()
    # one obs buffer for every plain step (the delta-store path of the 10x10 bit-plane kernels), seeded with full rows by observe()
    buf = g.env.observe(g.env.new_obs()) if enc != abi.ENC_NONE and rng.random() < 0.5 else None
    desc = "case %d: %s %dx%d N=%d enc=%d dt=%d slide=%d policy=%d auto=%s reuse_obs=%s" % (case, layout, W, H, N, enc, dt, slide, policy,
                                                                                         kw["auto_reset"], buf is not None)
    if os.environ.get("FUZZ_VERBOSE"):
        print(desc, flush=True)
    assert (a is None and b is None) or np.array_equal(a, b), desc
    if slide == abi.SLIDE_TEMPER:
        assert np.array_equal(g.env.slide_params.cpu().numpy(), o.slide_params), desc + " temper draws"
    terminal_ok = layout != "trail" or abi.trail_bulk_ok(W, H, enc, dt)  # trail: bulk-store kernel only
    want_terminal = enc != abi.ENC_NONE and terminal_ok and rng.random() < 0.3
    use_tape = rng.random() < 0.5
    for t in range(int(rng.integers(5, 40))):
        act = rng.integers(0, 4, size=(N, 2)).astype(rng.choice([np.uint8, np.int32, np.int64])) if use_tape else None
        st = rng.integers(0, 2, size=(N, 2)).astype(np.uint8) if slide == abi.SLIDE_TAPE else None
        r = rng.random()
        if r < 0.15 and slide != abi.SLIDE_TAPE:
            T = int(rng.integers(2, 6))
            acts = rng.integers(0, 4, size=(T, N, 2)).astype(np.uint8) if use_tape else None
            every = bool(rng.integers(0, 2))
            assert_same_step(g.step_many(T, actions=acts, obs_every_tick=every), o.step_many(T, actions=acts, obs_every_tick=every), desc + " step_many")
        elif r < 0.2:
            mask = rng.integers(0, 2, size=N).astype(np.uint8)
            x, y = g.reset(mask=mask), o.reset(mask=mask)
            assert (x is None and y is None) or np.array_equal(x, y), desc + " masked reset"
        elif want_terminal:
            gt = torch.full(tuple(a.shape), 3, dtype=TORCH_DT[dt], device="cuda")
            ot = to_np(torch.full(tuple(a.shape), 3, dtype=TORCH_DT[dt])).copy()
            res = g.env.step(None if act is None else torch.as_tensor(act), slide_tape=st, obs_terminal=gt)
            assert_same_step(tuple(to_np(x) for x in res), o.step(act, slide_tape=st, obs_terminal=ot), desc + " tick %d" % t)
            assert np.array_equal(to_np(gt), ot), desc + " terminal frames, tick %d" % t
        elif buf is not None:
            res = g.env.step(None if act is None else torch.as_tensor(act), slide_tape=st, obs=buf)
            assert_same_step(tuple(to_np(x) for x in res), o.step(act, slide_tape=st), desc + " tick %d (reused obs)" % t)
        else:
            assert_same_step(g.step(act, slide_tape=st), o.step(act, slide_tape=st), desc + " tick %d" % t)
    if slide == abi.SLIDE_TEMPER:
        assert np.array_equal(g.env.extra.cpu().numpy(), o.extra()), desc + " extra"
    assert_same_state(g, o, desc)
    assert np.array_equal(g.stats, o.stats), desc
    return desc


def violations():
    """(count, first code) of the range-checked debug library; None for the release library"""
    import ctypes as C
    from tron_b200 import _lib
    n, code = C.c_uint64(), C.c_int32()
    rc = _lib.load().tron_debug_violations(C.byref(n), C.byref(code))
    return None if rc != 0 else (n.value, code.value)


if __name__ == "__main__":
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("seconds", nargs="?", type=float, default=60.0)
    ap.add_argument("seed", nargs="?", type=int, default=0)
    ap.add_argument("--seeds", type=int, default=0)
    ap.add_argument("--debug-checks", action="store_true")
    ap.add_argument("--log", default=None)
    a = ap.parse_args()
    log = open(a.log, "a") if a.log else None

    def say(msg):
        print(msg, flush=True)
        if log:
            log.write(msg + "\n"); log.flush()
    t0, n = time.time(), 0
    if a.seeds:
        for sd in range(a.seed, a.seed + a.seeds):
            rng = np.random.default_rng(sd)
            for case in range(60):
                last = one_case(rng, case)
                n += 1
            say(last)
    else:
        rng = np.random.default_rng(a.seed)
        while time.time() - t0 < a.seconds:
            last = one_case(rng, n)
            n += 1
            if n % 25 == 0:
                say(last)
    say("fuzz ok: %d random configurations bit-exact vs oracle in %.0f s (seed %d)" % (n, time.time() - t0, a.seed))
    if a.debug_checks:
        v = violations()
        if v is None:
            say("debug checks: release library loaded (set TRON_B200_DEBUG=1)")
            sys.exit(2)
        say("debug checks: violations %d (first code %d)" % v)
        sys.exit(0 if v[0] == 0 else 1)
