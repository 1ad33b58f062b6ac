"""The state replay ring (StateRing, replay_states_sample_gather): it stores each tick's pre-tick env state and actions and
re-simulates sampled transitions.  Checked bit for bit against the frame ring driven by a twin env, against explicit transitions
(oracle and GPU), over a long horizon, under a captured CUDA graph with the device counter, on its own reused obs buffer, in the
debug build and in the training loops; plus the status codes of every sample / gather entry point."""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tron_b200 import abi  # noqa: E402

TORCH_DT = {abi.BF16: torch.bfloat16, abi.F32: torch.float32, abi.I8: torch.int8}


def _bits(t):
    """exact bit pattern of a tensor (so -0.0 != 0.0 and NaN payloads count)"""
    return t.contiguous().view(torch.uint8).cpu().numpy()


def _env(N, W, H, layout, dt, enc, **kw):
    from tron_b200.batch_env import BatchedTron
    return BatchedTron(N, W, H, layout=layout, obs_dtype=TORCH_DT[dt], obs_enc=enc, seed=4, **kw)


def _tape(rng, N):
    """uniform moves with ~3 % bad actions (>= 4: the game is left untouched for that tick)"""
    act = rng.integers(0, 4, size=(N, 2)).astype(np.uint8)
    bad = rng.random((N, 2)) < 0.03
    act[bad] = rng.choice(np.array([4, 7, 255], np.uint8), size=int(bad.sum()))
    return torch.as_tensor(act).cuda()


def run_equivalence(N, W, H, layout, dt, enc, out_dtype, S=4, T=11, **kw):
    """two envs with the same seed follow one action tape; FrameRing(S + 1, keep_terminal) and StateRing(S) must hand out identical
    samples after every tick"""
    from tron_b200.replay import FrameRing, StateRing
    ea, eb = _env(N, W, H, layout, dt, enc, **kw), _env(N, W, H, layout, dt, enc, **kw)
    fr, sr = FrameRing(ea, S + 1, keep_terminal=True, seed=9), StateRing(eb, S, seed=9)
    fr.begin()
    obs = sr.begin(obs=eb.new_obs())
    rng = np.random.default_rng(2)
    for t in range(T):
        a = _tape(rng, N)
        fr.step(actions=a)
        sr.step(actions=a, obs=obs)
        assert len(sr) == len(fr) == min(t + 1, S) * 2 * N
        for k in (64, len(sr)):
            want = fr.sample(k, out_dtype, counter=t, want_indices=True)
            got = sr.sample(k, out_dtype, counter=t, want_indices=True)
            for name, w, g in zip(("s", "a", "r", "s2", "d", "idx"), want, got):
                assert w.dtype == g.dtype and w.shape == g.shape, name
                assert np.array_equal(_bits(w), _bits(g)), (t, k, name)
    return ea, eb


EQUIV_CASES = [
    # (layout, W, H, env dtype, encoding, out dtype, extra env kwargs)
    ("bits10", 10, 10, abi.BF16, "popup3", torch.float32, {}),                       # DDQN
    ("bits10", 10, 10, abi.F32, "lut1", torch.bfloat16, {}),                         # DQN's obs into a bf16 batch
    ("bits10", 10, 10, abi.I8, "popup3_const", torch.float32, dict(const_plane=5.0)),
    ("bits10", 10, 10, abi.I8, "popup3_const", torch.float32, dict(const_plane=0.3)),
    ("bits10", 10, 10, abi.BF16, "popup3_const", torch.float32, dict(const_plane=0.3)),  # bf16-rounded before the f32 batch
    ("bits10", 10, 10, abi.BF16, "lut1", torch.float32, dict(lut=(5, 4, 3, 2, 1, -7))),
    ("bits", 10, 10, abi.BF16, "popup3", torch.float32, dict(slide_mode="ice", slide_rate=0.3)),
    ("bits", 10, 10, abi.BF16, "popup3", torch.float32, dict(slide_mode="temper")),
    ("bits", 7, 9, abi.BF16, "popup3", torch.float32, {}),                           # 99 cells: rows are not 16-byte chunks
    ("bits", 7, 9, abi.F32, "lut1", torch.bfloat16, dict(slide_mode="ice", slide_rate=0.3)),
    ("bits", 8, 8, abi.I8, "popup3_const", torch.float32, dict(const_plane=0.3, slide_mode="temper")),
]


@pytest.mark.parametrize("layout,W,H,dt,enc,out_dtype,kw", EQUIV_CASES,
                         ids=["%s-%dx%d-%d-%s-%s-%s" % (c[0], c[1], c[2], c[3], c[4], str(c[5])[6:], "-".join("%s=%s" % i for i in c[6].items()))
                              for c in EQUIV_CASES])
@pytest.mark.gpu
def test_state_ring_equals_frame_ring(layout, W, H, dt, enc, out_dtype, kw):
    run_equivalence(300, W, H, layout, dt, enc, out_dtype, **kw)


def _explicit_step(env, sr, a, obs):
    """one StateRing tick plus the transitions the DDQN loop would have stored for it: (s, a, r, s', d) per row, numpy"""
    N = env.N
    s = obs.clone()
    term = obs.clone()
    res = sr.step(actions=a, obs=obs, obs_terminal=term)
    s2 = torch.where(res.done.view(-1, 1, 1, 1, 1).bool(), term, res.obs)
    return (s.float().reshape(2 * N, -1).cpu().numpy(), sr.action_t[(sr.tick - 1) % sr.S].reshape(-1).cpu().numpy(),
            res.reward.reshape(-1).cpu().numpy(), s2.float().reshape(2 * N, -1).cpu().numpy(), res.done.cpu().numpy())


def _check_against(explicit, got, N):
    s, a, r, s2, d, idx = (x.cpu().numpy() for x in got)
    k = s.shape[0]
    s, s2 = s.reshape(k, -1).astype(np.float32), s2.reshape(k, -1).astype(np.float32)
    n = 0
    for j in range(k):
        tick, row = int(idx[j]) // (2 * N), int(idx[j]) % (2 * N)
        if tick not in explicit:
            continue
        es, ea, er, es2, ed = explicit[tick]
        assert np.array_equal(s[j], es[row]) and np.array_equal(s2[j], es2[row]), (tick, row)
        assert int(a[j, 0]) == int(ea[row]) and float(r[j, 0]) == float(er[row]) and float(d[j, 0]) == float(ed[row // 2]), (tick, row)
        n += 1
    return n


@pytest.mark.gpu
@pytest.mark.parametrize("dt,enc", [(abi.BF16, abi.ENC_LUT1), (abi.F32, abi.ENC_POPUP3), (abi.I8, abi.ENC_POPUP3_CONST)])
def test_state_ring_transitions_equal_the_explicit_ones(dt, enc):
    """every sampled transition equals the oracle's (s, a, r, s', d) of that tick (DDQN.py:264-308): s' of a finished game is its
    LAST frame, not the fresh game's first one"""
    from oracle import c_oracle as oc
    from tron_b200.batch_env import BatchedTron
    from tron_b200.replay import StateRing
    N, S, T = 600, 5, 13
    name = {abi.ENC_LUT1: "lut1", abi.ENC_POPUP3: "popup3", abi.ENC_POPUP3_CONST: "popup3_const"}[enc]
    env = BatchedTron(N, 10, 10, layout="bits10", obs_dtype=TORCH_DT[dt], obs_enc=name, seed=4, const_plane=2.0)
    o = oc.OracleEnv(N, 10, 10, obs_dtype=dt, obs_enc=enc, seed=4, const_plane=2.0)
    sr = StateRing(env, S, seed=9)
    obs = sr.begin(obs=env.new_obs())
    oobs = o.reset()
    explicit = {}
    finished = 0
    rng = np.random.default_rng(2)
    for t in range(T):
        act = rng.integers(0, 4, size=(N, 2)).astype(np.uint8)
        term = oobs.copy()
        nobs, rew, done, _, _ = o.step(act, obs_terminal=term)
        s2 = np.where(done.astype(bool)[:, None, None, None, None], term, nobs)
        explicit[t] = (oc.obs_to_float(oobs, dt).reshape(2 * N, -1), act.reshape(-1), rew.reshape(-1), oc.obs_to_float(s2, dt).reshape(2 * N, -1),
                       done.astype(np.float32))
        finished += int(done.sum())
        sr.step(actions=torch.as_tensor(act).cuda(), obs=obs)
        oobs = nobs
        n_ticks = min(t + 1, S)
        for k in (64, n_ticks * 2 * N):
            got = sr.sample(k, counter=t, want_indices=True)
            ticks = got[5].cpu().numpy() // (2 * N)
            assert len(set(got[5].cpu().numpy().tolist())) == k and ticks.min() >= t + 1 - n_ticks and ticks.max() <= t
            assert _check_against(explicit, got, N) == k
    assert finished > 0


@pytest.mark.gpu
def test_state_ring_long_horizon():
    """300 slots (far beyond the frame ring's old 64-slot cap), 700 ticks of epsilon-greedy play: transitions of the oldest tick
    still in the window equal the explicit transitions recorded when that tick was played"""
    from tron_b200.batch_env import BatchedTron
    from tron_b200.replay import StateRing
    N, S, T = 256, 300, 700
    env = BatchedTron(N, 10, 10, layout="bits10", obs_dtype=torch.bfloat16, obs_enc="popup3", seed=11)
    sr = StateRing(env, S, seed=3)
    obs = sr.begin(obs=env.new_obs())
    g = torch.Generator(device=env.device).manual_seed(0)
    oldest = T - S
    explicit = {}
    for t in range(T):
        q = torch.rand((2 * N, 4), device=env.device, generator=g)
        env.select_actions(q, 0.3, counter=env.counter, out=sr.actions_slot().view(-1))
        if t == oldest:
            explicit[t] = _explicit_step(env, sr, None, obs)
        else:
            sr.step(obs=obs)
    assert len(sr) == S * 2 * N
    hits = 0
    for c in range(6):
        got = sr.sample(4096, counter=100 + c, want_indices=True)
        ticks = got[5] // (2 * N)
        assert int(ticks.min()) >= oldest and int(ticks.max()) <= T - 1
        hits += _check_against(explicit, got, N)
    assert hits > 20


@pytest.mark.gpu
def test_state_ring_device_counter_graph():
    """ice-mode env on the device counter: S ticks of (random_actions -> StateRing.step) captured in one CUDA graph and replayed;
    the samples equal the transitions a twin env on the host counter records explicitly"""
    from tron_b200.batch_env import BatchedTron
    from tron_b200.replay import StateRing
    N, S = 512, 4
    kw = dict(layout="bits", obs_dtype=torch.bfloat16, obs_enc="popup3", seed=6, slide_mode="ice", slide_rate=0.4)
    ea, eb = BatchedTron(N, 10, 10, **kw), BatchedTron(N, 10, 10, **kw)
    ea.use_device_counter()
    sr = StateRing(ea, S, seed=5)
    obs = sr.begin(obs=ea.new_obs())
    twin = StateRing(eb, S, seed=5)
    tobs = twin.begin(obs=eb.new_obs())

    def body():
        for _ in range(S):
            ea.random_actions(out=sr.actions_slot())
            sr.step(obs=obs)

    def follow(record):  # the twin plays the S ticks just played, with the same actions
        explicit = {}
        for i in range(S):
            t = twin.tick
            a = sr.action_t[t % S].clone()
            if record:
                explicit[t] = _explicit_step(eb, twin, a, tobs)
            else:
                twin.step(actions=a, obs=tobs)
        return explicit

    body()  # warm-up outside capture
    follow(False)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        body()
    for rep in range(3):
        if rep:
            sr.tick += S  # the graph replays the same S slots: the next S ticks
        graph.replay()
        torch.cuda.synchronize()
        explicit = follow(True)
        assert sr.tick == twin.tick and int(ea.counter_dev.item()) == eb.counter
        assert torch.equal(ea.state, eb.state)
        got = sr.sample(len(sr), counter=rep, want_indices=True)
        assert _check_against(explicit, got, N) == len(sr)
        # the twin's own ring (host counter) samples the same tensors
        for w, g in zip(twin.sample(len(twin), counter=rep, want_indices=True), got):
            assert np.array_equal(_bits(w), _bits(g))


@pytest.mark.gpu
def test_state_ring_steps_its_own_obs_buffer():
    """a StateRing begun without a buffer steps its own `obs`: one tensor every tick, which the env reports as holding the previous
    observation (so BatchedTron.step stores only the changed parts of each row); its samples equal a twin ring's on an explicit
    buffer"""
    from tron_b200.replay import StateRing
    N, S, T = 300, 4, 11
    ea, eb = _env(N, 10, 10, "bits10", abi.BF16, "popup3"), _env(N, 10, 10, "bits10", abi.BF16, "popup3")
    sr, twin = StateRing(ea, S, seed=9), StateRing(eb, S, seed=9)
    assert sr.begin() is sr.obs
    ptr = sr.obs.data_ptr()
    tobs = twin.begin(obs=eb.new_obs())
    rng = np.random.default_rng(2)
    for t in range(T):
        a = _tape(rng, N)
        assert ea._obs_is_prev(sr.obs), t
        res = sr.step(actions=a)
        assert res.obs is sr.obs and sr.obs.data_ptr() == ptr, t
        twin.step(actions=a, obs=tobs)
        assert np.array_equal(_bits(sr.obs), _bits(tobs)), t
        for k in (64, len(sr)):
            for name, w, g in zip(("s", "a", "r", "s2", "d", "idx"), twin.sample(k, counter=t, want_indices=True),
                                  sr.sample(k, counter=t, want_indices=True)):
                assert np.array_equal(_bits(w), _bits(g)), (t, k, name)


def _call(sr, env_args, first, n_ticks, k, out, out_dtype=abi.F32, rs=None):
    from tron_b200 import _lib
    s, a, r, s2, d = out
    return _lib.load().replay_states_sample_gather(C.byref(rs or sr.rs), C.byref(env_args), first, n_ticks, k, 0, 0, s, s2, out_dtype,
                                                   a.data_ptr(), r.data_ptr(), d.data_ptr(), None, torch.cuda.current_stream().cuda_stream)


@pytest.mark.gpu
def test_state_ring_refusals():
    from tron_b200 import _lib
    from tron_b200.batch_env import BatchedTron
    from tron_b200.replay import StateRing
    N, S = 64, 3
    for layout in ("tile8", "trail"):
        with pytest.raises(ValueError, match="bit-plane"):
            StateRing(BatchedTron(N, 10, 10, layout=layout, obs_enc="lut1"), S)
    with pytest.raises(ValueError, match="tape"):
        StateRing(BatchedTron(N, 10, 10, layout="bits", slide_mode="tape"), S)
    with pytest.raises(ValueError, match="auto_reset"):
        StateRing(BatchedTron(N, 10, 10, layout="bits10", auto_reset=False), S)
    with pytest.raises(ValueError, match="observations"):
        StateRing(BatchedTron(N, 10, 10, layout="bits10", obs_enc="none"), S)
    env = BatchedTron(N, 10, 10, layout="bits10", obs_dtype=torch.bfloat16, obs_enc="popup3")
    sr = StateRing(env, S)
    obs = sr.begin(obs=env.new_obs())
    for _ in range(2):
        sr.step(obs=obs)
    with pytest.raises(ValueError):
        sr.sample(len(sr) + 1)
    with pytest.raises(ValueError):
        sr.sample(8, out_dtype=torch.int8)
    # the C entry point
    F = 3 * 144
    buf = torch.zeros(2 * 64 * F + 16, dtype=torch.float32, device=env.device)
    side = [torch.zeros((64, 1), dtype=dt, device=env.device) for dt in (torch.int64, torch.float32, torch.float32)]
    good = (buf.data_ptr(), side[0], side[1], buf.data_ptr() + 64 * F * 4, side[2])
    args = env._args()
    assert _call(sr, args, 0, 2, 64, good) == abi.OK
    torch.cuda.synchronize()
    assert _call(sr, args, 0, 2, 64, good, out_dtype=abi.I8) == abi.ERR_INVALID
    assert _call(sr, args, 0, 2, 64, (buf.data_ptr() + 4,) + good[1:]) == abi.ERR_ALIGN
    assert _call(sr, args, 0, 2, 64, good[:3] + (buf.data_ptr() + 8 + 64 * F * 4,) + good[4:]) == abi.ERR_ALIGN
    assert _call(sr, args, 0, S + 1, 64, good) == abi.ERR_INVALID            # n_ticks > S
    assert _call(sr, args, 0, 2, 2 * 2 * N + 1, good) == abi.ERR_INVALID     # k > n_ticks * rows
    bad = abi.ReplayStates.from_buffer_copy(sr.rs)
    bad.struct_size = 12
    assert _call(sr, args, 0, 2, 64, good, rs=bad) == abi.ERR_INVALID
    bad = abi.ReplayStates.from_buffer_copy(sr.rs)
    bad.slot_bytes = 16
    assert _call(sr, args, 0, 2, 64, good, rs=bad) == abi.ERR_INVALID
    for layout, extra in ((abi.LAYOUT_TILE8, {}), (abi.LAYOUT_TRAIL, {}), (abi.LAYOUT_BITS, dict(slide_mode=abi.SLIDE_TAPE))):
        other = BatchedTron(N, 10, 10, layout={abi.LAYOUT_TILE8: "tile8", abi.LAYOUT_TRAIL: "trail", abi.LAYOUT_BITS: "bits"}[layout],
                            obs_dtype=torch.bfloat16, obs_enc="popup3")
        a2 = other._args(**extra)
        assert _call(sr, a2, 0, 2, 64, good) == abi.ERR_UNSUPPORTED, layout
    with pytest.raises(_lib.TronError):
        _lib.check(_call(sr, args, 0, S + 1, 64, good), "replay_states_sample_gather")


@pytest.mark.gpu
def test_sample_gather_status_codes():
    """replay_gather, replay_sample_gather and replay_frames_sample_gather on real, correctly sized buffers: the valid call returns
    OK and every refused call differs from it in exactly one argument"""
    from tron_b200 import _lib
    from tron_b200.batch_env import BatchedTron
    from tron_b200.replay import FrameRing, ReplayRing
    lib, stream = _lib.load(), torch.cuda.current_stream().cuda_stream
    k, F = 64, 3 * 144
    buf = torch.zeros(2 * k * F + 16, dtype=torch.float32, device="cuda")
    side = [torch.zeros((k, 1), dtype=dt, device="cuda") for dt in (torch.int64, torch.float32, torch.float32)]
    good = [buf.data_ptr(), buf.data_ptr() + k * F * 4] + [t.data_ptr() for t in side]  # s, s', a, r, d
    idx = torch.arange(k, dtype=torch.int64, device="cuda")
    ring = ReplayRing(256, (3, 12, 12), torch.bfloat16)
    fr = FrameRing(BatchedTron(k, 10, 10, layout="bits10", obs_dtype=torch.bfloat16, obs_enc="popup3"), 3, keep_terminal=True)

    def gather(rg, win, o, dt):
        return lib.replay_gather(C.byref(rg), idx.data_ptr(), k, o[0], o[1], dt, o[2], o[3], o[4], stream)

    def sample_gather(rg, win, o, dt):  # win = size
        return lib.replay_sample_gather(C.byref(rg), win, k, 0, 0, o[0], o[1], dt, o[2], o[3], o[4], None, stream)

    def frames_sample_gather(rg, win, o, dt):  # win = (first_tick, n_ticks)
        return lib.replay_frames_sample_gather(C.byref(rg), win[0], win[1], k, 0, 0, o[0], o[1], dt, o[2], o[3], o[4], None, stream)

    for call, rg, ring_ptrs, win, past in ((gather, ring.ring, ("state", "next_state"), None, []),
                                           (sample_gather, ring.ring, ("state", "next_state"), 256, [257, k - 1]),
                                           (frames_sample_gather, fr.fr, ("frames", "terminal"), (0, 2), [(0, 3), (-1, 2)])):
        name = call.__name__
        assert call(rg, win, good, abi.F32) == abi.OK, name
        torch.cuda.synchronize()
        for i in range(5):
            assert call(rg, win, good[:i] + [None] + good[i + 1:], abi.F32) == abi.ERR_INVALID, (name, i)
        assert call(rg, win, good, abi.I8) == abi.ERR_INVALID, name
        assert call(rg, win, [good[0] + 4] + good[1:], abi.F32) == abi.ERR_ALIGN, name
        assert call(rg, win, good[:1] + [good[1] + 8] + good[2:], abi.F32) == abi.ERR_ALIGN, name
        for field in ring_ptrs:
            bad = type(rg).from_buffer_copy(rg)
            setattr(bad, field, getattr(rg, field) + 4)
            assert call(bad, win, good, abi.F32) == abi.ERR_ALIGN, (name, field)
        for w in past:  # a window past the ring: size > capacity or k > size; n_ticks > S - 1 or first_tick < 0
            assert call(rg, w, good, abi.F32) == abi.ERR_INVALID, (name, w)


@pytest.mark.gpu
def test_debug_build_state_ring_reports_no_violation():
    """libtron_b200_debug.so: the slot, row, env and unit indices of the sample kernel are range-checked while the frame-ring
    equivalence runs on the 10x10 kernel and on a generic board"""
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import torch, test_gpu_state_ring as t\n"
            "from tron_b200 import abi, _lib\n"
            "t.run_equivalence(300, 10, 10, 'bits10', abi.BF16, 'popup3', torch.float32)\n"
            "t.run_equivalence(300, 7, 9, 'bits', abi.F32, 'popup3_const', torch.bfloat16, const_plane=0.3, slide_mode='temper')\n"
            "import ctypes as C\n"
            "n, f = C.c_uint64(), C.c_int32()\n"
            "_lib.check(_lib.load().tron_debug_violations(C.byref(n), C.byref(f)), 'tron_debug_violations')\n"
            "print('violations', n.value, 'first', f.value)\n") % (ROOT, os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, TRON_B200_DEBUG="1", PYTHONPATH=ROOT)
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900, cwd=d)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "violations 0 " in out.stdout, out.stdout[-2000:]


_SHIMS = ("tron", "config", "DQN", "DDQN", "Net")


@pytest.fixture
def loops():
    from tron_b200 import dropin
    for m in [k for k in sys.modules if k.split(".")[0] in _SHIMS]:
        del sys.modules[m]
    dropin.install()
    import DDQN
    import DQN
    yield DDQN, DQN
    for m in [k for k in sys.modules if k.split(".")[0] in _SHIMS]:
        del sys.modules[m]


@pytest.mark.gpu
def test_training_loops_replay_states(loops, monkeypatch):
    import tron_b200.replay as replay
    DDQN, DQN = loops
    rings = []

    class Spy(replay.StateRing):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            rings.append(self)
    monkeypatch.setattr(DDQN, "StateRing", Spy)
    monkeypatch.setattr(replay, "StateRing", Spy)
    tm = {}
    agent, env = DDQN.train(n_envs=1024, env_steps=48, replay="states", buffer_size=2048 * 100, timings=tm)
    assert len(rings) == 1 and rings[0].S == 100 and len(rings[0]) == 48 * 2048
    assert tm["learn_steps"] == 12 and np.isfinite(agent.totalloss) and agent.totalloss > 0
    assert env.stats_dict()["env_steps"] == 48 * 1024
    model, losses = DQN.train(n_envs=128, iterations=2, replay="states")
    assert len(rings) == 2 and rings[1].S == 40 and len(losses) == 2 and all(np.isfinite(l) for l in losses)


def test_replay_states_struct_layout_matches_header():
    """CPU: sizeof and field offsets of replay_states, compiled from the header with gcc, equal the ctypes mirror"""
    prog = r'''
    #include <stdio.h>
    #include <stddef.h>
    #include "tron_b200.h"
    int main(void) {
      printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(replay_states), offsetof(replay_states, struct_size), offsetof(replay_states, n_slots),
             offsetof(replay_states, slot_bytes), offsetof(replay_states, states), offsetof(replay_states, action), offsetof(replay_states, counter),
             offsetof(replay_states, slide_params));
      return 0; }'''
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "p.c"), "w").write(prog)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(d, "p"), os.path.join(d, "p.c")])
        v = list(map(int, subprocess.check_output([os.path.join(d, "p")]).decode().split()))
    R = abi.ReplayStates
    assert v == [C.sizeof(R), R.struct_size.offset, R.n_slots.offset, R.slot_bytes.offset, R.states.offset, R.action.offset, R.counter.offset,
                 R.slide_params.offset]
