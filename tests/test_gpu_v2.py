"""ABI version 2 features against the oracle: Game.__init__'s temper draws on reset, terminal frames (obs_terminal), the
[degree, weight] side features, the one-launch sampler + gather, the frame-sharing replay ring, the pipelined host front end
and the range-checked debug build."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from oracle import c_oracle as oc  # noqa: E402
from tron_b200 import abi  # noqa: E402

from _gpu import TORCH_DT, GpuEnvNumpy, assert_same_state, assert_same_step, make_pair, to_np  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------ temper parameters are drawn by reset (Game.__init__, game.py:83,87)
@pytest.mark.parametrize("layout", ["tile8", "bits", "trail"])
def test_reset_draws_temper_parameters(layout):
    N = 4000
    enc = abi.ENC_NONE if layout == "trail" else abi.ENC_LUT1
    g, o = make_pair(N, 10, 10, layout=layout, obs_dtype=abi.I8, obs_enc=enc, seed=5, slide_mode=abi.SLIDE_TEMPER, auto_reset=False)
    g.reset(); o.reset()
    prm = g.env.slide_params.cpu().numpy()
    assert np.array_equal(prm, o.slide_params)
    assert prm[:, 0].min() >= -30 and prm[:, 0].max() <= 30 and prm[:, 1:3].min() >= 40 and prm[:, 1:3].max() <= 101
    assert len(np.unique(prm[:, 0])) > 30 and len(np.unique(prm[:, 1])) > 30
    assert np.array_equal(g.env.extra.cpu().numpy(), o.extra())
    # the very first episode after reset() slides (before: parameters were only drawn on auto-reset)
    slid = 0
    for t in range(6):
        assert_same_step(g.step(), o.step(), "tick %d" % t)
        slid += int((o.export()["tiles"] >= 5).sum())
    assert slid > 0
    # masked reset re-draws only the flagged games
    before = g.env.slide_params.cpu().numpy().copy()
    mask = (np.arange(N) % 2 == 0).astype(np.uint8)
    g.reset(mask=mask); o.reset(mask=mask)
    after = g.env.slide_params.cpu().numpy()
    assert np.array_equal(after, o.slide_params)
    assert np.array_equal(after[1::2], before[1::2]) and not np.array_equal(after[0::2], before[0::2])
    assert_same_state(g, o)


@pytest.mark.parametrize("layout", ["tile8", "bits"])
def test_extra_side_features_follow_the_observed_game(layout):
    """Game.get_multy (game.py:137-139): [degree, weight_p] of the game the observation shows, also across auto-resets"""
    N = 3000
    g, o = make_pair(N, 10, 10, layout=layout, obs_dtype=abi.I8, seed=8, slide_mode=abi.SLIDE_TEMPER)
    g.reset(); o.reset()
    for t in range(12):
        assert_same_step(g.step(), o.step(), "tick %d" % t)
        x = g.env.extra.cpu().numpy()
        assert np.array_equal(x, o.extra()), t
        prm = g.env.slide_params.cpu().numpy()
        assert np.array_equal(x[:, 0, 0], prm[:, 0]) and np.array_equal(x[:, 0, 1], prm[:, 1]) and np.array_equal(x[:, 1, 1], prm[:, 2])
    g.env.observe()
    assert np.array_equal(g.env.extra.cpu().numpy(), o.extra())


# ------------------------------------------------------------------ terminal frames
@pytest.mark.parametrize("layout,W,dt,enc", [("tile8", 10, abi.BF16, abi.ENC_LUT1), ("bits10", 10, abi.BF16, abi.ENC_POPUP3), ("bits", 10, abi.F32, abi.ENC_LUT1),
                                             ("bits", 7, abi.I8, abi.ENC_POPUP3_CONST), ("tile8", 20, abi.I8, abi.ENC_LUT1), ("tile8", 50, abi.BF16, abi.ENC_LUT1),
                                             ("trail", 10, abi.BF16, abi.ENC_POPUP3), ("trail", 20, abi.F32, abi.ENC_LUT1), ("trail", 46, abi.I8, abi.ENC_POPUP3_CONST),
                                             ("trail", 19, abi.I8, abi.ENC_LUT1), ("trail", 7, abi.BF16, abi.ENC_LUT1), ("trail", 33, abi.I8, abi.ENC_POPUP3)])
def test_obs_terminal_holds_the_last_frame_of_finished_games(layout, W, dt, enc):
    N = 1500 if W <= 20 else 200
    g, o = make_pair(N, W, W, layout=layout, obs_dtype=dt, obs_enc=enc, seed=13, const_plane=2.0)
    g.reset(); o.reset()
    shape = (N, 2, abi.enc_planes(enc), W + 2, W + 2)
    sentinel = 7
    for t in range(10):
        gt = torch.full(shape, sentinel, dtype=TORCH_DT[dt], device="cuda")
        ot = to_np(torch.full(shape, sentinel, dtype=TORCH_DT[dt])).copy()
        r = g.env.step(obs_terminal=gt)
        want = o.step(obs_terminal=ot)
        assert_same_step(tuple(to_np(x) for x in r), want, "tick %d" % t)
        got_t = to_np(gt)
        assert np.array_equal(got_t, ot), t
        done = want[2].astype(bool)
        assert done.any() and not done.all()
        assert (got_t[~done] == ot[~done]).all() and not np.array_equal(got_t[done], to_np(r.obs)[done])  # finished rows differ from the fresh game


@pytest.mark.parametrize("mode", [abi.SLIDE_ICE, abi.SLIDE_TEMPER])
def test_obs_terminal_trail_with_slide_tiles(mode):
    """a game that ends on a slide tick leaves an uncommitted body AND slide tile per player: both belong to its terminal frame"""
    N, W = 2000, 12
    g, o = make_pair(N, W, W, layout="trail", obs_dtype=abi.BF16, obs_enc=abi.ENC_POPUP3, seed=31, slide_mode=mode, slide_rate=0.6)
    g.reset(); o.reset()
    shape = (N, 2, 3, W + 2, W + 2)
    for t in range(12):
        gt = torch.full(shape, 7, dtype=torch.bfloat16, device="cuda")
        ot = to_np(torch.full(shape, 7, dtype=torch.bfloat16)).copy()
        r = g.env.step(obs_terminal=gt)
        assert_same_step(tuple(to_np(x) for x in r), o.step(obs_terminal=ot), "tick %d" % t)
        assert np.array_equal(to_np(gt), ot), t


def test_obs_terminal_is_refused_where_unsupported():
    from tron_b200 import _lib
    from tron_b200.batch_env import BatchedTron
    # the trail layout renders terminal frames with its bulk-store kernel, which keeps whole observation rows in shared memory
    assert not abi.trail_bulk_ok(126, 126, abi.ENC_POPUP3_CONST, abi.F32)
    env = BatchedTron(4, 126, 126, layout="trail", obs_dtype=torch.float32, obs_enc="popup3_const")  # 512 KB per game
    env.reset()
    with pytest.raises(_lib.TronError):
        env.step(obs_terminal=env.new_obs())


# ------------------------------------------------------------------ sampler fused with the gather
@pytest.mark.parametrize("dt,F", [(abi.BF16, 144), (abi.F32, 432), (abi.I8, 100)])
def test_sample_gather_one_launch_matches_oracle(dt, F):
    from tron_b200.replay import ReplayRing
    cap = 5000
    ring = ReplayRing(cap, (F,), TORCH_DT[dt], seed=5)
    oring = oc.OracleRing(cap, F, dt)
    rng = np.random.default_rng(6)
    for n in (3000, 4000):
        s = rng.integers(-10, 11, size=(n, F)); s2 = rng.integers(-10, 11, size=(n, F))
        a = rng.integers(0, 4, size=n).astype(np.uint8); r = rng.normal(size=n).astype(np.float32)
        d = rng.integers(0, 2, size=n).astype(np.uint8)
        ts, ts2 = torch.as_tensor(s).to(TORCH_DT[dt]), torch.as_tensor(s2).to(TORCH_DT[dt])
        ring.push(ts.cuda(), ts2.cuda(), torch.as_tensor(a), torch.as_tensor(r), torch.as_tensor(d))
        oring.push(to_np(ts), to_np(ts2), a, r, d)
    for k, counter in ((64, 3), (4096, 4), (cap, 5)):
        s, a, r, s2, d, idx = ring.sample(k, counter=counter, want_indices=True)
        want_idx = oc.sample_indices(len(oring), k, 5, counter)
        assert np.array_equal(idx.cpu().numpy(), want_idx) and len(set(want_idx.tolist())) == k
        want = oring.gather(want_idx, abi.F32)
        for gg, ww in zip((s, a, r, s2, d), want):
            assert np.array_equal(to_np(gg).reshape(ww.shape), ww)
    assert sorted(ring.sample_indices(cap, counter=9).cpu().numpy().tolist()) == list(range(cap))
    a = ring.sample(64, counter=11)
    b = ring.sample(64, counter=12)
    again = ring.sample(64, counter=11, out=b)  # same tensors, new content
    assert again[0].data_ptr() == b[0].data_ptr() and all(torch.equal(x, y) for x, y in zip(a, again))
    with pytest.raises(ValueError):
        ring.sample(32, out=b)


def test_sampler_is_uniform_over_sizes_that_are_not_powers_of_two():
    from tron_b200.replay import ReplayRing
    ring = ReplayRing(1000, (16,), torch.int8, seed=3)
    for size in (3, 40, 257, 1000):
        ring.cursor = size
        counts = np.zeros(size)
        k = max(1, size // 4)
        reps = 1200
        for c in range(reps):
            idx = ring.sample_indices(k, counter=c).cpu().numpy()
            assert len(set(idx.tolist())) == k and idx.min() >= 0 and idx.max() < size
            counts[idx] += 1
        exp = reps * k / size
        assert counts.min() > 0.6 * exp and counts.max() < 1.5 * exp, (size, counts.min(), counts.max(), exp)
        first = np.bincount(np.array([int(ring.sample_indices(1, counter=c)[0]) for c in range(300)]), minlength=size)
        assert first.max() < 300 * max(0.5, 8.0 / size)  # position 0 of the permutation is not stuck on one slot


# ------------------------------------------------------------------ frame-sharing replay ring
@pytest.mark.parametrize("layout,dt,enc,keep_terminal", [("bits10", abi.BF16, abi.ENC_POPUP3, True), ("tile8", abi.F32, abi.ENC_LUT1, True),
                                                         ("bits", abi.I8, abi.ENC_LUT1, False)])
def test_frame_ring_transitions_equal_the_explicit_ones(layout, dt, enc, keep_terminal):
    """every transition the frame ring hands out equals the (s, a, r, s', d) the DDQN loop would have stored explicitly
    (DDQN.py:264-308): s' of a finished game is its LAST frame, not the fresh game's first one."""
    from tron_b200.batch_env import BatchedTron
    from tron_b200.replay import FrameRing
    N, S, T = 600, 5, 13  # wraps the ring several times
    env = BatchedTron(N, 10, 10, layout=layout, obs_dtype=TORCH_DT[dt], obs_enc=enc, seed=4)
    o = oc.OracleEnv(N, 10, 10, obs_dtype=dt, obs_enc=enc, seed=4)
    ring = FrameRing(env, S, keep_terminal=keep_terminal, seed=9)
    obs = to_np(ring.begin())
    oobs = o.reset()
    assert np.array_equal(obs, oobs)
    P, C = abi.enc_planes(enc), 144
    explicit = {}  # (tick, row) -> (s, a, r, s2, d)
    rng = np.random.default_rng(2)
    for t in range(T):
        act = rng.integers(0, 4, size=(N, 2)).astype(np.uint8)
        term = oobs.copy()
        nobs, rew, done, winner, _ = o.step(act, obs_terminal=term)
        s2 = np.where(done.astype(bool)[:, None, None, None, None], term, nobs) if keep_terminal else nobs
        for row in range(2 * N):
            explicit[(t, row)] = (oobs.reshape(2 * N, -1)[row], act.reshape(-1)[row], rew.reshape(-1)[row], s2.reshape(2 * N, -1)[row], float(done[row // 2]))
        res = ring.step(actions=torch.as_tensor(act).cuda())
        assert np.array_equal(to_np(res.obs), nobs) and np.array_equal(to_np(ring.frames()), nobs)
        oobs = nobs
        n_ticks = min(t + 1, S - 1)
        assert len(ring) == n_ticks * 2 * N
        for k in (64, n_ticks * 2 * N):
            s, a, r, sn, d, idx = ring.sample(k, counter=t, want_indices=True)
            idx = idx.cpu().numpy()
            assert len(set(idx.tolist())) == k
            ticks = idx // (2 * N)
            assert ticks.min() >= t + 1 - n_ticks and ticks.max() <= t
            sf, snf = to_np(s).reshape(k, -1).astype(np.float32), to_np(sn).reshape(k, -1).astype(np.float32)
            for j in (range(k) if k == 64 else range(0, k, 97)):
                es, ea, er, es2, ed = explicit[(int(ticks[j]), int(idx[j] % (2 * N)))]
                assert np.array_equal(sf[j], oc.obs_to_float(es, dt)) and np.array_equal(snf[j], oc.obs_to_float(es2, dt)), (t, j)
                assert int(a[j, 0]) == ea and float(r[j, 0]) == er and float(d[j, 0]) == ed
    # same sample through the C oracle of the ring
    fr = ring
    want = oc.frames_sample_gather(to_np(fr.frames_t).reshape(S, 2 * N, P * C), None if fr.terminal_t is None else to_np(fr.terminal_t).reshape(S, 2 * N, P * C),
                                   to_np(fr.action_t).reshape(S, 2 * N), to_np(fr.reward_t).reshape(S, 2 * N), to_np(fr.done_t), dt, T - (S - 1), S - 1, 500, 9, 77)
    got = ring.sample(500, counter=77, want_indices=True)
    for gg, ww in zip(got, want):
        assert np.array_equal(to_np(gg).reshape(ww.shape), ww)


# ------------------------------------------------------------------ host front end: pipelined steps
@pytest.mark.parametrize("layout,W,dt", [("bits10", 10, abi.I8), ("tile8", 10, abi.BF16), ("bits", 9, abi.I8), ("trail", 20, abi.I8)])
def test_host_env_pipelined_steps_match_oracle(layout, W, dt):
    from tron_b200.batch_env import HostTron
    N = 9000
    h = HostTron(N, W, W, obs_dtype=dt, n_chunks=6, seed=31, layout=layout, double_buffer=True)
    o = oc.OracleEnv(N, W, W, obs_dtype=dt, seed=31)
    assert np.array_equal(h.reset(), o.reset())
    rng = np.random.default_rng(9)
    acts = [rng.integers(0, 4, size=(N, 2)).astype(np.uint8) for _ in range(9)]
    want = [o.step(a) for a in acts]
    h.step_begin(acts[0])
    for t in range(len(acts)):
        if t + 1 < len(acts):
            h.step_begin(acts[t + 1])  # two steps in flight
        obs, rew, done, winner = h.step_wait()
        wo, wr, wd, ww, _ = want[t]
        assert np.array_equal(obs, wo) and np.array_equal(rew, wr) and np.array_equal(done, wd) and np.array_equal(winner, ww), t
    h.close()


def test_host_env_guards():
    from tron_b200 import _lib
    from tron_b200.batch_env import HostTron, host_copy_bandwidth
    h = HostTron(100, 10, 10)
    assert h.obs.dtype == np.int8  # the reference returns integer observations
    with pytest.raises(_lib.TronError):
        h.step(np.zeros((100, 2), np.uint8))  # step before reset
    h.reset()
    h.step_begin(np.zeros((100, 2), np.uint8)); h.step_begin(np.zeros((100, 2), np.uint8))
    with pytest.raises(_lib.TronError):
        h.step_begin(np.zeros((100, 2), np.uint8))  # a third step in flight
    h.step_wait(); h.step_wait()
    with pytest.raises(_lib.TronError):
        h.step_wait()
    h.close()
    for direction in ("h2d", "d2h"):
        assert host_copy_bandwidth(64 << 20, direction, 2) > 1.0


# ------------------------------------------------------------------ range-checked debug build
def test_debug_build_fuzz_reports_no_violation():
    """libtron_b200_debug.so (-DTRON_DEBUG): every cell index, bit index, trail-list position, ring slot and env ownership is
    range-checked on the device while the randomised differential fuzz runs (stands in for compute-sanitizer on this pool)."""
    env = dict(os.environ, TRON_B200_DEBUG="1", PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_gpu.py"), "--seeds", "3", "--debug-checks"], env=env, capture_output=True, text=True, timeout=1500)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "violations 0" in out.stdout, out.stdout[-2000:]


# ------------------------------------------------------------------ the benchmarked configuration at full size
def test_four_million_envs_bits10_properties():
    """bench.py's workload (2^22 games, bit-plane layout): exact agreement with the oracle on the first and last 2048 env ids, and
    size-independent invariants over the whole batch."""
    from tron_b200.batch_env import BatchedTron
    N, K = 1 << 22, 2048
    env = BatchedTron(N, 10, 10, layout="bits10", obs_dtype=torch.bfloat16, seed=0)
    lo = oc.OracleEnv(K, 10, 10, obs_dtype=abi.BF16, seed=0, env_id_base=0)
    hi = oc.OracleEnv(K, 10, 10, obs_dtype=abi.BF16, seed=0, env_id_base=N - K)
    obs = env.reset()
    assert np.array_equal(to_np(obs[:K]), lo.reset()) and np.array_equal(to_np(obs[N - K:]), hi.reset())
    for t in range(12):
        r = env.step(obs=obs)
        wl, wh = lo.step(), hi.step()
        for i, name in enumerate(("obs", "reward", "done", "winner", "ep_len")):
            assert np.array_equal(to_np(r[i][:K]), wl[i]) and np.array_equal(to_np(r[i][N - K:]), wh[i]), (t, name)
        o16 = r.obs.view(torch.int16)
        # every observation holds exactly 44 wall cells per player plane; a game shows its own head (10) at most once per player
        walls = (o16 == torch.tensor(-1.0, dtype=torch.bfloat16).view(torch.int16)).sum(dim=(2, 3, 4))
        assert int(walls.min()) >= 42 and int(walls.max()) <= 44  # a head that crashed into the border overwrites up to two wall cells
        own = (o16 == torch.tensor(10.0, dtype=torch.bfloat16).view(torch.int16)).sum(dim=(2, 3, 4))
        assert int(own.max()) <= 1
        assert bool(((r.winner == 0) | (r.done == 1)).all())
    st = env.stats_dict()
    assert st["env_steps"] == 12 * N and st["episodes"] == st["p1_wins"] + st["p2_wins"] + st["draws"]
    ex = env.export()
    assert np.array_equal(ex["tiles"][:K].cpu().numpy(), lo.export()["tiles"]) and np.array_equal(ex["tiles"][N - K:].cpu().numpy(), hi.export()["tiles"])


# ------------------------------------------------------------------ importing a grid given as tiles only
@pytest.mark.parametrize("layout,W", [("tile8", 10), ("bits10", 10), ("bits", 10), ("bits", 7), ("trail", 10), ("trail", 20)])
def test_import_of_tiles_only_recovers_the_heads(layout, W):
    """the compact layouts keep heads outside the cell data; a grid imported without a head array takes them from its head tiles
    (incl. heads that crashed into the border and the shared-cell head-on state)"""
    N = 3000
    o = oc.OracleEnv(N, W, W, obs_dtype=abi.I8, seed=21, auto_reset=False)
    o.reset()
    for t in range(5):
        o.step()
    ex = o.export()
    assert ex["done"].any() and not ex["done"].all()
    g = GpuEnvNumpy(N, W, W, obs_dtype=abi.I8, seed=99, auto_reset=False, layout=layout)
    g.reset()
    g.import_(tiles=ex["tiles"])
    assert np.array_equal(g.observe(), o.observe())
    back = g.export()
    assert np.array_equal(back["tiles"], ex["tiles"])
    one_head = (ex["tiles"] == 2).sum((1, 2)) == 1  # both heads visible (not the shared-cell case)
    assert np.array_equal(back["heads"][one_head], ex["heads"][one_head])


def test_bound_step_equals_step():
    """bind_step (arguments packed once) is the same tick as step(): external actions, in-kernel policy, device-side counter"""
    from tron_b200.batch_env import BatchedTron
    N = 3000
    for layout in ("bits10", "tile8"):
        a = BatchedTron(N, 10, 10, obs_dtype=torch.bfloat16, seed=6, layout=layout)
        b = BatchedTron(N, 10, 10, obs_dtype=torch.bfloat16, seed=6, layout=layout)
        a.reset(); b.reset()
        act = torch.zeros((N, 2), dtype=torch.uint8, device="cuda")
        bound = b.bind_step(actions=act)
        g = torch.Generator(device="cpu").manual_seed(1)
        for t in range(12):
            act.copy_(torch.randint(0, 4, (N, 2), generator=g, dtype=torch.uint8))
            ra = a.step(act)
            rb = bound()
            assert torch.equal(ra.obs.view(torch.int16), rb.obs.view(torch.int16)) and torch.equal(ra.reward, rb.reward) and torch.equal(ra.done, rb.done)
        pol = b.bind_step()
        for t in range(6):
            ra = a.step(); rb = pol()
            assert torch.equal(ra.obs.view(torch.int16), rb.obs.view(torch.int16)) and torch.equal(ra.winner, rb.winner)
        assert a.stats_dict() == b.stats_dict()


def test_tuning_options_do_not_change_results():
    """CTA caps (shared-memory padding) and the store-schedule switch are performance knobs only: identical outputs"""
    import _geometry as geo
    from tron_b200 import _lib
    from tron_b200.batch_env import BatchedTron
    L = _lib.load()
    sms = geo.sm_count()
    N = 1 << 18  # 128 games per CTA and 2,048 CTAs on 148 SMs: more than 8 CTAs per SM, so the caps pad shared memory
    codes = {torch.bfloat16: abi.BF16, torch.float32: abi.F32, torch.int8: abi.I8}
    encs = {"lut1": abi.ENC_LUT1, "popup3": abi.ENC_POPUP3}

    def run(layout, enc, dtype, slide=None):
        env = BatchedTron(N, 10, 10, obs_dtype=dtype, obs_enc=enc, seed=12, layout=layout, slide_mode=slide)
        env.reset()
        for _ in range(3):
            r = env.step()
        return r.obs.clone().view(torch.uint8), r.reward.clone(), env.export()["tiles"].clone()

    def want_geometry(layout, enc, dtype, slide, opt):
        if layout == "tile8":
            return geo.tile_geometry(N, 10, 10, codes[dtype], encs[enc], sms, cap_opt=opt[1] if opt[0] == abi.OPT_TILE_CTAS_PER_SM else 0)
        return geo.bits_geometry(N, 10, 10, layout, codes[dtype], encs[enc], False, sms, cap_opt=opt[1] if opt[0] == abi.OPT_BITS_CTAS_PER_SM else 0)
    cases = [("bits10", "lut1", torch.bfloat16, None), ("bits10", "popup3", torch.int8, None), ("bits", "lut1", torch.float32, "temper"), ("tile8", "popup3", torch.bfloat16, None)]
    opts = ((abi.OPT_BITS_CTAS_PER_SM, 2), (abi.OPT_BITS_CTAS_PER_SM, 32), (abi.OPT_TILE_CTAS_PER_SM, 3), (abi.OPT_ENCODE_VARIANT, 8))
    # the geometry guard: every case under every setting launches with 128 games per CTA, 2,048 CTAs and the padding its cap gives
    probes = [(c, o) for o in [(0, 0)] + list(opts) for c in cases]
    launched = geo.step_launches_in_fresh_process([dict(env=dict(n_envs=N, width=10, height=10, obs_dtype=str(c[2]).split(".")[1], obs_enc=c[1], seed=12,
                                                                 layout=c[0], slide_mode=c[3]), options=[o] if o[0] else []) for c, o in probes])
    for (c, o), got in zip(probes, launched):
        want = want_geometry(*c, o)
        assert want.G == 128 and want.grid > 8 * sms
        geo.assert_geometry(got, want, (c, o))
    try:
        base = [run(*c) for c in cases]
        for opt, val in opts:
            _lib.check(L.tron_set_option(opt, val))
            for c, want in zip(cases, base):
                got = run(*c)
                assert all(torch.equal(g, w) for g, w in zip(got, want)), (opt, val, c)
            _lib.check(L.tron_set_option(opt, 0))
    finally:
        for opt in (abi.OPT_BITS_CTAS_PER_SM, abi.OPT_TILE_CTAS_PER_SM, abi.OPT_ENCODE_VARIANT):
            L.tron_set_option(opt, 0)
