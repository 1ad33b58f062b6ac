"""The fused kernels against the C oracle at the launch geometries bench.py, DDQN.train and DQN.train run.

Every fused kernel derives its launch geometry from the batch size: games per CTA, how many of a CTA's warps own games, whether
shared-memory padding caps the resident CTAs per SM, and on the trail layout how many groups of games each warp renders.  The other
parity tests use batches small enough that all of these collapse to their smallest case (16 games per CTA: only warp 0 owns games;
one group per warp; no padding).  Here each case takes its batch size from the mirror of the launch rules in _geometry.py, asserts
on the first call that the kernel really launched with that geometry, and then compares the whole batch with
oracle.c_oracle.OracleEnv after every tick: obs, reward, done, winner, ep_len, terminal frames, then the exported state and the
statistics.  Batches are ragged (the last CTA is partial), some ticks carry spawn tapes and ~1 % of the actions are invalid (the
game is frozen for that tick)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from oracle import c_oracle as oc  # noqa: E402
from tron_b200 import abi  # noqa: E402

import _geometry as geo  # noqa: E402
from _gpu import TORCH_DT  # noqa: E402

# bit patterns are compared, so -0.0 != 0.0 and NaN payloads count
_INT_VIEW = {1: (np.int8, torch.int8), 2: (np.int16, torch.int16), 4: (np.int32, torch.int32)}
_SENTINEL = {abi.BF16: np.uint16(0x4040), abi.F32: np.float32(3.0), abi.I8: np.int8(3)}  # 3.0 in every obs dtype


@pytest.fixture(scope="module")
def sms():
    return geo.sm_count()


def assert_same(got, want, what):
    """device tensor == numpy array, bit for bit, compared on the device (the batches here hold up to ~0.7 GB of observations)"""
    want = np.ascontiguousarray(want)
    assert got.element_size() == want.itemsize and tuple(got.shape) == want.shape, (what, tuple(got.shape), want.shape, got.dtype, want.dtype)
    npv, tv = _INT_VIEW[want.itemsize]
    g = got.contiguous().view(tv)
    w = torch.from_numpy(want.view(npv)).to(got.device)
    if not torch.equal(g, w):
        bad = (g != w).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError("%s differs at %d places, first %s: got %d want %d" % (what, bad.shape[0], i, int(g[i]), int(w[i])))


def assert_same_step(res, want, what):
    for name, g, w in zip(("obs", "reward", "done", "winner", "ep_len"), res, want):
        assert_same(g, w, "%s %s" % (what, name))


def actions(rng, n):
    a = rng.integers(0, 4, size=(n, 2)).astype(np.uint8)
    a[rng.random(n) < 0.01, rng.integers(0, 2)] = 9  # invalid: the game is frozen this tick
    return a


def spawn_tape(rng, n, W, H):
    s = rng.integers(0, min(W, H), size=(n, 4)).astype(np.int8)
    same = (s[:, 0] == s[:, 2]) & (s[:, 1] == s[:, 3])
    s[same, 2] = (s[same, 2] + 1) % min(W, H)
    return s


def run_case(tmp_path, N, W, H, layout, dt, enc, want, ticks=8, term_every=3, reset_at=5, seed=3, **kw):
    """One oracle and one BatchedTron per entry of `want` ({"fresh" | "reused": Geometry}) play the same tapes.  "fresh" steps
    into a new buffer every tick (full rows); "reused" hands back the buffer it wrote last (tron_step_args.obs_prev: the delta
    store where it applies).  The first step of each env runs under the geometry guard.  obs_terminal every `term_every` ticks
    (None: never), a masked reset into the same buffers after tick `reset_at`."""
    from tron_b200.batch_env import BatchedTron
    kw.setdefault("slide_rate", 0.0)
    o = oc.OracleEnv(N, W, H, obs_dtype=dt, obs_enc=enc, seed=seed, **kw)
    envs = {m: BatchedTron(N, W, H, layout=layout, obs_dtype=TORCH_DT[dt], obs_enc=enc, seed=seed, **kw) for m in want}
    wobs = o.reset()
    bufs = {}
    for m, env in envs.items():
        bufs[m] = env.reset()
        assert_same(bufs[m], wobs, "%s reset" % m)
    shape = (N, 2, abi.enc_planes(enc), W + 2, H + 2)
    rng = np.random.default_rng(seed)
    for t in range(ticks):
        act = actions(rng, N)
        sp = spawn_tape(rng, N, W, H) if t % 3 == 1 else None
        term = term_every is not None and t % term_every == term_every - 1
        ot = np.full(shape, _SENTINEL[dt]) if term else None
        wres = o.step(act, spawn=sp, obs_terminal=ot)
        act_d = torch.as_tensor(act).cuda()
        sp_d = None if sp is None else torch.as_tensor(sp).cuda()
        for m, env in envs.items():
            gt = torch.full(shape, 3, dtype=TORCH_DT[dt], device="cuda") if term else None
            call = lambda: env.step(act_d, spawn=sp_d, obs=bufs[m] if m == "reused" else None, obs_terminal=gt)  # noqa: E731
            what = "%s tick %d" % (m, t)
            res = geo.guarded(call, tmp_path, want[m], what) if t == 0 else call()
            if m == "reused":
                assert res.obs is bufs[m]
            assert_same_step(res, wres, what)
            if term:
                assert_same(gt, ot, what + " obs_terminal")
        if term:
            assert wres[2].any(), "tick %d: no game finished, the terminal frames went unchecked" % t
        if t == reset_at:
            mask = rng.integers(0, 2, size=N).astype(np.uint8)
            wobs = o.reset(mask=mask)
            for m, env in envs.items():
                r = env.reset(mask=torch.as_tensor(mask).cuda(), obs=bufs[m] if m == "reused" else None)
                assert_same(r, wobs, "%s masked reset" % m)
    wex = o.export()
    for m, env in envs.items():
        ex = env.export()
        for k in wex:
            assert_same(ex[k], wex[k], "%s export %s" % (m, k))
        st = env.stats.view(abi.STATS_SLOTS, abi.STATS_FIELDS).sum(0).cpu().numpy().astype(np.uint64)
        assert np.array_equal(st, o.stats), (m, st, o.stats)
    assert int(o.stats[abi.STAT_BAD_ACTION]) > 0 and int(o.stats[abi.STAT_EPISODES]) > 0
    return envs, o


# ------------------------------------------------------------------ bits10: the headline kernel
BITS10_ENCS = [
    (abi.BF16, abi.ENC_LUT1, {}),
    (abi.BF16, abi.ENC_POPUP3, {}),
    (abi.BF16, abi.ENC_POPUP3_CONST, dict(const_plane=2.5)),
    (abi.F32, abi.ENC_LUT1, {}),
    (abi.F32, abi.ENC_POPUP3_CONST, dict(const_plane=-1.5)),
    (abi.I8, abi.ENC_LUT1, {}),
    (abi.I8, abi.ENC_POPUP3, {}),
]
DT_NAME = {abi.BF16: "bf16", abi.F32: "f32", abi.I8: "i8"}
ENC_NAME = {abi.ENC_LUT1: "lut1", abi.ENC_POPUP3: "popup3", abi.ENC_POPUP3_CONST: "popup3_const"}


@pytest.mark.parametrize("dt,enc,kw", BITS10_ENCS, ids=["%s-%s" % (DT_NAME[c[0]], ENC_NAME[c[1]]) for c in BITS10_ENCS])
@pytest.mark.parametrize("G", [32, 64, 96, 128], ids=["G32", "G64", "G96", "G128-capped"])
def test_bits10_matches_oracle_at_launch_geometry(tmp_path, sms, G, dt, enc, kw):
    """warps 1, 2 and 3 of a CTA own games from G = 64, 96 and 128, so the delta store's CTA scan adds earlier warps' counts;
    G = 128 with more than 8 CTAs per SM pads shared memory (to 4 CTAs per SM for full rows, 5 for the delta store, 5 or none
    for int8 planes)"""
    N = geo.n_for_small_grid(G, sms, ragged=20, capped=G == 128)
    want = {m: geo.bits_geometry(N, 10, 10, "bits10", dt, enc, prev=m == "reused", sms=sms) for m in ("fresh", "reused")}
    assert all(w.G == G for w in want.values())
    run_case(tmp_path, N, 10, 10, "bits10", dt, enc, want, **kw)


@pytest.mark.parametrize("slide,dt,enc,kw", [(abi.SLIDE_ICE, abi.BF16, abi.ENC_POPUP3, dict(slide_rate=0.3)),
                                              (abi.SLIDE_TEMPER, abi.F32, abi.ENC_LUT1, {})], ids=["ice-bf16-popup3", "temper-f32-lut1"])
def test_bits_slide_plane_delta_matches_oracle_capped(tmp_path, sms, slide, dt, enc, kw):
    """the 10x10 slide-plane instantiation of the delta store at G = 128, padded to 5 CTAs per SM"""
    N = geo.n_for_small_grid(128, sms, ragged=33, capped=True)
    want = {"reused": geo.bits_geometry(N, 10, 10, "bits", dt, enc, prev=True, sms=sms)}
    assert want["reused"].args[-1] == "true" and want["reused"].grid > 8 * sms
    run_case(tmp_path, N, 10, 10, "bits", dt, enc, want, slide_mode=slide, **kw)


GENERIC = [
    # (W, H, obs dtype, encoding, extra kwargs): the largest G each board reaches, with more than 8 CTAs per SM
    (7, 7, abi.I8, abi.ENC_LUT1, {}),                                                   # G 128, 81 cells: element encode
    (11, 11, abi.F32, abi.ENC_LUT1, dict(slide_mode=abi.SLIDE_ICE, slide_rate=0.3)),    # G 96, 169 cells
    (8, 16, abi.BF16, abi.ENC_POPUP3, {}),                                              # G 96, 180 cells: encode_tile_linear4
    (6, 11, abi.I8, abi.ENC_POPUP3_CONST, dict(const_plane=2.0, slide_mode=abi.SLIDE_TEMPER)),  # G 128, 104 cells: linear4
]


@pytest.mark.parametrize("W,H,dt,enc,kw", GENERIC, ids=["%dx%d-%s-%s" % (c[0], c[1], DT_NAME[c[2]], ENC_NAME[c[3]]) for c in GENERIC])
def test_bits_generic_boards_match_oracle_at_largest_G(tmp_path, sms, W, H, dt, enc, kw):
    N = geo.n_for_bits_capped(W, H, sms, ragged=7)
    want = {m: geo.bits_geometry(N, W, H, "bits", dt, enc, prev=m == "reused", sms=sms) for m in ("fresh", "reused")}
    assert want["fresh"].G == geo.bits_staging_G(W, H) >= 96
    run_case(tmp_path, N, W, H, "bits", dt, enc, want, **kw)


# ------------------------------------------------------------------ tile8: the int8-grid kernels
def test_tile8_10x10_matches_oracle_capped(tmp_path, sms):
    N = geo.n_for_small_grid(128, sms, ragged=45, capped=True)
    want = geo.tile_geometry(N, 10, 10, abi.BF16, abi.ENC_POPUP3, sms)
    assert want.G == 128 and want.smem == geo.smem_for_ctas_per_sm(want.smem, 5) > 20 * 1024  # padded to 5 CTAs per SM
    envs, o = run_case(tmp_path, N, 10, 10, "tile8", abi.BF16, abi.ENC_POPUP3, {"fresh": want}, ticks=6)
    # four ticks in one launch, every tick's observation stored
    rng = np.random.default_rng(11)
    acts = np.stack([actions(rng, N) for _ in range(4)])
    r = geo.guarded(lambda: envs["fresh"].step_many(4, actions=torch.as_tensor(acts).cuda(), obs_every_tick=True), tmp_path, want, "step_many")
    assert_same_step(r, o.step_many(4, actions=acts, obs_every_tick=True), "step_many")


def test_tile8_64x64_matches_oracle_capped(tmp_path, sms):
    W = 64
    G = geo.tile_G(1, W, W, sms)  # 4 games per CTA on a 64x64 board (step_generic.cu:8-16)
    N = geo._ragged(G * 8 * sms + 1, G)
    want = geo.tile_geometry(N, W, W, abi.BF16, abi.ENC_LUT1, sms)
    assert want.G == 4 and want.grid > 8 * sms and want.smem == geo.smem_for_ctas_per_sm(want.smem, 6) > 30 * 1024
    run_case(tmp_path, N, W, W, "tile8", abi.BF16, abi.ENC_LUT1, {"fresh": want}, ticks=6)


# ------------------------------------------------------------------ trail: the bulk-store kernel with two or more groups per warp
TRAIL = [
    # (W, H, obs dtype, encoding, groups per warp, ragged games, extra kwargs)
    (12, 12, abi.BF16, abi.ENC_LUT1, 2, 53, {}),                                            # grp 16, 4 warps: a partial second group
    (16, 16, abi.BF16, abi.ENC_POPUP3, 2, 22, dict(slide_mode=abi.SLIDE_ICE, slide_rate=0.3)),  # grp 4
    (64, 64, abi.F32, abi.ENC_POPUP3_CONST, 2, 1, dict(const_plane=-2.0)),                    # grp 1, one warp per CTA
    (21, 21, abi.I8, abi.ENC_POPUP3, 2, 11, {}),                                              # odd rows (3,174 B): grp 8
]


@pytest.mark.parametrize("W,H,dt,enc,groups,ragged,kw", TRAIL, ids=["%dx%d-%s-%s" % (c[0], c[1], DT_NAME[c[2]], ENC_NAME[c[3]]) for c in TRAIL])
def test_trail_bulk_store_matches_oracle_with_groups_per_warp(tmp_path, sms, W, H, dt, enc, groups, ragged, kw):
    """the `s0 > 0` iterations of both render loops of step_trail_obs_bulk_kernel: the terminal-frame ballot shifted to a later
    group, the lane of sub-row j of group s0 and the destination of that group"""
    N = geo.n_for_trail_groups(W, H, dt, enc, sms, groups, ragged)
    want, grp, nwarp, gpw = geo.trail_bulk_geometry(N, W, H, dt, enc, sms)
    assert gpw >= 2 * grp and N % want.G != 0
    run_case(tmp_path, N, W, H, "trail", dt, enc, {"fresh": want}, ticks=7, term_every=2, **kw)


def test_trail_element_store_kernel_matches_oracle_with_games_per_warp(tmp_path, sms):
    """the element-store kernel (TRON_OPT_ENCODE_VARIANT 32) with more than one game per warp"""
    from tron_b200 import _lib
    W, dt, enc = 12, abi.BF16, abi.ENC_LUT1
    N = 2 * 6 * 4 * sms * 4 + 5  # step_trail.cu:662: gpw = N / (6 waves * 4 CTAs * SMs * 4 warps) = 2
    want, gpw = geo.trail_fallback_geometry(N, W, W, dt, enc, sms)
    assert gpw == 2 and N % want.G != 0
    L = _lib.load()
    try:
        _lib.check(L.tron_set_option(abi.OPT_ENCODE_VARIANT, 32))
        run_case(tmp_path, N, W, W, "trail", dt, enc, {"fresh": want}, ticks=7, term_every=None)
    finally:
        L.tron_set_option(abi.OPT_ENCODE_VARIANT, 0)


# ------------------------------------------------------------------ state ring: 32 transitions per CTA
@pytest.mark.parametrize("layout,W,H,dt,enc,out_dtype,kw", [("bits10", 10, 10, abi.BF16, "popup3", torch.float32, {}),
                                                           ("bits", 7, 9, abi.F32, "lut1", torch.bfloat16, dict(slide_mode="ice", slide_rate=0.3))],
                         ids=["bits10-bf16-popup3", "bits-7x9-f32-lut1-ice"])
def test_state_ring_at_32_transitions_per_cta(tmp_path, sms, layout, W, H, dt, enc, out_dtype, kw):
    """StateRing samples of k >= 2 * 31 * SMs + 1 (32 transitions per CTA, a partial last CTA) equal a twin FrameRing's bit for bit;
    on bits10 they also equal the oracle's explicit transitions"""
    from test_gpu_state_ring import _bits, _check_against, _env, _tape
    from tron_b200.replay import FrameRing, StateRing
    k = geo._ragged(2 * sms * 31 + 1, 32)
    N, S, T = 2502, 4, 6  # even, so that every frame-ring slot (792 B per game on 7x9 f32) starts 16-byte aligned
    ea, eb = _env(N, W, H, layout, dt, enc, **kw), _env(N, W, H, layout, dt, enc, **kw)
    fr, sr = FrameRing(ea, S + 1, keep_terminal=True, seed=9), StateRing(eb, S, seed=9)
    fr.begin()
    obs = sr.begin(obs=eb.new_obs())
    o = None
    if layout == "bits10":
        o = oc.OracleEnv(N, W, H, obs_dtype=dt, obs_enc={"popup3": abi.ENC_POPUP3}[enc], seed=4)
        oobs = o.reset()
        assert np.array_equal(_bits(obs), oobs.view(np.uint8))
    explicit = {}
    rng = np.random.default_rng(2)
    sampled = 0
    for t in range(T):
        a = _tape(rng, N)
        if o is not None:
            act = a.cpu().numpy()
            term = oobs.copy()
            nobs, rew, done, _, _ = o.step(act, obs_terminal=term)
            s2 = np.where(done.astype(bool)[:, None, None, None, None], term, nobs)
            explicit[t] = (oc.obs_to_float(oobs, dt).reshape(2 * N, -1), act.reshape(-1), rew.reshape(-1), oc.obs_to_float(s2, dt).reshape(2 * N, -1),
                           done.astype(np.float32))
            explicit.pop(t - S, None)
            oobs = nobs
        fr.step(actions=a)
        sr.step(actions=a, obs=obs)
        if len(sr) < k:
            continue
        for kk in (k, len(sr)):
            want_geo = geo.replay_states_geometry(kk, W, H, layout, sms)
            assert want_geo.G == 32 and (kk != k or kk % 32 != 0)
            want = fr.sample(kk, out_dtype, counter=t, want_indices=True)
            got = geo.guarded(lambda: sr.sample(kk, out_dtype, counter=t, want_indices=True), tmp_path, want_geo, "k %d" % kk)
            for name, w, g in zip(("s", "a", "r", "s2", "d", "idx"), want, got):
                assert w.dtype == g.dtype and w.shape == g.shape, name
                assert np.array_equal(_bits(w), _bits(g)), (t, kk, name)
            if o is not None:
                assert _check_against(explicit, got, N) == kk
            sampled += 1
    assert sampled >= 6
