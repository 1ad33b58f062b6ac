"""Observation buffers reused across ticks (tron_step_args.obs_prev): when `step` is handed the buffer it wrote last, the 10x10
bit-plane kernels store only the parts of each row that the tick changes.  Every output must stay bit-identical to the CPU oracle,
tick after tick, and every way the buffer or the env's state can change behind the env's back must fall back to full rows."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

from oracle import c_oracle as oc  # noqa: E402
from tron_b200 import abi  # noqa: E402
from tron_b200.batch_env import BatchedTron, GraphedStep  # noqa: E402

from _gpu import TORCH_DT, assert_same_state, assert_same_step, to_np  # noqa: E402

N = 4096 + 37  # a ragged last CTA


def pair(n=N, layout="bits10", dt=abi.BF16, enc=abi.ENC_LUT1, slide=abi.SLIDE_NONE, seed=0, **kw):
    g = BatchedTron(n, 10, 10, obs_dtype=TORCH_DT[dt], obs_enc=enc, slide_mode=slide, seed=seed, layout=layout, **kw)
    o = oc.OracleEnv(n, 10, 10, obs_dtype=dt, obs_enc=enc, slide_mode=slide, seed=seed, **kw)
    return g, o


def actions(rng, n=N):
    a = rng.integers(0, 4, size=(n, 2)).astype(np.uint8)
    a[rng.random(n) < 0.01, rng.integers(0, 2)] = 9  # invalid: the game is frozen this tick
    return a


def spawn_tape(rng, n=N):
    s = rng.integers(0, 10, size=(n, 4)).astype(np.int8)
    same = (s[:, 0] == s[:, 2]) & (s[:, 1] == s[:, 3])
    s[same, 2] = (s[same, 2] + 1) % 10
    return s


def check_step(g, o, buf, rng, what, act=None, slide=abi.SLIDE_NONE):
    act = actions(rng, g.N) if act is None else act
    st = rng.integers(0, 2, size=(g.N, 2)).astype(np.uint8) if slide == abi.SLIDE_TAPE else None
    res = g.step(torch.as_tensor(act), slide_tape=st, obs=buf)
    assert res.obs is buf
    assert_same_step(tuple(to_np(x) for x in res), o.step(act, slide_tape=st), what)


CASES = [
    ("bits10", abi.BF16, abi.ENC_LUT1, abi.SLIDE_NONE, {}),
    ("bits10", abi.F32, abi.ENC_POPUP3, abi.SLIDE_NONE, {}),
    ("bits10", abi.BF16, abi.ENC_POPUP3_CONST, abi.SLIDE_NONE, dict(const_plane=2.5)),
    ("bits10", abi.I8, abi.ENC_LUT1, abi.SLIDE_NONE, {}),
    ("bits10", abi.BF16, abi.ENC_LUT1, abi.SLIDE_NONE, dict(lut=(0, 0, 5, 5, 1, -1))),  # two tiles map to one value
    ("bits10", abi.F32, abi.ENC_POPUP3_CONST, abi.SLIDE_NONE, dict(const_plane=-1.0, auto_reset=False)),
    ("bits", abi.BF16, abi.ENC_LUT1, abi.SLIDE_TAPE, {}),
    ("bits", abi.F32, abi.ENC_POPUP3_CONST, abi.SLIDE_ICE, dict(slide_rate=0.3, const_plane=4.0)),
    ("bits", abi.BF16, abi.ENC_POPUP3, abi.SLIDE_TEMPER, {}),
    ("bits", abi.I8, abi.ENC_POPUP3, abi.SLIDE_ICE, dict(slide_rate=0.15)),
]


@pytest.mark.parametrize("layout,dt,enc,slide,kw", CASES, ids=["-".join(map(str, c[:4])) + ("-%d" % i) for i, c in enumerate(CASES)])
def test_reused_buffer_matches_oracle_every_tick(layout, dt, enc, slide, kw):
    rng = np.random.default_rng(7)
    g, o = pair(layout=layout, dt=dt, enc=enc, slide=slide, seed=3, **kw)
    buf = g.reset()
    assert np.array_equal(to_np(buf), o.reset())
    shape = tuple(buf.shape)
    for t in range(300):
        act = actions(rng)
        sp = spawn_tape(rng) if t % 3 == 0 else None
        st = rng.integers(0, 2, size=(N, 2)).astype(np.uint8) if slide == abi.SLIDE_TAPE else None
        what = "%s tick %d" % (layout, t)
        if t == 150:  # masked reset into the same buffer: full rows, then the delta path resumes
            mask = rng.integers(0, 2, size=N).astype(np.uint8)
            assert g.reset(mask=mask, obs=buf) is buf
            assert np.array_equal(to_np(buf), o.reset(mask=mask)), what
        if t % 7 == 0:  # terminal frames of the games that finish this tick (rows written in full, into their own buffer)
            gt = torch.full(shape, 3, dtype=TORCH_DT[dt], device="cuda")
            ot = to_np(torch.full(shape, 3, dtype=TORCH_DT[dt])).copy()
            res = g.step(torch.as_tensor(act), spawn=sp, slide_tape=st, obs=buf, obs_terminal=gt)
            assert_same_step(tuple(to_np(x) for x in res), o.step(act, spawn=sp, slide_tape=st, obs_terminal=ot), what)
            assert np.array_equal(to_np(gt), ot), what + " obs_terminal"
        else:
            res = g.step(torch.as_tensor(act), spawn=sp, slide_tape=st, obs=buf)
            assert_same_step(tuple(to_np(x) for x in res), o.step(act, spawn=sp, slide_tape=st), what)
    assert_same_state(_Exp(g), o)


class _Exp:
    def __init__(self, env):
        self.env = env

    def export(self):
        return {k: to_np(v) for k, v in self.env.export().items()}


def test_delta_path_is_taken():
    """A write the version counter cannot see (through .data) survives in the cells the tick leaves alone: proof that the kernel
    skipped them, and the documented limit of the fast path.  observe() repairs the buffer."""
    rng = np.random.default_rng(1)
    g, o = pair()
    buf = g.reset(); o.reset()
    check_step(g, o, buf, rng, "warm-up")
    buf.data.fill_(7.0)
    act = actions(rng)
    res = g.step(torch.as_tensor(act), obs=buf)
    want = o.step(act)
    assert not np.array_equal(to_np(res.obs), want[0])
    assert np.array_equal(to_np(g.observe(buf)), o.observe())
    check_step(g, o, buf, rng, "after observe")


def test_in_place_writes_between_steps():
    rng = np.random.default_rng(2)
    g, o = pair()
    buf = g.reset(); o.reset()
    for t in range(12):
        check_step(g, o, buf, rng, "tick %d" % t)
        if t % 3 == 0:
            buf.fill_(5.0)
        elif t % 3 == 1:
            buf[t * 7].zero_()
            buf[-1, 1].fill_(-2.0)


def test_two_envs_alternating_on_one_buffer():
    rng = np.random.default_rng(3)
    ga, oa = pair(seed=1)
    gb, ob = pair(seed=2)
    buf = ga.reset(); oa.reset()
    gb.reset(obs=buf); ob.reset()
    for t in range(10):
        check_step(ga, oa, buf, rng, "A tick %d" % t)
        check_step(gb, ob, buf, rng, "B tick %d" % t)
        if t >= 5:  # and twice in a row each
            check_step(gb, ob, buf, rng, "B again %d" % t)


def test_buffers_a_b_a():
    rng = np.random.default_rng(4)
    g, o = pair()
    a = g.reset(); o.reset()
    b = g.new_obs()
    for t in range(6):
        check_step(g, o, a, rng, "A %d" % t)
        check_step(g, o, b, rng, "B %d" % t)
        check_step(g, o, b, rng, "B again %d" % t)


def test_state_changes_between_steps():
    rng = np.random.default_rng(5)
    g, o = pair()
    buf = g.reset(); o.reset()
    g2, o2 = pair(seed=9)
    g2.reset(); o2.reset()
    for _ in range(5):
        check_step(g2, o2, g2.new_obs(), rng, "donor")
    check_step(g, o, buf, rng, "first")
    # step_many
    acts = rng.integers(0, 4, size=(3, N, 2)).astype(np.uint8)
    r = g.step_many(3, actions=torch.as_tensor(acts))
    assert_same_step(tuple(to_np(x) for x in r), o.step_many(3, actions=acts), "step_many")
    check_step(g, o, buf, rng, "after step_many")
    # import_
    ex = g2.export()
    g.import_(**ex)
    o.import_(**o2.export())
    check_step(g, o, buf, rng, "after import_")
    # bind_step with its own buffer, and with this one
    for obs in (None, buf):
        bs = g.bind_step(obs=obs)
        bs()
        w = o.step(None)
        assert np.array_equal(to_np(bs.obs), w[0]) and np.array_equal(to_np(bs.reward), w[1])
        check_step(g, o, buf, rng, "after bind_step")
    # load_state_dict
    sd = g2.state_dict()
    g.load_state_dict(sd)
    o.state[...] = o2.state
    o.counter = o2.counter
    check_step(g, o, buf, rng, "after load_state_dict")


def test_graphed_step_env():
    g, o = pair(seed=6)
    g.reset(); o.reset()
    gs = GraphedStep(g, policy="random")  # plays one tick while warming up
    w = o.step(None)
    for t in range(4):
        gs.replay()
        w = o.step(None)
        assert np.array_equal(to_np(gs.obs), w[0]), t
    r = g.step(obs=gs.obs)
    assert_same_step(tuple(to_np(x) for x in r), o.step(None), "step after graph replays")
