"""BatchedTron -- the vectorised batch API: N independent 2-player TRON games stepped in lockstep on one GPU.

Semantics follow the reference one game at a time (tron/game.py:149-277 Game.next_frame/step,
tron/map.py:67-84 state_for_player, tron/util.py:11-37 pop_up, tron/util.py:46-84 make_game,
ACKTR.py:285-317 auto-reset).  All compute happens in libtron_b200.so through the C ABI; torch only
owns the device memory and supplies the stream.
"""
import ctypes as C
import weakref

import torch

from . import _abi as abi
from . import _lib

_TORCH_OF = {abi.BF16: torch.bfloat16, abi.F32: torch.float32, abi.I8: torch.int8}
_CODE_OF = {torch.bfloat16: abi.BF16, torch.float32: abi.F32, torch.int8: abi.I8, torch.uint8: abi.U8,
            torch.int32: abi.I32, torch.int64: abi.I64}
_ENC_OF = {"none": abi.ENC_NONE, "lut1": abi.ENC_LUT1, "popup3": abi.ENC_POPUP3, "popup3_const": abi.ENC_POPUP3_CONST}
_LAYOUT_OF = {"tile8": abi.LAYOUT_TILE8, "bits10": abi.LAYOUT_BITS10, "trail": abi.LAYOUT_TRAIL, "bits": abi.LAYOUT_BITS}


def auto_layout(width, height, obs_enc, slide_mode, obs_dtype=torch.bfloat16):
    """fastest state layout that can represent a configuration (all layouts are bit-identical through the API)"""
    enc_none = obs_enc in ("none", abi.ENC_NONE)
    no_slide = slide_mode in (None, abi.SLIDE_NONE)
    if width == 10 and height == 10 and no_slide:
        return "bits10"
    if width == 10 and height == 10:
        return "bits"   # config.py's board with a slide mode (GAME_MODE="temper"): three bit planes
    cells = (width + 2) * (height + 2)
    if enc_none:
        return "trail" if cells >= 1024 else "tile8"
    # fused observations on boards from 12x12 up: the trail lists with bulk-stored template rows beat the int8 grid (no grid
    # traffic at all; profiles/r2_trail_obs.jsonl, r2_small_boards_trail.jsonl) wherever that kernel applies
    enc = _ENC_OF[obs_enc] if isinstance(obs_enc, str) else int(obs_enc)
    dt = _CODE_OF[obs_dtype] if isinstance(obs_dtype, torch.dtype) else int(obs_dtype)
    if width * height >= 144 and width <= 126 and height <= 126 and abi.trail_bulk_ok(width, height, enc, dt):
        return "trail"
    return "tile8"
_SLIDE_OF = {None: abi.SLIDE_NONE, "tape": abi.SLIDE_TAPE, "ice": abi.SLIDE_ICE, "temper": abi.SLIDE_TEMPER}


def _ptr(t):
    return None if t is None else t.data_ptr()


class _OnDevice:
    """`with _OnDevice(dev):` -- like torch.cuda.device(dev) but free when `dev` already is the current device (the common case;
    the torch context manager costs ~4 us per call, more than a small tick kernel)."""
    __slots__ = ("dev", "ctx")

    def __init__(self, dev):
        self.dev, self.ctx = dev, None

    def __enter__(self):
        if torch.cuda.current_device() != self.dev.index:
            self.ctx = torch.cuda.device(self.dev)
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
            self.ctx = None


class StepResult(tuple):
    """(obs, reward, done, winner, ep_len) with attribute access."""
    __slots__ = ()
    obs = property(lambda s: s[0])
    reward = property(lambda s: s[1])
    done = property(lambda s: s[2])
    winner = property(lambda s: s[3])
    ep_len = property(lambda s: s[4])


class BatchedTron:
    """N games of width x height on `device`.

    obs layout: [N, 2, P, width+2, height+2]; obs[:, p] is player p+1's NCHW view (zero-copy).
    reward: name in abi.REWARD_POLICIES or a 5-tuple (step_base, step_per_tick, win, lose, draw).
    layout: "auto" (default: the fastest one that fits), "tile8" (int8 grid), "bits10" (32-byte bit planes, 10x10 without slide
    modes), "bits" (48-byte bit planes, any board with W*H <= 128, every mode) or "trail" (trail lists, made for pure ticks on large grids).
    game_params: keep the per-game parameters Game.__init__ draws for every game (weight x2, degree; tron/game.py:83,87) in
    `self.slide_params` ([N,4] int8 {degree, weight1, weight2, 0}) and the [degree, weight] side features of the games the latest
    observation shows (Game.get_multy, tron/game.py:137-139) in `self.extra` ([N,2,2] f32: per player {degree, weight_p}).
    Default: only with slide_mode="temper" (which needs them for the slip rate).
    """

    def __init__(self, n_envs, width=10, height=10, device="cuda", obs_dtype=torch.bfloat16, obs_enc="lut1", lut=None,
                 const_plane=0.0, reward="ddqn", auto_reset=True, seed=0, env_id_base=0, slide_mode=None,
                 slide_rate=0.15, collect_stats=True, layout="auto", spawn_mode="uniform",
                 policy="uniform", policy_epsilon=0.0, game_params=None):
        _lib.require_cuda()
        self.lib = _lib.load()
        if layout == "auto":
            layout = auto_layout(width, height, obs_enc, slide_mode, obs_dtype)
        self.layout = _LAYOUT_OF[layout] if isinstance(layout, str) else int(layout)
        self.spawn_mode = {"uniform": abi.SPAWN_UNIFORM, "fair": abi.SPAWN_FAIR}[spawn_mode] if isinstance(spawn_mode, str) else int(spawn_mode)
        self.policy = {"uniform": abi.POLICY_UNIFORM, "free_eps": abi.POLICY_FREE_EPS}[policy] if isinstance(policy, str) else int(policy)
        self.policy_epsilon = float(policy_epsilon)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.TronError("BatchedTron needs a CUDA device; there is no CPU fallback")
        if self.device.index is None:  # "cuda" -> "cuda:<current>", so device comparisons with tensors are exact
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.N, self.W, self.H = int(n_envs), int(width), int(height)
        self.C = abi.cells_per_env(width, height)
        self.obs_enc = _ENC_OF[obs_enc] if isinstance(obs_enc, str) else int(obs_enc)
        self.P = abi.enc_planes(self.obs_enc)
        self.obs_dtype = obs_dtype if isinstance(obs_dtype, int) else _CODE_OF[obs_dtype]
        self.lut = tuple(lut) if lut is not None else (0,) * 6
        self.const_plane = float(const_plane)
        self.reward_table = abi.Reward(*(abi.REWARD_POLICIES[reward] if isinstance(reward, str) else reward))
        self.auto_reset = bool(auto_reset)
        self.seed, self.env_id_base = int(seed), int(env_id_base)
        self.slide_mode = _SLIDE_OF[slide_mode] if (slide_mode is None or isinstance(slide_mode, str)) else int(slide_mode)
        self.slide_rate = float(slide_rate)
        self._tmpl = self._tmpl_key = None
        self.counter = 0
        self.counter_dev = None  # device u64; set by use_device_counter() so captured CUDA graphs advance the RNG between replays
        self._obs_last = None  # (weakref, _version) of the obs tensor that holds the current state's observation (see step)
        nbytes = C.c_size_t()
        _lib.check(self.lib.tron_state_bytes(self.N, self.W, self.H, self.layout, C.byref(nbytes)), "tron_state_bytes")
        with _OnDevice(self.device):
            self.state = torch.zeros(nbytes.value, dtype=torch.uint8, device=self.device)
            self.stats = torch.zeros(abi.STATS_SLOTS * abi.STATS_FIELDS, dtype=torch.int64, device=self.device) if collect_stats else None
            if game_params is None:
                game_params = self.slide_mode == abi.SLIDE_TEMPER
            if self.slide_mode == abi.SLIDE_TEMPER and not game_params:
                raise ValueError("slide_mode='temper' needs game_params")
            self.slide_params = torch.zeros((self.N, 4), dtype=torch.int8, device=self.device) if game_params else None
            self.extra = torch.zeros((self.N, 2, 2), dtype=torch.float32, device=self.device) if self.slide_params is not None else None

    # ------------------------------------------------------------------ buffers
    def new_obs(self, ticks=None):
        shape = (self.N, 2, self.P, self.W + 2, self.H + 2)
        if ticks is not None:
            shape = (ticks,) + shape
        return torch.empty(shape, dtype=_TORCH_OF[self.obs_dtype], device=self.device)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def use_device_counter(self):
        """Keep the tick counter in device memory: every call then reads it on the GPU and bumps it with tron_advance_counter,
        so a sequence of calls captured in a torch.cuda.CUDAGraph draws fresh random numbers on every replay."""
        if self.counter_dev is None:
            self.counter_dev = torch.full((1,), self.counter, dtype=torch.int64, device=self.device)
            self.counter = 0
        return self.counter_dev

    def _take_counter(self, counter, n=1):
        """-> (counter value for the call, device pointer or None, advance-after-call)"""
        if counter is not None:
            return counter, None, 0
        if self.counter_dev is not None:
            return 0, self.counter_dev.data_ptr(), n
        c, self.counter = self.counter, self.counter + n
        return c, None, 0

    def _advance(self, n):
        if n:
            _lib.check(self.lib.tron_advance_counter(self.counter_dev.data_ptr(), n, self._stream()), "tron_advance_counter")

    def _args(self, **kw):
        """argument block of one call: a copy of the per-environment template with the per-call fields filled in"""
        key = (self.policy, self.policy_epsilon, self.auto_reset, self.slide_rate, self.seed, self.env_id_base)
        if self._tmpl is None or self._tmpl_key != key:
            self._tmpl = abi.new_step_args(n_envs=self.N, width=self.W, height=self.H, layout=self.layout, state=self.state.data_ptr(),
                                           obs_dtype=self.obs_dtype, obs_enc=self.obs_enc, lut=self.lut, const_plane=self.const_plane,
                                           reward_table=self.reward_table, auto_reset=int(self.auto_reset), seed=self.seed,
                                           env_id_base=self.env_id_base, slide_mode=self.slide_mode, slide_rate=self.slide_rate, spawn_mode=self.spawn_mode,
                                           policy=self.policy, policy_epsilon=self.policy_epsilon,
                                           slide_params=_ptr(self.slide_params), stats=_ptr(self.stats), extra=_ptr(self.extra))
            self._tmpl_key = key
        a = abi.StepArgs.from_buffer_copy(self._tmpl)
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    def _obs_written(self, obs):
        """`obs` now holds the observation of the current state.  Its version is bumped so that a later write by anyone, another
        env included, is visible as a version change.  Graph capture and the device counter replay state changes without Python
        seeing them, so nothing is remembered then."""
        self._obs_last = None
        if obs.is_inference() or self.counter_dev is not None or torch.cuda.is_current_stream_capturing():
            return
        torch.autograd.graph.increment_version(obs)
        self._obs_last = (weakref.ref(obs), obs._version)

    def _obs_is_prev(self, obs):
        last = self._obs_last
        return (last is not None and last[0]() is obs and obs._version == last[1] and self.counter_dev is None
                and not torch.cuda.is_current_stream_capturing())

    def _dev(self, t, dtype, shape=None, name="tensor"):
        """move/cast a user input to a contiguous device tensor and check its shape (the kernels trust sizes)"""
        if t is None:
            return None
        if not torch.is_tensor(t):
            t = torch.as_tensor(t)
        t = t.to(device=self.device, dtype=dtype).contiguous()
        if shape is not None and tuple(t.shape) != tuple(shape):
            raise ValueError("%s must have shape %s, got %s" % (name, tuple(shape), tuple(t.shape)))
        return t

    def _out(self, t, shape, dtype, name):
        """validate a caller-provided output buffer"""
        if t is None:
            return None
        if (not torch.is_tensor(t) or t.device != self.device or t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous()):
            raise ValueError("%s must be a contiguous %s tensor of shape %s on %s" % (name, dtype, tuple(shape), self.device))
        return t

    # ------------------------------------------------------------------ API
    def reset(self, spawn=None, mask=None, obs=None, counter=None):
        """Fresh games (Game.__init__, incl. its weight/degree draws in temper mode).  spawn: [N,4] int8 {x1,y1,x2,y2} or None
        (RNG, make_game rule).  mask: [N] uint8, reset only the flagged games.  Returns the initial observation (or None for
        obs_enc='none')."""
        if counter is None:
            if self.counter_dev is not None:
                counter = int(self.counter_dev.item())
                self.counter_dev += 1
            else:
                counter, self.counter = self.counter, self.counter + 1
        sp = self._dev(spawn, torch.int8, (self.N, 4), "spawn")
        mk = self._dev(mask, torch.uint8, (self.N,), "mask")
        a = self._args(spawn=_ptr(sp), counter=counter, obs_enc=abi.ENC_NONE)
        self._obs_last = None
        with _OnDevice(self.device):
            _lib.check(self.lib.tron_reset_ex(C.byref(a), _ptr(mk), self._stream()), "tron_reset_ex")
        return self.observe(obs) if self.P else None

    def observe(self, obs=None):
        if not self.P:
            raise ValueError("this environment was created with obs_enc='none'")
        if obs is None:
            obs = self.new_obs()
        self._out(obs, (self.N, 2, self.P, self.W + 2, self.H + 2), _TORCH_OF[self.obs_dtype], "obs")
        a = self._args(obs=obs.data_ptr())
        with _OnDevice(self.device):
            _lib.check(self.lib.tron_observe(C.byref(a), self._stream()), "tron_observe")
        self._obs_written(obs)
        return obs

    def step(self, actions=None, spawn=None, slide_tape=None, obs=None, reward=None, done=None, winner=None, ep_len=None,
             counter=None, want_ep_len=True, obs_terminal=None):
        """One tick of every game.  actions: [N,2] uint8/int32/int64 tensor (P1,P2) or None (uniform random policy).
        Output tensors may be passed in to avoid allocation.  obs_terminal: tensor like obs; the rows of games that finished in this
        tick (and were auto-reset) receive the finished game's last frame (DDQN.py:270-308 next_state), other rows are untouched.
        -> StepResult(obs, reward, done, winner, ep_len)

        Passing the same `obs` tensor every tick is the fast path: when it is the very tensor this env last wrote (by step,
        observe or reset), unchanged since by torch's version counter, and the env's state has not changed in between, the
        kernel is told that the buffer holds the previous observation (tron_step_args.obs_prev) and may store only the parts of
        each row that this tick changes.  Writes that bypass the version counter (through `.data`, a raw pointer or another
        library) are not seen: after one, pass the buffer through observe() first, which always writes full rows."""
        counter, cdev, adv = self._take_counter(counter)
        N, dev = self.N, self.device
        if actions is not None:
            if not torch.is_tensor(actions):
                actions = torch.as_tensor(actions)
            if actions.device != dev or not actions.is_contiguous() or actions.dtype not in (torch.uint8, torch.int32, torch.int64):
                # other dtypes go through int64 so that out-of-range values stay out of range (and are counted as bad actions)
                actions = actions.to(device=dev, dtype=actions.dtype if actions.dtype in (torch.uint8, torch.int32, torch.int64) else torch.int64).contiguous()
            if tuple(actions.shape) != (N, 2):
                raise ValueError("actions must have shape (%d, 2), got %s" % (N, tuple(actions.shape)))
        sp = self._dev(spawn, torch.int8, (N, 4), "spawn")
        sl = self._dev(slide_tape, torch.uint8, (N, 2), "slide_tape")
        if self.slide_mode == abi.SLIDE_TAPE and sl is None:
            raise ValueError("slide_mode='tape' needs a slide_tape for every step")
        self._out(obs, (N, 2, self.P, self.W + 2, self.H + 2), _TORCH_OF.get(self.obs_dtype), "obs") if self.P else None
        self._out(reward, (N, 2), torch.float32, "reward"); self._out(done, (N,), torch.uint8, "done")
        self._out(winner, (N,), torch.uint8, "winner"); self._out(ep_len, (N,), torch.int32, "ep_len")
        if obs_terminal is not None:
            self._out(obs_terminal, (N, 2, self.P, self.W + 2, self.H + 2), _TORCH_OF.get(self.obs_dtype), "obs_terminal")
        prev = obs is not None and self._obs_is_prev(obs)
        if obs is None and self.P:
            obs = self.new_obs()
        if reward is None:
            reward = torch.empty((N, 2), dtype=torch.float32, device=dev)
        if done is None:
            done = torch.empty(N, dtype=torch.uint8, device=dev)
        if winner is None:
            winner = torch.empty(N, dtype=torch.uint8, device=dev)
        if ep_len is None and want_ep_len:
            ep_len = torch.empty(N, dtype=torch.int32, device=dev)
        a = self._args(actions=_ptr(actions), action_dtype=0 if actions is None else _CODE_OF[actions.dtype], obs=_ptr(obs),
                       reward=reward.data_ptr(), done=done.data_ptr(), winner=winner.data_ptr(), ep_len_out=_ptr(ep_len),
                       spawn=_ptr(sp), slide_tape=_ptr(sl), counter=counter, counter_dev=cdev, obs_terminal=_ptr(obs_terminal),
                       obs_prev=int(prev))
        self._obs_last = None
        with _OnDevice(dev):
            _lib.check(self.lib.tron_step(C.byref(a), self._stream()), "tron_step")
            self._advance(adv)
        if obs is not None:
            self._obs_written(obs)
        return StepResult((obs, reward, done, winner, ep_len))

    def bind_step(self, actions=None, obs=None, reward=None, done=None, winner=None, ep_len=None, obs_terminal=None):
        """Pre-bound tick for small batches, where Python overhead (not the 3-5 us kernel) sets the pace: validates and packs the
        argument block ONCE for fixed buffers; each call of the returned object then only bumps the counter and makes the one C
        call.  Buffers default to freshly allocated ones and are exposed as attributes (.obs .reward .done .winner .ep_len)."""
        return BoundStep(self, actions, obs, reward, done, winner, ep_len, obs_terminal)

    def step_many(self, n_ticks, actions=None, spawn=None, obs_every_tick=True, counter=None):
        """n_ticks ticks in one launch.  actions [T,N,2] or None (RNG), spawn [T,N,4] or None (RNG)."""
        counter, cdev, adv = self._take_counter(counter, int(n_ticks))
        T, N, dev = int(n_ticks), self.N, self.device
        act = None
        if actions is not None:
            act = actions if torch.is_tensor(actions) else torch.as_tensor(actions)
            dt = act.dtype if act.dtype in (torch.uint8, torch.int32, torch.int64) else torch.int64
            act = act.to(device=dev, dtype=dt).contiguous()
            if tuple(act.shape) != (T, N, 2):
                raise ValueError("actions must have shape (%d, %d, 2), got %s" % (T, N, tuple(act.shape)))
        sp = self._dev(spawn, torch.int8, (T, N, 4), "spawn")
        if self.slide_mode == abi.SLIDE_TAPE:
            raise ValueError("step_many does not take a slide tape; use step() or slide_mode 'ice'/'temper'")
        obs = (self.new_obs(T) if obs_every_tick else self.new_obs()) if self.P else None
        reward = torch.empty((T, N, 2), dtype=torch.float32, device=dev)
        done = torch.empty((T, N), dtype=torch.uint8, device=dev)
        winner = torch.empty((T, N), dtype=torch.uint8, device=dev)
        ep_len = torch.empty((T, N), dtype=torch.int32, device=dev)
        self._obs_last = None
        a = self._args(actions=_ptr(act), action_dtype=0 if act is None else _CODE_OF[act.dtype], obs=_ptr(obs),
                       reward=reward.data_ptr(), done=done.data_ptr(), winner=winner.data_ptr(), ep_len_out=ep_len.data_ptr(),
                       spawn=_ptr(sp), counter=counter, counter_dev=cdev, n_ticks=T, obs_every_tick=int(obs_every_tick))
        with _OnDevice(dev):
            _lib.check(self.lib.tron_step_many(C.byref(a), self._stream()), "tron_step_many")
            self._advance(adv)
        return StepResult((obs, reward, done, winner, ep_len))

    def export(self):
        """Tile.value grids + per-player state as torch tensors (for history / shims / tests)."""
        N, dev = self.N, self.device
        out = dict(tiles=torch.empty((N, self.W + 2, self.H + 2), dtype=torch.int8, device=dev),
                   heads=torch.empty((N, 4), dtype=torch.int8, device=dev), alive=torch.empty((N, 2), dtype=torch.uint8, device=dev),
                   done=torch.empty(N, dtype=torch.uint8, device=dev), winner=torch.empty(N, dtype=torch.uint8, device=dev),
                   ep_len=torch.empty(N, dtype=torch.int32, device=dev))
        with _OnDevice(dev):
            _lib.check(self.lib.tron_export_grid(self.state.data_ptr(), N, self.W, self.H, self.layout, out["tiles"].data_ptr(),
                                                 out["heads"].data_ptr(), out["alive"].data_ptr(), out["done"].data_ptr(),
                                                 out["winner"].data_ptr(), out["ep_len"].data_ptr(), self._stream()), "tron_export_grid")
        return out

    def import_(self, tiles=None, heads=None, alive=None, done=None, winner=None, ep_len=None):
        N = self.N
        t = self._dev(tiles, torch.int8, (N, self.W + 2, self.H + 2), "tiles"); h = self._dev(heads, torch.int8, (N, 4), "heads")
        al = self._dev(alive, torch.uint8, (N, 2), "alive"); d = self._dev(done, torch.uint8, (N,), "done")
        w = self._dev(winner, torch.uint8, (N,), "winner"); k = self._dev(ep_len, torch.int32, (N,), "ep_len")
        self._obs_last = None
        with _OnDevice(self.device):
            _lib.check(self.lib.tron_import_grid(self.state.data_ptr(), self.N, self.W, self.H, self.layout, _ptr(t), _ptr(h),
                                                 _ptr(al), _ptr(d), _ptr(w), _ptr(k), self._stream()), "tron_import_grid")

    def random_actions(self, counter=None, out=None):
        """counter=None with use_device_counter(): the draw of the *next* step() (same counter, not advanced)."""
        if out is None:
            out = torch.empty((self.N, 2), dtype=torch.uint8, device=self.device)
        cdev = None
        if counter is None:
            counter, cdev = (0, self.counter_dev.data_ptr()) if self.counter_dev is not None else (self.counter, None)
        with _OnDevice(self.device):
            _lib.check(self.lib.tron_random_actions(out.data_ptr(), self.N, self.seed, counter, cdev, self.env_id_base, self._stream()),
                       "tron_random_actions")
        return out

    def select_actions(self, q, epsilon, counter=None, out=None):
        """epsilon-greedy over q [N,2,4] or [2N,4] (float32/bfloat16) -> uint8 [N,2] (DDQN.py:90-110).
        counter=None: the counter of the next step() (host value, or the device counter after use_device_counter())."""
        if q.device != self.device or q.dtype not in (torch.float32, torch.bfloat16) or q.dim() < 1 or q.shape[-1] != 4:
            raise ValueError("q must be a float32/bfloat16 tensor [..., 4] on %s" % self.device)
        q2 = q.reshape(-1, 4).contiguous()
        if out is None:
            out = torch.empty(q2.shape[0], dtype=torch.uint8, device=self.device)
        elif out.numel() != q2.shape[0] or out.dtype != torch.uint8 or out.device != self.device or not out.is_contiguous():
            raise ValueError("out must be a contiguous uint8 tensor with one element per q row")
        cdev = None
        if counter is None:
            counter, cdev = (0, self.counter_dev.data_ptr()) if self.counter_dev is not None else (self.counter, None)
        with _OnDevice(self.device):
            _lib.check(self.lib.tron_select_actions(q2.data_ptr(), _CODE_OF[q2.dtype], q2.shape[0], float(epsilon), out.data_ptr(),
                                                    self.seed, counter, cdev, 2 * self.env_id_base, self._stream()), "tron_select_actions")
        return out.view(-1, 2) if out.numel() == 2 * self.N else out

    def minimax_actions(self, player, tie_mode=1, counter=None, out=None, want_values=False, want_ties=False):
        """The move (0..3) the reference's MinimaxPlayer(2, voronoi) would make for `player` (1|2) in every game
        (tron/minimax.py:296-310).  tie_mode 0 = first best move, 1 = uniform among the best (Philox).
        want_values: also the [N,4] root values; want_ties: also the [N,4] depth-1 tie counts (see tron_minimax_actions)."""
        tiles = self.state if self.layout == abi.LAYOUT_TILE8 else self.export()["tiles"].contiguous()
        if out is None:
            out = torch.empty(self.N, dtype=torch.uint8, device=self.device)
        vals = torch.empty((self.N, 4), dtype=torch.int32, device=self.device) if want_values else None
        ties = torch.empty((self.N, 4), dtype=torch.int32, device=self.device) if want_ties else None
        cdev = None
        if counter is None:
            counter, cdev = (0, self.counter_dev.data_ptr()) if self.counter_dev is not None else (self.counter, None)
        with _OnDevice(self.device):
            _lib.check(self.lib.tron_minimax_actions(tiles.data_ptr(), self.N, self.W, self.H, int(player), int(tie_mode), self.seed, counter, cdev,
                                                     self.env_id_base, out.data_ptr(), _ptr(vals), _ptr(ties), self._stream()), "tron_minimax_actions")
        if want_values or want_ties:
            return (out,) + ((vals,) if want_values else ()) + ((ties,) if want_ties else ())
        return out

    def state_dict(self):
        """Snapshot for checkpoint / resume (the reference only saves network weights; env state here is a few tensors)."""
        return dict(geometry=(self.N, self.W, self.H, self.layout), state=self.state.clone(),
                    counter=int(self.counter_dev.item()) if self.counter_dev is not None else self.counter,
                    stats=None if self.stats is None else self.stats.clone(),
                    slide_params=None if self.slide_params is None else self.slide_params.clone())

    def load_state_dict(self, sd):
        if tuple(sd["geometry"]) != (self.N, self.W, self.H, self.layout):
            raise ValueError("snapshot geometry %s does not match this environment %s" % (tuple(sd["geometry"]), (self.N, self.W, self.H, self.layout)))
        self._obs_last = None
        self.state.copy_(sd["state"])
        if self.counter_dev is not None:
            self.counter_dev.fill_(int(sd["counter"]))
        else:
            self.counter = int(sd["counter"])
        if self.stats is not None and sd.get("stats") is not None:
            self.stats.copy_(sd["stats"])
        if self.slide_params is not None and sd.get("slide_params") is not None:
            self.slide_params.copy_(sd["slide_params"])

    def stats_dict(self):
        """Summed on-device counters (episodes, wins, draws, ticks...).  Synchronises."""
        if self.stats is None:
            return {}
        s = self.stats.view(abi.STATS_SLOTS, abi.STATS_FIELDS).sum(0).tolist()
        return dict(episodes=s[abi.STAT_EPISODES], p1_wins=s[abi.STAT_P1_WINS], p2_wins=s[abi.STAT_P2_WINS], draws=s[abi.STAT_DRAWS],
                    ep_ticks=s[abi.STAT_EP_TICKS], bad_action=s[abi.STAT_BAD_ACTION], env_steps=s[abi.STAT_ENV_STEPS])


class BoundStep:
    """see BatchedTron.bind_step"""

    def __init__(self, env, actions, obs, reward, done, winner, ep_len, obs_terminal):
        N, dev = env.N, env.device
        if env.slide_mode == abi.SLIDE_TAPE:
            raise ValueError("bind_step does not take a slide tape; use step()")
        if actions is not None and (not torch.is_tensor(actions) or actions.device != dev or tuple(actions.shape) != (N, 2) or
                                    actions.dtype not in (torch.uint8, torch.int32, torch.int64) or not actions.is_contiguous()):
            raise ValueError("actions must be a contiguous uint8/int32/int64 tensor of shape (%d, 2) on %s" % (N, dev))
        shape = (N, 2, env.P, env.W + 2, env.H + 2)
        self.env, self.actions = env, actions
        self.obs = (env._out(obs, shape, _TORCH_OF[env.obs_dtype], "obs") if obs is not None else env.new_obs()) if env.P else None
        self.reward = env._out(reward, (N, 2), torch.float32, "reward") if reward is not None else torch.empty((N, 2), dtype=torch.float32, device=dev)
        self.done = env._out(done, (N,), torch.uint8, "done") if done is not None else torch.empty(N, dtype=torch.uint8, device=dev)
        self.winner = env._out(winner, (N,), torch.uint8, "winner") if winner is not None else torch.empty(N, dtype=torch.uint8, device=dev)
        self.ep_len = env._out(ep_len, (N,), torch.int32, "ep_len")
        self.obs_terminal = env._out(obs_terminal, shape, _TORCH_OF.get(env.obs_dtype), "obs_terminal") if obs_terminal is not None else None
        self._args = env._args(actions=_ptr(actions), action_dtype=0 if actions is None else _CODE_OF[actions.dtype], obs=_ptr(self.obs),
                               reward=self.reward.data_ptr(), done=self.done.data_ptr(), winner=self.winner.data_ptr(), ep_len_out=_ptr(self.ep_len),
                               obs_terminal=_ptr(self.obs_terminal), counter_dev=None if env.counter_dev is None else env.counter_dev.data_ptr())
        self._ref = C.byref(self._args)
        self._fn = env.lib.tron_step
        self._dev_counter = env.counter_dev is not None

    def __call__(self):
        env = self.env
        env._obs_last = None
        if not self._dev_counter:
            self._args.counter = env.counter
            env.counter += 1
        with _OnDevice(env.device):
            rc = self._fn(self._ref, torch.cuda.current_stream(env.device).cuda_stream)
            if rc:
                _lib.check(rc, "tron_step")
            if self._dev_counter:
                env._advance(1)
        return self


class HostTron:
    """Host-buffer front end (tron_host_env_*): numpy in, numpy out.  Observations default to int8 (the reference's Game.step
    returns integer arrays, tron/map.py:83-84); bf16 / f32 are available for callers that feed a net directly.

    step() blocks until the outputs have landed.  step_begin() / step_wait() pipeline consecutive steps (two in flight at most):
    the outputs of step t land in the buffer set t % 2 (self.obs2[t % 2] ...), and the tick kernels of step t+1 run while step t
    is still draining over PCIe."""

    def __init__(self, n_envs, width=10, height=10, obs_dtype=abi.I8, obs_enc=abi.ENC_LUT1, lut=None, const_plane=0.0,
                 reward="ddqn", auto_reset=True, seed=0, env_id_base=0, n_chunks=8, layout="auto", double_buffer=False):
        import numpy as np
        _lib.require_cuda()
        self.np = np
        self.lib = _lib.load()
        self.N, self.W, self.H = n_envs, width, height
        self.P, self.obs_dtype = abi.enc_planes(obs_enc), obs_dtype
        if layout == "auto":
            layout = auto_layout(width, height, obs_enc, None)
            if layout == "trail":
                layout = "tile8"
        proto = abi.new_step_args(n_envs=n_envs, width=width, height=height, obs_dtype=obs_dtype, obs_enc=obs_enc,
                                  layout=_LAYOUT_OF[layout] if isinstance(layout, str) else int(layout),
                                  lut=tuple(lut) if lut is not None else (0,) * 6, const_plane=const_plane,
                                  reward_table=abi.REWARD_POLICIES[reward] if isinstance(reward, str) else reward,
                                  auto_reset=int(auto_reset), seed=seed, env_id_base=env_id_base)
        self.handle = C.c_void_p()
        _lib.check(self.lib.tron_host_env_create(C.byref(self.handle), C.byref(proto), n_chunks), "tron_host_env_create")
        self._pinned = []
        npdt = {abi.BF16: np.uint16, abi.F32: np.float32, abi.I8: np.int8}[obs_dtype]
        nb = 2 if double_buffer else 1
        self.obs2 = [self.pinned((n_envs, 2, self.P, width + 2, height + 2), npdt) if self.P else None for _ in range(nb)]
        self.actions2 = [self.pinned((n_envs, 2), np.uint8) for _ in range(nb)]
        self.reward2 = [self.pinned((n_envs, 2), np.float32) for _ in range(nb)]
        self.done2 = [self.pinned((n_envs,), np.uint8) for _ in range(nb)]
        self.winner2 = [self.pinned((n_envs,), np.uint8) for _ in range(nb)]
        self.obs, self.actions, self.reward, self.done, self.winner = self.obs2[0], self.actions2[0], self.reward2[0], self.done2[0], self.winner2[0]
        self._begun = self._waited = 0

    def pinned(self, shape, dtype):
        """pinned host array, pages on the NUMA node of the current CUDA device (tron_host_alloc)"""
        np = self.np
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        _lib.check(self.lib.tron_host_alloc(C.byref(p), nbytes), "tron_host_alloc")
        self._pinned.append(p)
        buf = (C.c_uint8 * nbytes).from_address(p.value)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def reset(self, spawn=None):
        sp = None if spawn is None else self.np.ascontiguousarray(spawn, self.np.int8)
        _lib.check(self.lib.tron_host_env_reset(self.handle, None if sp is None else sp.ctypes.data, None if self.obs is None else self.obs.ctypes.data),
                   "tron_host_env_reset")
        self._begun = self._waited = 0
        return self.obs

    def _call(self, fn, name, b, actions, spawn):
        if actions is not None:
            self.actions2[b][...] = actions
        sp = None if spawn is None else self.np.ascontiguousarray(spawn, self.np.int8)
        self._spawn_keepalive = sp
        _lib.check(fn(self.handle, self.actions2[b].ctypes.data, None if sp is None else sp.ctypes.data,
                      None if self.obs2[b] is None else self.obs2[b].ctypes.data, self.reward2[b].ctypes.data,
                      self.done2[b].ctypes.data, self.winner2[b].ctypes.data), name)

    def step(self, actions=None, spawn=None):
        self._call(self.lib.tron_host_env_step, "tron_host_env_step", 0, actions, spawn)
        return self.obs, self.reward, self.done, self.winner

    def step_begin(self, actions=None, spawn=None):
        """enqueue one step and return; its outputs belong to the library until the matching step_wait()"""
        b = self._begun % len(self.obs2)
        self._call(self.lib.tron_host_env_step_begin, "tron_host_env_step_begin", b, actions, spawn)
        self._begun += 1
        return b

    def step_wait(self):
        """block until the oldest outstanding step has landed -> (obs, reward, done, winner) of that step"""
        _lib.check(self.lib.tron_host_env_step_wait(self.handle), "tron_host_env_step_wait")
        b = self._waited % len(self.obs2)
        self._waited += 1
        return self.obs2[b], self.reward2[b], self.done2[b], self.winner2[b]

    def state_ptr(self):
        return self.lib.tron_host_env_state(self.handle)

    def close(self):
        if self.handle:
            self.lib.tron_host_env_destroy(self.handle)
            self.handle = None
        self.obs = self.actions = self.reward = self.done = self.winner = None
        self.obs2 = self.actions2 = self.reward2 = self.done2 = self.winner2 = []
        for p in self._pinned:
            self.lib.tron_host_free(p)
        self._pinned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def host_copy_bandwidth(nbytes=1 << 30, direction="d2h", repeats=3):
    """measured PCIe ceiling of the current device: GB/s of back-to-back cudaMemcpyAsync between NUMA-local pinned memory and HBM"""
    out = C.c_double()
    _lib.check(_lib.load().tron_host_copy_bandwidth(int(nbytes), 0 if direction == "h2d" else 1, int(repeats), C.byref(out)), "tron_host_copy_bandwidth")
    return out.value


class GraphedStep:
    """One env tick captured as a CUDA graph (static buffers), for batch sizes where launch + Python overhead dominate.

        gs = GraphedStep(env, policy="random")      # or policy="external": fill gs.actions before each replay
        for _ in range(T): gs.replay()               # gs.obs / gs.reward / gs.done / gs.winner hold the latest tick

    The RNG counter lives on the device (BatchedTron.use_device_counter), so every replay draws fresh actions / spawns.
    Construction plays `ticks_per_replay` real ticks once (warm-up before capture); capture itself executes nothing.
    `ticks_per_replay` > 1 captures that many consecutive ticks in one graph.
    """

    def __init__(self, env, policy="random", ticks_per_replay=1):
        self.env = env
        env.use_device_counter()
        N, dev = env.N, env.device
        self.actions = torch.zeros((N, 2), dtype=torch.uint8, device=dev)
        self.obs = env.new_obs() if env.P else None
        self.reward = torch.empty((N, 2), dtype=torch.float32, device=dev)
        self.done = torch.empty(N, dtype=torch.uint8, device=dev)
        self.winner = torch.empty(N, dtype=torch.uint8, device=dev)
        self.ticks = int(ticks_per_replay)

        def body():
            for _ in range(self.ticks):
                act = None if policy == "random" else self.actions
                env.step(act, obs=self.obs, reward=self.reward, done=self.done, winner=self.winner, want_ep_len=False)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):  # warm-up outside capture
            body()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            body()

    def replay(self):
        self.graph.replay()
