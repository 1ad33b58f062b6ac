"""GPU replay ring behind the reference's replay containers (DQN.py:81-132 ReplayMemory, DDQN.py:167-203 ReplayBuffer).

Three containers:
  ReplayRing  -- a ring of whole transitions (s, a, r, s', d) in HBM; push and gather are CUDA kernels, uniform sampling without
                 replacement is a keyed permutation evaluated inside the gather (replay_sample_gather: one launch per batch).
  FrameRing   -- the frame-sharing ring of the batched training loops (DDQN.py:264-308, DQN.py:198-252): the tick kernel writes
                 observations / rewards / done flags straight into time slot t % S, next_state of tick t is the frame of tick t+1,
                 so "push" moves no data at all; replay_frames_sample_gather draws a batch in one launch.
  StateRing   -- the same transitions from the env's bit-plane state: each tick stores the pre-tick state and the actions
                 (42 B per game-tick on bits10, against 3,467 B for DDQN's frame ring), and replay_states_sample_gather re-runs
                 the sampled ticks and renders s and s' in one launch, so the horizon can be thousands of ticks.

All three sample through one contract (_Sampler.sample): the same argument checks, `out=` reuse, `want_indices` and output
tuple; each ring supplies only its length and its C entry point.  FrameRing and StateRing share one loop interface:

    ring = FrameRing(env, n_slots)  or  StateRing(env, n_slots)
    obs = ring.begin()                                          # reset; the policy reads ring.obs
    loop:  env.select_actions(q(obs), eps, out=ring.actions_slot().view(-1)); obs = ring.step().obs
           batch = ring.sample(64)
"""
import ctypes as C

import torch

from . import _abi as abi
from . import _lib
from .batch_env import _CODE_OF, _TORCH_OF, _OnDevice


class _Sampler:
    """The sampling contract of the replay rings.  A ring has `lib`, `device`, `frame_shape`, `seed` and `sample_counter`,
    supplies __len__ (the transitions it can hand out) and _sample_call() -> (C entry point, its arguments before k)."""

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _next_counter(self, counter):
        """the sampler counter of this call: `counter`, or the ring's own, which then advances"""
        if counter is None:
            counter, self.sample_counter = self.sample_counter, self.sample_counter + 1
        return counter

    def _outputs(self, k, out_dtype, out=None):
        """(s, a, r, s', d) for k transitions: `out` (a tuple an earlier call returned, checked) or new tensors"""
        if out_dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("out_dtype must be float32 or bfloat16")
        if out is not None:
            s = out[0]
            if s.shape[0] != k or s.dtype != out_dtype or tuple(s.shape[1:]) != self.frame_shape:
                raise ValueError("sample: `out` does not match k / out_dtype / the frame shape")
            return tuple(out[:5])
        s = torch.empty((k,) + self.frame_shape, dtype=out_dtype, device=self.device)
        return (s, torch.empty((k, 1), dtype=torch.int64, device=self.device), torch.empty((k, 1), dtype=torch.float32, device=self.device),
                torch.empty_like(s), torch.empty((k, 1), dtype=torch.float32, device=self.device))

    def sample(self, k, out_dtype=torch.float32, counter=None, want_indices=False, out=None):
        """k distinct transitions, uniformly (random.sample, DDQN.py:191-200), sampled and gathered in ONE launch
        -> (s [k,*frame] out_dtype, a i64 [k,1], r f32 [k,1], s', d f32 [k,1]) (+ idx i64 [k] with want_indices).
        out: the 5-tuple a previous call returned, to write into the same tensors again (saves five allocations per batch)."""
        counter = self._next_counter(counter)
        if not 0 < k <= len(self):
            raise ValueError("sample: need 0 < k <= len(ring)=%d, got %d" % (len(self), k))
        s, a, r, s2, d = self._outputs(k, out_dtype, out)
        idx = torch.empty(k, dtype=torch.int64, device=self.device) if want_indices else None
        name, head = self._sample_call()
        with _OnDevice(self.device):
            _lib.check(getattr(self.lib, name)(*head, k, self.seed, counter, s.data_ptr(), s2.data_ptr(), _CODE_OF[out_dtype], a.data_ptr(),
                                               r.data_ptr(), d.data_ptr(), None if idx is None else idx.data_ptr(), self._stream()), name)
        return (s, a, r, s2, d, idx) if want_indices else (s, a, r, s2, d)


class ReplayRing(_Sampler):
    def __init__(self, capacity, frame_shape, frame_dtype=torch.bfloat16, device="cuda", seed=0):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type == "cuda" and self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.capacity = int(capacity)
        self.frame_shape = tuple(frame_shape)
        self.F = 1
        for d in self.frame_shape:
            self.F *= int(d)
        self.dt = frame_dtype if isinstance(frame_dtype, int) else _CODE_OF[frame_dtype]
        tdt = _TORCH_OF[self.dt]
        self.state = torch.zeros((self.capacity, self.F), dtype=tdt, device=self.device)
        self.next_state = torch.zeros((self.capacity, self.F), dtype=tdt, device=self.device)
        self.action = torch.zeros(self.capacity, dtype=torch.uint8, device=self.device)
        self.reward = torch.zeros(self.capacity, dtype=torch.float32, device=self.device)
        self.done = torch.zeros(self.capacity, dtype=torch.uint8, device=self.device)
        self.cursor = 0  # total transitions ever pushed
        self.seed, self.sample_counter = int(seed), 0
        self.ring = abi.ReplayRing(struct_size=C.sizeof(abi.ReplayRing), frame_elems=self.F, frame_dtype=self.dt, capacity=self.capacity,
                                   state=self.state.data_ptr(), next_state=self.next_state.data_ptr(), action=self.action.data_ptr(),
                                   reward=self.reward.data_ptr(), done=self.done.data_ptr())

    def __len__(self):
        return min(self.cursor, self.capacity)

    def push(self, state, next_state, action, reward, done, done_stride=1):
        """Append n transitions.  state/next_state: [n, *frame_shape] (ring dtype), action uint8 [n], reward f32 [n],
        done uint8 [n] (done_stride=1) or [n/2] (done_stride=2: one flag per env, two players per env)."""
        n = action.numel()
        if state.numel() != n * self.F or next_state.numel() != n * self.F or reward.numel() != n:
            raise ValueError("push: state/next_state must hold %d frames of %d elements and reward %d values" % (n, self.F, n))
        if done_stride not in (1, 2) or done.numel() * done_stride != n:
            raise ValueError("push: done must hold n/done_stride flags (n=%d, done_stride=%d, got %d)" % (n, done_stride, done.numel()))
        tdt = _TORCH_OF[self.dt]
        state = state.to(device=self.device, dtype=tdt).contiguous()
        next_state = next_state.to(device=self.device, dtype=tdt).contiguous()
        action = action.to(device=self.device, dtype=torch.uint8).contiguous()
        reward = reward.to(device=self.device, dtype=torch.float32).contiguous()
        done = done.to(device=self.device, dtype=torch.uint8).contiguous()
        off = 0
        chunk = self.capacity - self.capacity % done_stride  # whole envs per call, so the per-env done flags stay aligned
        if chunk <= 0:
            raise ValueError("push: capacity %d is smaller than done_stride %d" % (self.capacity, done_stride))
        while off < n:  # the ABI takes at most `capacity` transitions per call
            m = min(chunk, n - off)
            fo = off * self.F
            with _OnDevice(self.device):
                _lib.check(self.lib.replay_push(C.byref(self.ring), self.cursor, state.view(-1)[fo:].data_ptr(),
                                                next_state.view(-1)[fo:].data_ptr(), action[off:].data_ptr(), reward.view(-1)[off:].data_ptr(),
                                                done[(off // done_stride):].data_ptr(), done_stride, m, self._stream()), "replay_push")
            self.cursor += m
            off += m

    def sample_indices(self, k, counter=None):
        counter = self._next_counter(counter)
        if not 0 < k <= len(self):
            raise ValueError("sample_indices: need 0 < k <= len(ring)=%d, got %d" % (len(self), k))
        idx = torch.empty(k, dtype=torch.int64, device=self.device)
        with _OnDevice(self.device):
            _lib.check(self.lib.replay_sample_indices(len(self), k, self.seed, counter, idx.data_ptr(), self._stream()),
                       "replay_sample_indices")
        return idx

    def gather(self, idx, out_dtype=torch.float32):
        """-> (states [k,*frame], actions i64 [k,1], rewards f32 [k,1], next_states, dones f32 [k,1])  (DDQN.py:191-200)"""
        idx = idx.to(device=self.device, dtype=torch.int64).contiguous()
        k = idx.numel()
        s, a, r, s2, d = self._outputs(k, out_dtype)
        with _OnDevice(self.device):
            _lib.check(self.lib.replay_gather(C.byref(self.ring), idx.data_ptr(), k, s.data_ptr(), s2.data_ptr(), _CODE_OF[out_dtype],
                                              a.data_ptr(), r.data_ptr(), d.data_ptr(), self._stream()), "replay_gather")
        return s, a, r, s2, d

    def _sample_call(self):
        return "replay_sample_gather", (C.byref(self.ring), len(self))


class FrameRing(_Sampler):
    """Frame-sharing replay ring for a BatchedTron: S time slots of [rows = 2N] frames.

        ring = FrameRing(env, n_slots)
        obs = ring.begin()                                     # reset observation lands in slot 0
        loop:  act = policy(ring.obs); ring.step(act)          # tick t -> obs of tick t+1 lands in slot (t+1) % S
               batch = ring.sample(64)

    Transition (t, row): state = slot t % S, action/reward/done stored in slot t % S, next_state = slot (t+1) % S, or the
    terminal frame the tick kernel left in `terminal[t % S]` when the env finished at tick t (tron_step_args.obs_terminal).
    """

    def __init__(self, env, n_slots, keep_terminal=True, seed=0):
        if n_slots < 2:
            raise ValueError("FrameRing needs at least 2 slots")
        if not env.P:
            raise ValueError("FrameRing needs an environment with observations")
        self.lib = _lib.load()
        self.env, self.device = env, env.device
        self.S, self.rows = int(n_slots), 2 * env.N
        self.frame_shape = (env.P, env.W + 2, env.H + 2)
        self.F = env.P * env.C
        self.dt = env.obs_dtype
        tdt = _TORCH_OF[self.dt]
        N = env.N
        self.frames_t = torch.zeros((self.S, N, 2) + self.frame_shape, dtype=tdt, device=self.device)
        self.terminal_t = torch.zeros_like(self.frames_t) if keep_terminal else None
        self.action_t = torch.zeros((self.S, N, 2), dtype=torch.uint8, device=self.device)
        self.reward_t = torch.zeros((self.S, N, 2), dtype=torch.float32, device=self.device)
        self.done_t = torch.zeros((self.S, N), dtype=torch.uint8, device=self.device)
        self.winner = torch.empty(N, dtype=torch.uint8, device=self.device)
        self.tick = 0  # ticks played
        self.seed, self.sample_counter = int(seed), 0
        self.fr = abi.ReplayFrames(struct_size=C.sizeof(abi.ReplayFrames), frame_elems=self.F, frame_dtype=self.dt, n_slots=self.S, rows=self.rows,
                                   frames=self.frames_t.data_ptr(), terminal=None if self.terminal_t is None else self.terminal_t.data_ptr(),
                                   action=self.action_t.data_ptr(), reward=self.reward_t.data_ptr(), done=self.done_t.data_ptr())

    def _window(self):
        """(first_tick, n_ticks): the ticks whose transitions are complete, the last min(tick, S-1) (slot t+1 holds s' of tick t)"""
        n = min(self.tick, self.S - 1)
        return self.tick - n, n

    def __len__(self):
        return self._window()[1] * self.rows

    def frames(self, tick=None):
        """the observation the policy sees at `tick` (default: the current one): [N, 2, P, W+2, H+2], a view of the ring"""
        return self.frames_t[(self.tick if tick is None else tick) % self.S]

    @property
    def obs(self):
        """the observation the policy reads now: frames()"""
        return self.frames()

    def begin(self, spawn=None):
        self.tick = 0
        return self.env.reset(spawn=spawn, obs=self.frames_t[0])

    def actions_slot(self):
        """uint8 [N,2] view the policy writes the actions of the current tick into (select_actions(out=...))"""
        return self.action_t[self.tick % self.S]

    def step(self, actions=None, **kw):
        """one env tick whose outputs land in the ring; actions None -> the ones already written into actions_slot()"""
        env, t, S = self.env, self.tick, self.S
        slot, nslot = t % S, (t + 1) % S
        if actions is not None:
            self.action_t[slot].copy_(actions.reshape(env.N, 2))
        res = env.step(self.action_t[slot], obs=self.frames_t[nslot], reward=self.reward_t[slot], done=self.done_t[slot], winner=self.winner,
                       obs_terminal=None if self.terminal_t is None else self.terminal_t[slot], want_ep_len=False, **kw)
        self.tick = t + 1
        return res

    def _sample_call(self):
        return "replay_frames_sample_gather", (C.byref(self.fr),) + self._window()


class StateRing(_Sampler):
    """Replay ring of env states for a BatchedTron on a bit-plane layout: S time slots, each the state blob (planes + meta) BEFORE
    tick t, the actions of tick t and the RNG counter it ran with (plus the temper mode's game parameters).  A transition
    (s, a, r, s', d) is re-simulated when it is sampled: the sample kernel re-runs tick t of the game with tron_step's rules and
    renders the row's view of the pre- and post-tick states, so s' of a finished game is its last frame, as FrameRing's terminal
    frames.  Drop-in for FrameRing in a training loop:

        ring = StateRing(env, n_slots)
        obs = ring.begin()                                          # the policy reads ring.obs, refreshed in place every tick
        loop:  env.select_actions(q, eps, counter=env.counter, out=ring.actions_slot().view(-1)); obs = ring.step().obs
               batch = ring.sample(64)

    Same (seed, counter) and window as a FrameRing -> the same sampled transitions, bit for bit.  `obs` is one buffer that every
    step reuses, which lets BatchedTron.step store only the parts of each row that a tick changes; begin(obs=buf) or
    step(obs=buf) makes `buf` that buffer.
    """

    def __init__(self, env, n_slots, seed=0):
        if n_slots < 1:
            raise ValueError("StateRing needs at least 1 slot")
        if env.layout not in (abi.LAYOUT_BITS10, abi.LAYOUT_BITS):
            raise ValueError("StateRing re-runs ticks on bit-plane states: the env needs layout 'bits10' or 'bits' (got layout %d)" % env.layout)
        if env.slide_mode == abi.SLIDE_TAPE:
            raise ValueError("StateRing cannot replay slide_mode='tape': the tape is not recorded")
        if not env.P:
            raise ValueError("StateRing needs an environment with observations (obs_enc != 'none')")
        if not env.auto_reset:
            raise ValueError("StateRing needs auto_reset=True: a frozen finished game has no next state")
        self.lib = _lib.load()
        self.env, self.device = env, env.device
        self.S, self.rows = int(n_slots), 2 * env.N
        self.frame_shape = (env.P, env.W + 2, env.H + 2)
        N = env.N
        meta_off = C.c_size_t()
        _lib.check(self.lib.tron_state_offsets(N, env.W, env.H, env.layout, None, C.byref(meta_off), None), "tron_state_offsets")
        self.state_bytes = meta_off.value + 8 * N  # planes + meta: what a tick reads (the dirty boxes are the sparse kernel's)
        slot_bytes = (self.state_bytes + 15) & ~15
        self.states_t = torch.zeros((self.S, slot_bytes), dtype=torch.uint8, device=self.device)
        self.action_t = torch.zeros((self.S, N, 2), dtype=torch.uint8, device=self.device)
        self.counter_t = torch.zeros(self.S, dtype=torch.int64, device=self.device)
        self.params_t = torch.zeros((self.S, N, 4), dtype=torch.int8, device=self.device) if env.slide_mode == abi.SLIDE_TEMPER else None
        self.obs = env.new_obs()  # the observation the policy reads now
        self.tick = 0  # ticks played
        self.seed, self.sample_counter = int(seed), 0
        self.rs = abi.ReplayStates(struct_size=C.sizeof(abi.ReplayStates), n_slots=self.S, slot_bytes=slot_bytes, states=self.states_t.data_ptr(),
                                   action=self.action_t.data_ptr(), counter=self.counter_t.data_ptr(),
                                   slide_params=None if self.params_t is None else self.params_t.data_ptr())

    def _window(self):
        """(first_tick, n_ticks): the ticks in the ring, the last min(tick, S) (s' is re-simulated, no slot holds it)"""
        n = min(self.tick, self.S)
        return self.tick - n, n

    def __len__(self):
        return self._window()[1] * self.rows

    def begin(self, spawn=None, obs=None):
        """reset the env (its first observation lands in `obs`, which becomes self.obs) and start at tick 0"""
        if obs is not None:
            self.obs = obs
        self.tick = 0
        return self.env.reset(spawn=spawn, obs=self.obs)

    def actions_slot(self):
        """uint8 [N,2] view the policy writes the actions of the current tick into (select_actions(out=...))"""
        return self.action_t[self.tick % self.S]

    def step(self, actions=None, obs=None, **kw):
        """record the pre-tick state, then one env tick into self.obs (or `obs`, which becomes self.obs); actions None -> the ones
        already written into actions_slot().  All on the env's stream, so the step can be captured in a CUDA graph (with
        env.use_device_counter())."""
        env, slot = self.env, self.tick % self.S
        if actions is not None:
            self.action_t[slot].copy_(actions.reshape(env.N, 2))
        self.states_t[slot, :self.state_bytes].copy_(env.state[:self.state_bytes])
        if kw.get("counter") is not None:
            self.counter_t[slot].fill_(int(kw["counter"]))
        elif env.counter_dev is not None:
            self.counter_t[slot:slot + 1].copy_(env.counter_dev)
        else:
            self.counter_t[slot].fill_(env.counter)
        if self.params_t is not None:
            self.params_t[slot].copy_(env.slide_params)
        if obs is not None:
            self.obs = obs
        res = env.step(self.action_t[slot], obs=self.obs, want_ep_len=False, **kw)
        self.tick += 1
        return res

    def _sample_call(self):
        return "replay_states_sample_gather", (C.byref(self.rs), C.byref(self.env._args())) + self._window()
