"""Drop-in for the replay side of the reference's DDQN.py -- ReplayBuffer (DDQN.py:167-203) on the GPU replay ring -- and a
batched restatement of Agent.learn / train (DDQN.py:73-165, 206-346): 65,536+ self-play games per GPU, epsilon-greedy from the
live Q-net, Double-DQN target, MSE, Adam, soft update; optional data-parallel gradient all-reduce over NCCL (one flat bucket,
overlapped with the next env tick)."""
import os

import torch

import tron_b200
from tron_b200.replay import FrameRing, ReplayRing, StateRing

EPSILON_START, ESPILON_END, DECAY_RATE = 1, 0.003, 0.999  # DDQN.py:18-20
TAU = 0.001             # DDQN.py:21
MEM_CAPACITY = int(1e5)  # DDQN.py:26
UPDATE_EVERY = 4        # DDQN.py:29
GAME_CYCLE = 20         # DDQN.py:30
BATCH_SIZE = 64         # config.py:7
GAMMA = 0.9             # config.py:5


class ReplayBuffer:
    """add(state (1,P,R,C), action int, reward number, next_state, done bool); sample() -> (states, actions i64, rewards f32,
    next_states, dones f32) on the device, batch_size rows without replacement (DDQN.py:191-200)."""

    def __init__(self, action_size, buffer_size, batch_size, frame_dtype=torch.float32, device="cuda"):
        self.action_size = action_size
        self.buffer_size = int(buffer_size)
        self.batch_size = batch_size
        self._ring = None
        self._dt, self._dev = frame_dtype, device

    def _ensure(self, frame):
        if self._ring is None:
            self._ring = ReplayRing(self.buffer_size, tuple(frame.shape[1:]), self._dt, device=self._dev)

    def add(self, state, action, reward, next_state, done):
        state, next_state = torch.as_tensor(state), torch.as_tensor(next_state)
        self._ensure(state)
        self._ring.push(state, next_state, torch.tensor([int(action)], dtype=torch.uint8), torch.tensor([float(reward)]),
                        torch.tensor([int(bool(done))], dtype=torch.uint8))

    def add_batch(self, state, action, reward, next_state, done, done_stride=1):
        self._ensure(state)
        self._ring.push(state, next_state, action, reward, done, done_stride)

    def sample(self, out_dtype=torch.float32):
        return self._ring.sample(self.batch_size, out_dtype)

    def __len__(self):
        return 0 if self._ring is None else len(self._ring)


class Agent:
    """Batched counterpart of DDQN.Agent (DDQN.py:34-165).

    All gradients live in ONE flat fp32 buffer (every parameter's .grad is a view of it), so the data-parallel exchange is a
    single NCCL all-reduce with no concatenation or copy-back.  learn() is the reference's learn step; learn_begin() /
    learn_finish() split it around the collective so that the caller can run the next env tick while the all-reduce is in flight."""

    def __init__(self, in_planes=3, device="cuda", buffer_size=1 << 20, batch_size=BATCH_SIZE, frame_dtype=torch.bfloat16, lr=1e-3,
                 data_parallel=False):
        from Net.DQNNet import Net
        self.device = torch.device(device)
        self.qnetwork_local = Net(in_planes).to(self.device)
        self.qnetwork_target = Net(in_planes).to(self.device)
        self.qnetwork_target.load_state_dict(self.qnetwork_local.state_dict())
        self.optimizer = torch.optim.Adam(self.qnetwork_local.parameters(), lr=lr)
        self.memory = ReplayBuffer(4, buffer_size, batch_size, frame_dtype, device=self.device)
        self.epsilon = 0.0
        self.totalloss, self.steps = 0.0, 0
        self._loss_sum = torch.zeros((), device=self.device)
        self.data_parallel = data_parallel
        params = list(self.qnetwork_local.parameters())
        self.flat_grad = torch.zeros(sum(p.numel() for p in params), dtype=torch.float32, device=self.device)
        off = 0
        for p in params:
            p.grad = self.flat_grad[off:off + p.numel()].view_as(p)
            off += p.numel()
        self._comm = None          # side stream of the overlapped all-reduce
        self._pending = None       # event: the all-reduce of the learn step in flight has finished
        self.allreduce_events = []  # (start, end) CUDA events of every overlapped all-reduce (timing)
        if data_parallel:  # identical initial weights on every rank
            import torch.distributed as dist
            for p in list(self.qnetwork_local.parameters()) + list(self.qnetwork_target.parameters()):
                dist.broadcast(p.data, 0)

    def q_values(self, obs, amp=False):
        """acting forward; amp=True runs it under bf16 autocast (cuDNN/cuBLAS tensor-core paths, observations are already bf16)"""
        self.qnetwork_local.eval()
        with torch.no_grad():
            if amp:
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    q = self.qnetwork_local(obs).float()
            else:
                q = self.qnetwork_local(obs)
        self.qnetwork_local.train()
        return q

    # ---- the learn step (DDQN.py:115-165), in three pieces -----------------------------------------------------------
    def _backward(self, experiences, gamma):
        states, actions, rewards, next_state, dones = experiences
        self.qnetwork_local.train(); self.qnetwork_target.eval()
        predicted = self.qnetwork_local(states).gather(1, actions)
        self.qnetwork_local.eval()
        with torch.no_grad():  # Double DQN: argmax from the local net, value from the target net (DDQN.py:131-134)
            a_loc = self.qnetwork_local(next_state).max(1)[1].unsqueeze(1)
            labels_next = self.qnetwork_target(next_state).gather(1, a_loc)
        self.qnetwork_local.train()
        labels = rewards + gamma * labels_next * (1 - dones)
        loss = torch.nn.functional.mse_loss(predicted, labels)
        self.optimizer.zero_grad(set_to_none=False)  # keep the views into flat_grad
        loss.backward()
        return loss.detach()

    def _apply(self):
        self.optimizer.step()
        with torch.no_grad():  # soft update (DDQN.py:154-165)
            tp = list(self.qnetwork_target.parameters())
            torch._foreach_mul_(tp, 1 - TAU)
            torch._foreach_add_(tp, list(self.qnetwork_local.parameters()), alpha=TAU)

    def learn(self, experiences, gamma=GAMMA):
        """one learn step, blocking form (the reference's order of operations)"""
        self.learn_finish()
        loss = self._backward(experiences, gamma)
        if self.data_parallel:
            allreduce_gradients(self.qnetwork_local, self.flat_grad)
        self._apply()
        self._loss_sum += loss; self.steps += 1
        return loss

    def learn_begin(self, experiences, gamma=GAMMA):
        """forward + backward, then launch the gradient all-reduce on a side stream and return; the optimizer step and the soft
        update happen in learn_finish() (call it after the next tick's kernels have been enqueued)."""
        self.learn_finish()
        loss = self._backward(experiences, gamma)
        self._loss_sum += loss; self.steps += 1
        if self.data_parallel:
            import torch.distributed as dist
            if self._comm is None:
                self._comm = torch.cuda.Stream(device=self.device)
            cur = torch.cuda.current_stream(self.device)
            ready = torch.cuda.Event()
            ready.record(cur)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(self._comm):
                self._comm.wait_event(ready)
                e0.record(self._comm)
                dist.all_reduce(self.flat_grad, op=dist.ReduceOp.AVG)
                e1.record(self._comm)
            self.allreduce_events.append((e0, e1))
            self._pending = e1
        else:
            self._apply()  # no collective to hide: same order of operations as learn()
        return loss

    def learn_finish(self):
        if self._pending is None:
            return
        torch.cuda.current_stream(self.device).wait_event(self._pending)
        self._pending = None
        self._apply()

    def get_loss(self):
        """mean loss since the last call (DDQN.py:65-70); synchronises"""
        out = float(self._loss_sum) / max(self.steps, 1)
        self.totalloss = out
        self._loss_sum.zero_(); self.steps = 0
        return out

    # ---- checkpoints: the reference's files (DDQN.py:60-63 local_ai.bak / target_ai.bak, DDQN.py:326 save/DDQN.bak) + resume bundle
    def save(self, directory, env=None, extra=None):
        self.learn_finish()
        os.makedirs(directory, exist_ok=True)
        torch.save(self.qnetwork_target.state_dict(), os.path.join(directory, "DDQN.bak"))
        torch.save(self.qnetwork_local.state_dict(), os.path.join(directory, "local_ai.bak"))
        torch.save(self.qnetwork_target.state_dict(), os.path.join(directory, "target_ai.bak"))
        bundle = dict(optimizer=self.optimizer.state_dict(), epsilon=self.epsilon, extra=extra or {},
                      env=None if env is None else env.state_dict())
        torch.save(bundle, os.path.join(directory, "resume.pt"))

    def load(self, directory, env=None):
        """-> the `extra` dict stored by save()"""
        self.qnetwork_local.load_state_dict(torch.load(os.path.join(directory, "local_ai.bak"), map_location=self.device))
        self.qnetwork_target.load_state_dict(torch.load(os.path.join(directory, "target_ai.bak"), map_location=self.device))
        path = os.path.join(directory, "resume.pt")
        if not os.path.exists(path):
            return {}
        bundle = torch.load(path, map_location=self.device, weights_only=False)
        self.optimizer.load_state_dict(bundle["optimizer"])
        self.epsilon = bundle["epsilon"]
        if env is not None and bundle.get("env") is not None:
            env.load_state_dict(bundle["env"])
        return bundle.get("extra", {})


def allreduce_gradients(model, flat=None):
    """One all-reduce of the flattened gradient (501,924 fp32 = 2.0 MB for the DQN net), averaged over ranks.  With the Agent's
    flat gradient buffer this is the whole exchange; without one the gradients are packed and unpacked around it."""
    import torch.distributed as dist
    world = dist.get_world_size()
    if flat is not None:
        if dist.get_backend() == "nccl":
            dist.all_reduce(flat, op=dist.ReduceOp.AVG)
        else:
            dist.all_reduce(flat, op=dist.ReduceOp.SUM)
            flat.div_(world)
        return
    grads = [p.grad for p in model.parameters() if p.grad is not None]
    packed = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(packed, op=dist.ReduceOp.SUM)
    packed.div_(world)
    off = 0
    for g in grads:
        n = g.numel()
        g.copy_(packed[off:off + n].view_as(g))
        off += n


def train(n_envs=65536, env_steps=64, device=None, seed=0, obs_dtype=torch.bfloat16, learn_every=UPDATE_EVERY, data_parallel=None, log=None,
          amp=False, layout="auto", replay="frames", buffer_size=None, overlap=True, save_every=0, save_dir="save", resume=None,
          on_cycle=None, timings=None, warmup_steps=0):
    """Batched DDQN loop (DDQN.py:206-346 restated): every tick both players of all envs act epsilon-greedily from the
    local net, 2*n_envs transitions enter the GPU replay, and every `learn_every` ticks one Double-DQN learn step runs.
    Under torchrun each rank owns n_envs envs (env_id_base = rank * n_envs) and gradients are all-reduced.

    replay="frames": the tick kernel writes observations / rewards / done flags straight into a frame-sharing ring (no push);
    replay="ring": explicit (s, a, r, s', d) ring filled by replay_push (round-1 path, kept for comparison).
    replay="states": a StateRing keeps each tick's env state (42 B per game-tick) and re-simulates the sampled transitions, so the
    window is ceil(buffer_size / (2 n_envs)) ticks with no slot cap; the env steps one reused observation buffer.
    overlap: launch the gradient all-reduce on a side stream and run the next tick's forward + env step while it is in flight
    (the optimizer step then lands one tick later than in the reference's strictly sequential loop).
    save_every: every that many GAME_CYCLEs write the reference's checkpoint files + a resume bundle into save_dir (DDQN.py:326).
    on_cycle(cycle, stats): called every GAME_CYCLE ticks with the counters the reference logs (DDQN.py:328-344): mean loss,
    mean episode duration, win/draw counts since the last call.
    timings: optional dict that receives per-phase device times in ms (q_forward, env_replay, learn, allreduce) summed over the
    ticks after `warmup_steps`."""
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if data_parallel is None:
        data_parallel = world > 1
    if device is None:
        device = "cuda:%d" % int(os.environ.get("LOCAL_RANK", "0"))
    if data_parallel and not dist.is_initialized():
        dist.init_process_group("nccl")
    torch.manual_seed(seed)
    agent = Agent(3, device, frame_dtype=obs_dtype, data_parallel=data_parallel, buffer_size=buffer_size or (1 << 20))
    env = tron_b200.BatchedTron(n_envs, 10, 10, device=device, obs_dtype=obs_dtype, obs_enc="popup3", reward="ddqn", seed=seed,
                                env_id_base=rank * n_envs, layout=layout)
    epsilon = float(EPSILON_START)
    start_tick = 0
    if resume:
        extra = agent.load(resume, env)
        epsilon = float(extra.get("epsilon", epsilon)); start_tick = int(extra.get("tick", 0))
    rows = 2 * n_envs
    want = buffer_size or MEM_CAPACITY
    ring = None
    if replay == "frames":
        ring = FrameRing(env, max(3, min(64, -(-want // rows) + 1)), keep_terminal=True, seed=seed)
    elif replay == "states":  # buffer_size transitions, at least two ticks
        ring = StateRing(env, max(2, -(-want // rows)), seed=seed)
    if ring is not None:
        obs = ring.begin() if not resume else env.observe(ring.obs)
    else:
        obs = env.reset() if not resume else env.observe()
    events = []
    sample_bufs = None
    n_learn = 0
    last_stats = env.stats_dict()
    batch = agent.memory.batch_size
    for t in range(start_tick, start_tick + env_steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        q = agent.q_values(obs.view(rows, 3, 12, 12), amp=amp)
        ev[1].record()
        if ring is not None:
            env.select_actions(q, epsilon, counter=env.counter, out=ring.actions_slot().view(-1))
            obs = ring.step().obs
        else:
            act = env.select_actions(q, epsilon, counter=env.counter)
            term = obs.clone()  # finished games: next_state is their last frame (DDQN.py:270-308), other rows are overwritten below
            res = env.step(act, obs_terminal=term)
            nxt = torch.where(res.done.view(-1, 1, 1, 1, 1).bool(), term, res.obs)
            agent.memory.add_batch(obs.view(rows, 3, 12, 12), act.view(-1), res.reward.view(-1), nxt.view(rows, 3, 12, 12), res.done, done_stride=2)
            obs = res.obs
        ev[2].record()
        agent.learn_finish()  # the learn step begun last tick: its all-reduce ran behind this tick's forward + env step
        have = len(ring) if ring is not None else len(agent.memory)
        if (t + 1) % learn_every == 0 and have > batch:
            # the sampled batch is consumed by backward before the next learn step, so its buffers are reused
            exp = sample_bufs = (ring.sample(batch, out=sample_bufs) if ring is not None else agent.memory.sample())
            n_learn += 1
            if overlap:
                agent.learn_begin(exp)
            else:
                agent.learn(exp)
        ev[3].record()
        if t - start_tick >= warmup_steps:
            events.append(ev)
        if (t + 1) % GAME_CYCLE == 0:
            if epsilon * DECAY_RATE > ESPILON_END:  # DDQN.py:311-313
                epsilon *= DECAY_RATE
            agent.epsilon = epsilon
            cycle = (t + 1) // GAME_CYCLE
            if on_cycle is not None:
                st = env.stats_dict()
                d = {k: st[k] - last_stats[k] for k in st}
                last_stats = st
                on_cycle(cycle, dict(loss=agent.get_loss(), duration=d["ep_ticks"] / max(1, d["episodes"]), episodes=d["episodes"],
                                     p1_wins=d["p1_wins"], p2_wins=d["p2_wins"], draws=d["draws"], epsilon=epsilon, env_steps=d["env_steps"]))
            if save_every and cycle % save_every == 0 and rank == 0:
                agent.save(save_dir, env, extra=dict(epsilon=epsilon, tick=t + 1))
        if log:
            torch.cuda.synchronize()
            log(t, dict(forward_ms=ev[0].elapsed_time(ev[1]), env_replay_ms=ev[1].elapsed_time(ev[2]), learn_ms=ev[2].elapsed_time(ev[3]),
                        loss=float(agent._loss_sum) / max(agent.steps, 1)))
    agent.learn_finish()
    torch.cuda.synchronize()
    agent.totalloss = float(agent._loss_sum)
    if timings is not None:
        # device time of each overlapped all-reduce, from "backward finished" to "reduced gradient ready": includes waiting for the
        # slowest rank to reach the collective, which is why min (~ the collective itself) and median are reported next to the sum
        ar = [a.elapsed_time(b) for a, b in agent.allreduce_events]
        timings.update(ticks=len(events), q_forward_ms=sum(e[0].elapsed_time(e[1]) for e in events),
                       env_replay_ms=sum(e[1].elapsed_time(e[2]) for e in events), learn_ms=sum(e[2].elapsed_time(e[3]) for e in events),
                       allreduce_ms=sum(ar), allreduce_calls=len(ar), allreduce_us_min=1e3 * min(ar) if ar else 0.0,
                       allreduce_us_median=1e3 * sorted(ar)[len(ar) // 2] if ar else 0.0, allreduce_us_max=1e3 * max(ar) if ar else 0.0,
                       learn_steps=n_learn, replay=replay, layout=env.layout)
    return agent, env
