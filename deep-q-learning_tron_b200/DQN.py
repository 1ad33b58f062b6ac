"""Drop-in for the replay side of the reference's DQN.py: Transition (DQN.py:78) and ReplayMemory (DQN.py:81-132),
stored in the GPU replay ring (replay_push / replay_gather kernels), plus a batched restatement of the survivor
training loop (DQN.py:135-309) on the vectorised environment."""
import random
from collections import namedtuple

import numpy as np
import torch

from tron.player import Direction, Player

import tron_b200
from tron_b200.replay import ReplayRing

device = 'cuda' if torch.cuda.is_available() else 'cpu'  # DQN.py:16
MEM_CAPACITY = 10000  # DQN.py:32
BATCH_SIZE = 128      # DQN.py:19
GAMMA = 0.9           # DQN.py:20
EPSILON_START, ESPILON_END, DECAY_RATE = 1, 0.003, 0.999  # DQN.py:23-25
GAME_CYCLE = 20       # DQN.py:35

class Ai(Player):
    """Drop-in for DQN.Ai (DQN.py:39-75): a player that owns a Q-net and picks epsilon-greedy moves from its own 1-plane observation.
    (In the reference's fork Game can no longer step such a player -- SURVEY section 0; the drop-in Game can.)"""

    def __init__(self, epsilon=0, net=None):
        super(Ai, self).__init__()
        from Net.DQNNet import Net
        self.net = net if net is not None else Net(in_planes=1).to(device)
        self.epsilon = epsilon

    def action(self, map, id):
        game_map = map.state_for_player(id)
        x = torch.from_numpy(np.reshape(game_map, (1, 1, game_map.shape[0], game_map.shape[1]))).float()
        with torch.no_grad():
            next_action = int(torch.argmax(self.net(x), 1)[0]) + 1
        if random.random() <= self.epsilon:
            next_action = random.randint(1, 4)
        return Direction(next_action)


Transition = namedtuple('Transition', ('old_state', 'action', 'new_state', 'reward', 'terminal'))


class ReplayMemory(object):
    """push(old_state (1,1,R,C) f32, action (1,1) f32, new_state, reward (1,1) f32, terminal bool); sample(k) -> [Transition]."""

    def __init__(self, capacity, frame_dtype=torch.float32, device="cuda"):
        self.capacity = capacity
        self._ring = None
        self._dt, self._dev = frame_dtype, device

    def _ensure(self, frame):
        if self._ring is None:
            self._ring = ReplayRing(self.capacity, tuple(frame.shape[1:]), self._dt, device=self._dev)

    def push(self, *args):
        old_state, action, new_state, reward, terminal = args
        self._ensure(old_state)
        self._ring.push(old_state, new_state, action.reshape(-1), reward.reshape(-1), torch.tensor([int(bool(terminal))], dtype=torch.uint8))

    def push_batch(self, old_state, action, new_state, reward, terminal, done_stride=1):
        self._ensure(old_state)
        self._ring.push(old_state, new_state, action, reward, terminal, done_stride)

    @property
    def position(self):
        return 0 if self._ring is None else self._ring.cursor % self.capacity

    def sample_batch(self, batch_size):
        """-> (old_state [k,...] f32, action i64 [k,1], reward f32 [k,1], new_state, terminal f32 [k,1]) on the device"""
        return self._ring.sample(batch_size)

    def sample(self, batch_size):
        s, a, r, s2, d = self.sample_batch(batch_size)
        return [Transition(s[i:i + 1], a[i:i + 1].float(), s2[i:i + 1], r[i:i + 1], bool(d[i, 0].item())) for i in range(batch_size)]

    def __len__(self):
        return 0 if self._ring is None else len(self._ring)


def learn_step(model, optimizer, batch):
    """One DQN learn step as in the reference's train() (DQN.py:263-292): predicted Q of the taken action, target r for a terminal
    transition else r + gamma * max_a Q(s', a) (same net, detached), smooth-L1 loss, one optimizer step.
    batch = (old_state [k,...], action i64 [k,1], reward f32 [k,1], new_state, terminal f32 [k,1]).  -> detached loss"""
    import torch.nn.functional as F
    s, a, r, s2, d = batch
    pred = model(s).gather(1, a).sum(dim=1)
    nxt = model(s2)
    target = (r.squeeze(1) + (1 - d.squeeze(1)) * model.gamma * nxt.max(1)[0]).detach()
    loss = F.smooth_l1_loss(pred, target)
    model.zero_grad()
    loss.backward()
    optimizer.step()
    return loss.detach()


def train(model=None, n_envs=4096, iterations=100, learn_steps_per_iter=1, device="cuda", seed=0, log=None, layout="auto", replay="frames",
          save_every=0, save_dir="save", on_cycle=None, timings=None, amp=False, buffer_size=None):
    """Batched restatement of DQN.train (DQN.py:135-309): self-play with the survivor reward (step index / 100 / -25 / 0),
    1-plane observations, one smooth-L1 learn step per cycle on a uniform sample, target r or r + gamma * max Q(s').

    replay="frames": the tick kernel fills a frame-sharing ring (no push); "ring": explicit transitions through replay_push;
    "states": a StateRing of env states that re-simulates sampled transitions, buffer_size transitions (default: the reference's
    capacity and at least one cycle of ticks) with no slot cap.
    save_every: write the reference's checkpoint (save/DQN.bak, DQN.py:295) every that many cycles.
    on_cycle(cycle, stats): the numbers the reference logs per cycle (DQN.py:296-306): loss, p1 win rate, mean duration.
    timings: optional dict receiving device times in ms summed over all ticks (q_forward, env_replay, learn).
    amp: run the ACTING forward under bf16 autocast (the learn step stays fp32 like the reference)."""
    import os
    from Net.DQNNet import Net
    from tron_b200.replay import FrameRing, StateRing
    model = model or Net(in_planes=1, batch_size=BATCH_SIZE, gamma=GAMMA).to(device)
    opt = torch.optim.Adam(model.parameters())
    env = tron_b200.BatchedTron(n_envs, 10, 10, device=device, obs_dtype=torch.float32, obs_enc="lut1", reward="survivor", seed=seed, layout=layout)
    rows = 2 * n_envs
    ring = mem = None
    if replay == "frames":  # at least the reference's capacity (DQN.py:32) and one cycle of ticks
        ring = FrameRing(env, max(GAME_CYCLE + 1, min(64, -(-MEM_CAPACITY // rows) + 1)), keep_terminal=True, seed=seed)
    elif replay == "states":
        want = buffer_size or max(MEM_CAPACITY, rows * GAME_CYCLE)
        ring = StateRing(env, max(2, -(-want // rows)), seed=seed)
    else:
        mem = ReplayMemory(max(MEM_CAPACITY, rows * GAME_CYCLE), device=device)
    obs = ring.begin() if ring is not None else env.reset()
    epsilon = float(EPSILON_START)
    losses = []
    events, learn_events = [], []
    last_stats = env.stats_dict()
    for it in range(iterations):
        for _ in range(GAME_CYCLE):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record()
            with torch.no_grad():
                if amp:
                    with torch.autocast("cuda", dtype=torch.bfloat16):
                        q = model(obs.view(rows, 1, 12, 12)).float()
                else:
                    q = model(obs.view(rows, 1, 12, 12))
            ev[1].record()
            if ring is not None:
                env.select_actions(q, epsilon, counter=env.counter, out=ring.actions_slot().view(-1))
                obs = ring.step().obs
            else:
                act = env.select_actions(q, epsilon, counter=env.counter)
                term = obs.clone()
                res = env.step(act, obs_terminal=term)
                nxt = torch.where(res.done.view(-1, 1, 1, 1, 1).bool(), term, res.obs)  # a finished game's new_state is its last frame (DQN.py:205-252)
                mem.push_batch(obs.view(rows, 1, 12, 12), act.view(-1), nxt.view(rows, 1, 12, 12), res.reward.view(-1), res.done, done_stride=2)
                obs = res.obs
            ev[2].record()
            events.append(ev)
            if epsilon * DECAY_RATE > ESPILON_END:
                epsilon *= DECAY_RATE
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(learn_steps_per_iter):
            have = len(ring) if ring is not None else len(mem)
            k = min(have, model.batch_size)
            batch = ring.sample(k) if ring is not None else mem.sample_batch(k)
            losses.append(learn_step(model, opt, batch))
        e1.record()
        learn_events.append((e0, e1))
        if save_every and (it + 1) % save_every == 0:
            os.makedirs(save_dir, exist_ok=True)
            torch.save(model.state_dict(), os.path.join(save_dir, "DQN.bak"))
        if on_cycle is not None or log:
            st = env.stats_dict()
            d = {k: st[k] - last_stats[k] for k in st}
            last_stats = st
            info = dict(loss=float(losses[-1]), p1_winrate=d["p1_wins"] / max(1, d["episodes"]), duration=d["ep_ticks"] / max(1, d["episodes"]),
                        episodes=d["episodes"], p1_wins=d["p1_wins"], p2_wins=d["p2_wins"], draws=d["draws"], epsilon=epsilon)
            if on_cycle is not None:
                on_cycle(it + 1, info)
            if log:
                log(it, info["loss"], st)
    torch.cuda.synchronize()
    losses = [float(l) for l in losses]
    if timings is not None:
        timings.update(ticks=len(events), q_forward_ms=sum(e[0].elapsed_time(e[1]) for e in events),
                       env_replay_ms=sum(e[1].elapsed_time(e[2]) for e in events), learn_ms=sum(a.elapsed_time(b) for a, b in learn_events),
                       learn_steps=len(losses), replay=replay, layout=env.layout)
    return model, losses
