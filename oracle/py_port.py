"""Pure-Python port of the reference's one-game-at-a-time loop.  TEST INFRASTRUCTURE / CPU BASELINE ONLY.

The reference (ckawoalt/Deep-Q-Learning_TRON) is Python and cannot travel to the GPU box, so the
"reference arm" of bench.py times this port instead.  It keeps the reference's data structures and
per-tick work so that it costs what the reference costs: an object-dtype ndarray of enum tiles with a
freshly recomputed border on every clone/apply (tron/map.py:43-58), a per-cell colour callback for each
player's observation (tron/map.py:67-84), a full grid copy appended to the history every tick and
Direction enums for the moves (tron/game.py:149-252, tron/player.py:107-132).  Logic is written from the
normative restatement in SURVEY.md section 8a, not copied.

Pinned by tests/test_py_port.py: same SHA-256 digests as the reference on 2 x 1000 seeded games and cell-for-cell
equality with the reference's 300 recorded fuzz games.  Measured next to the live reference on one Xeon host, the port
ran 2.4-2.7k env-steps/s/core against the reference's 2.5k.
"""
import enum
import random

import numpy as np


class Tile(enum.Enum):  # tron/map.py:9-17
    EMPTY = 0
    WALL = -1
    P1_BODY = 1
    P1_HEAD = 2
    P2_BODY = 3
    P2_HEAD = 4
    P1_SLIDE = 5
    P2_SLIDE = 6


class Heading(enum.Enum):  # tron/player.py:4-8
    UP = 1
    RIGHT = 2
    DOWN = 3
    LEFT = 4


def _edge(i, j, rows, cols):
    return i == 0 or i == rows - 1 or j == 0 or j == cols - 1


def _bordered(w, h, inner, edge):
    # same double comprehension + ndarray construction the reference pays on every Map() (tron/map.py:48)
    return np.array([[edge if _edge(i, j, w + 2, h + 2) else inner for i in range(h + 2)] for j in range(w + 2)])


def _colour(tile, viewer):  # tron/map.py:67-81
    if tile == Tile.EMPTY:
        return 1
    if tile == Tile.WALL:
        return -1
    if tile == Tile.P1_BODY or tile == Tile.P1_SLIDE:
        return -2 if viewer == 1 else -3
    if tile == Tile.P1_HEAD:
        return 10 if viewer == 1 else -10
    if tile == Tile.P2_BODY or tile == Tile.P2_SLIDE:
        return -3 if viewer == 1 else -2
    if tile == Tile.P2_HEAD:
        return 10 if viewer == 2 else -10
    return None


class Board:
    def __init__(self, w, h, inner=Tile.EMPTY, edge=Tile.WALL):
        self.w, self.h = w, h
        self.cells = _bordered(w, h, inner, edge)

    def copy(self):  # tron/map.py:50-53: a new bordered Map is built, then its data replaced
        other = Board(self.w, self.h, 0, 0)
        other.cells = np.copy(self.cells)
        return other

    def mapped(self, fn):  # tron/map.py:55-58
        other = Board(self.w, self.h, 0, 0)
        other.cells = np.array([[fn(self.cells[i][j]) for i in range(self.h + 2)] for j in range(self.w + 2)])
        return other

    def view_for(self, viewer):  # tron/map.py:83-84
        return self.mapped(lambda t: _colour(t, viewer)).cells.T

    def get(self, pos):
        return self.cells[pos[0] + 1][pos[1] + 1]

    def put(self, pos, tile):
        self.cells[pos[0] + 1][pos[1] + 1] = tile


class Frame:  # tron/game.py:61-65
    def __init__(self, board):
        self.board = board
        self.heading = [None, None]


_BODY = (Tile.P1_BODY, Tile.P2_BODY)
_HEAD = (Tile.P1_HEAD, Tile.P2_HEAD)
_SLIDE = (Tile.P1_SLIDE, Tile.P2_SLIDE)


def _heading_of(action):  # tron/player.py:107-118
    return Heading(action + 1)


def _advance(pos, heading):  # tron/player.py:124-132
    if heading == Heading.UP:
        return (pos[0] - 1, pos[1])
    if heading == Heading.RIGHT:
        return (pos[0], pos[1] + 1)
    if heading == Heading.DOWN:
        return (pos[0] + 1, pos[1])
    return (pos[0], pos[1] - 1)


class PyGame:
    """One game; step(a1, a2) -> (obs_p1, obs_p2, done) like the reference's Game.step."""

    def __init__(self, w, h, start1, start2, mode=None, slide=0.15, bernoulli=None):
        self.w, self.h = w, h
        self.pos = [tuple(start1), tuple(start2)]
        self.alive = [True, True]
        self.winner = None
        self.done = False
        self.mode, self.slide, self.bernoulli = mode, slide, bernoulli
        board = Board(w, h)
        self.history = [Frame(board)]
        for i in (0, 1):
            board.put(self.pos[i], _HEAD[i])

    def board(self):
        return self.history[-1].board.copy()

    def step(self, a1, a2):
        scratch = self.board()
        acts = (a1, a2)
        for i in (0, 1):
            scratch.put(self.pos[i], _BODY[i])
        headings = [None, None]
        for i in (0, 1):
            headings[i] = _heading_of(acts[i])
            self.pos[i] = _advance(self.pos[i], headings[i])
            if self.mode is not None:
                p = self.pos[i]
                if 0 <= p[0] < self.w and 0 <= p[1] < self.h and scratch.get(p) is Tile.EMPTY:
                    slip = self.bernoulli(i) if self.bernoulli else (random.random() <= self.slide)
                    if slip:
                        scratch.put(p, _SLIDE[i])
                        self.pos[i] = _advance(p, headings[i])
        self.history[-1].heading = headings
        for i in (0, 1):
            p = self.pos[i]
            if p[0] < 0 or p[1] < 0 or p[0] >= self.w or p[1] >= self.h or scratch.get(p) is not Tile.EMPTY:
                self.alive[i] = False
            scratch.put(p, _HEAD[i])
        self.history.append(Frame(scratch))
        obs1 = scratch.view_for(1)
        obs2 = scratch.view_for(2)
        n_alive = sum(self.alive)
        if n_alive <= 1:
            if n_alive == 1 and self.pos[0] != self.pos[1]:
                self.winner = 1 if self.alive[0] else 2
            self.done = True
        return obs1, obs2, self.done


def pop_up(obs):  # tron/util.py:11-37 (per-cell Python loop, as the reference does it)
    rows, cols = obs.shape
    wall = np.zeros((rows, cols)); mine = np.zeros((rows, cols)); enemy = np.zeros((rows, cols))
    for i in range(rows):
        for j in range(cols):
            v = obs[i][j]
            if v == -1:
                wall[i][j] = 1
            elif v == -2:
                mine[i][j] = 1
            elif v == -3:
                enemy[i][j] = 1
            elif v == -10:
                enemy[i][j] = 10
            elif v == 10:
                mine[i][j] = 10
    return np.stack([wall, mine, enemy])


def spawn(rng, w, h):  # tron/util.py:70-78
    x1, y1 = rng.randint(0, w - 1), rng.randint(0, h - 1)
    x2, y2 = rng.randint(0, w - 1), rng.randint(0, h - 1)
    while x1 == x2 and y1 == y2:
        x1, y1 = rng.randint(0, w - 1), rng.randint(0, h - 1)
    return (x1, y1), (x2, y2)


def play_random(seed, env_steps, w=10, h=10, with_pop_up=False):
    """Auto-reset random-policy loop (the CPU-baseline workload): returns (env_steps_done, episodes)."""
    rng = random.Random(seed)
    done_steps = episodes = 0
    while done_steps < env_steps:
        s1, s2 = spawn(rng, w, h)
        g = PyGame(w, h, s1, s2)
        over = False
        while not over and done_steps < env_steps:
            o1, o2, over = g.step(rng.randrange(4), rng.randrange(4))
            if with_pop_up:
                pop_up(o1); pop_up(o2)
            done_steps += 1
        episodes += 1
    return done_steps, episodes
