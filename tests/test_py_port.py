"""The pure-Python loop port (bench.py's reference arm) against fixtures recorded from the reference: digests, pop_up planes,
slide-mode trajectories and the fuzz games cell for cell."""
import hashlib

import numpy as np

from oracle import py_port as pp

from _golden import load_json, load_npz


def digest_port(seed, ngames, W=10):
    rng = np.random.default_rng(seed)
    h = hashlib.sha256(); steps = 0; wins = [0, 0, 0]
    for _ in range(ngames):
        while True:
            x1, y1, x2, y2 = (int(v) for v in rng.integers(0, [W, W, W, W]))
            if (x1, y1) != (x2, y2):
                break
        g = pp.PyGame(W, W, (x1, y1), (x2, y2))
        h.update(g.board().view_for(1).astype(np.int8).tobytes())
        done = False
        while not done:
            a1, a2 = (int(v) for v in rng.integers(0, 4, size=2))
            s1, s2, done = g.step(a1, a2); steps += 1
            h.update(s1.astype(np.int8).tobytes()); h.update(s2.astype(np.int8).tobytes())
            h.update(bytes([int(done), g.winner or 0]))
        wins[g.winner or 0] += 1
    return h.hexdigest(), steps, wins


def test_port_reproduces_reference_digest():
    want = load_json("digests.json")["0"]
    got = digest_port(0, 1000)
    assert got[0] == want["sha256"] and got[1] == want["steps"] and got[2] == want["wins"]


def test_port_pop_up_matches_reference_fixture():
    pu = load_npz("popup.npz")
    for o, p in zip(pu["obs"][:16], pu["planes"][:16]):
        assert (pp.pop_up(o.astype(np.int64)) == p).all()


def test_port_slide_mode_matches_fixture():
    sl = load_npz("slide.npz")
    starts = np.concatenate([[0], np.cumsum(sl["length"] + 1)[:-1]])
    for gi in range(0, len(starts), 5):
        s = int(starts[gi]); sp = sl["spawn"][gi]
        tape = {"cur": (0, 0)}
        g = pp.PyGame(10, 10, (int(sp[0]), int(sp[1])), (int(sp[2]), int(sp[3])), mode="ice", bernoulli=lambda i: bool(tape["cur"][i]))
        for t in range(int(sl["length"][gi])):
            row = s + 1 + t
            tape["cur"] = tuple(int(x) for x in sl["slide"][row])
            o1, o2, done = g.step(int(sl["actions"][row][0]), int(sl["actions"][row][1]))
            assert (o1.astype(np.int8) == sl["obs1"][row]).all() and (o2.astype(np.int8) == sl["obs2"][row]).all()
            assert int(done) == int(sl["done"][row]) and (g.winner or 0) == int(sl["winner"][row])


def test_port_equals_reference_fuzz_games():
    """Cell for cell against the reference's own games in fuzz.json (W = H in [3, 16]): per tick, the per-game SHA-256 covers the
    Tile.value grid, both observations, alive flags, done, winner and both head positions, hashed as make_golden.make_fuzz does."""
    for g in load_json("fuzz.json"):
        W, sp = g["W"], g["spawn"]
        port = pp.PyGame(W, W, sp[:2], sp[2:])
        h = hashlib.sha256()
        for a1, a2 in g["actions"]:
            s1, s2, done = port.step(a1, a2)
            h.update(np.array([[t.value for t in row] for row in port.history[-1].board.cells], np.int8).tobytes())
            h.update(s1.astype(np.int8).tobytes()); h.update(s2.astype(np.int8).tobytes())
            h.update(bytes([int(a) for a in port.alive] + [int(done), port.winner or 0]))
            h.update(np.array(port.pos, np.int8).tobytes())
        assert port.done and (port.winner or 0) == g["winner"] and h.hexdigest() == g["sha256"], (W, sp)
