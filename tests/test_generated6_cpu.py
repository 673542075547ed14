"""CPU suite of the generated six-player games (SIXPLAYER.md §6) on the oracle alone: oracle/generated6.py's replay must produce
records that are one-hot at a legal action, only from recorded seats, the script's action on script seats, value targets that follow
the status rule, images the oracle can encode; and six random seats must be the rollout replay of tests/test_env6_gpu.py."""
import numpy as np
import pytest

from oracle import pyoracle as po
from oracle import script6
from oracle.generated6 import Generated6, play
from oracle.samples6 import LOSS

SEED = 0x5EED0006


def check_block(blob, script, record_seats, rules):
    recs = np.frombuffer(blob, np.uint8).reshape(-1, 288)
    o, enc = po.Oracle6Game(rules), po.Oracle6Mcts(rules)
    status = int(recs[0, 284].view(np.int8))
    assert (recs[:, 284].view(np.int8) == status).all() and status in (-2, 0, 1, 2, 3, 4, 5)
    assert (recs[:, 285:] == 0).all()
    pi = recs[:, 112:284].copy().view(np.float32)
    assert ((pi == 0.0) | (pi == 1.0)).all() and (pi.sum(1) == 1.0).all()
    z = recs[:, 108:112].copy().view(np.float32).reshape(-1)
    for r, a, v in zip(recs, pi.argmax(1), z):
        seat = int(r[98])
        assert (record_seats >> seat) & 1
        o.set_image(r[:108])
        assert o.status() == -1 and (o.valid() >> int(a)) & 1
        if (script >> seat) & 1:
            assert script6.script_action(o) == a
        assert v == (np.float32(0.0) if status == -2 else np.float32(1.0) if status == seat else LOSS)
        assert np.isfinite(enc.encode(o)).all()
    return len(recs)


@pytest.mark.parametrize("script,record_seats,kw", [(0x3f, 0x3f, {}), (0x01, 0x01, {}), (0x15, 0x3f, {}), (0x00, 0x22, dict(limit_attack=1))],
                         ids=["six_scripts", "one_script_recorded", "scripts_0_2_4", "random_limit_attack"])
def test_replay_records(script, record_seats, kw):
    rules = po.default_rules(**kw)
    g = Generated6(6, 30, SEED, rules)
    blocks = g.play(script, record_seats, 900) + g.play(script, record_seats, 900)
    assert len(blocks) >= 3
    n = sum(check_block(b, script, record_seats, rules) for b in blocks)
    assert n > 0
    # a game still running holds its staged samples, only from recorded seats
    for staged in g.staged:
        assert all((record_seats >> int(img[98])) & 1 for img, _ in staged)


def test_split_calls_equal_one_call():
    a = Generated6(4, 7, SEED)
    b1 = a.play(0x0b, 0x3f, 700) + a.play(0x0b, 0x3f, 1100)
    b = Generated6(4, 7, SEED)
    b2 = b.play(0x0b, 0x3f, 1800)
    assert (a.images() == b.images()).all() and a.counters == b.counters and sorted(b1) == sorted(b2)


def test_six_random_seats_are_the_rollout():
    n, steps, first = 6, 1500, 40
    img, cnt, blocks = play(n, first, SEED, 0, 0, steps)
    assert blocks == []
    games, draws, wins = 0, 0, [0] * 6
    o = po.Oracle6Game()
    for g in range(n):
        o.new_game(SEED, first + g, 0)
        for ply in range(steps):
            st = o.status()
            if st != -1:
                games += 1
                if st == -2:
                    draws += 1
                else:
                    wins[st] += 1
                o.new_game(SEED, first + g, ply)
            assert o.move(o.random_action(SEED, first + g, ply), SEED, first + g, ply) == 0
        assert (img[g] == o.image()).all(), g
    assert cnt == dict(steps=n * steps, games=games, draws=draws, wins=wins) and games > 0
