"""CPU checks of the six-player lockstep search on the oracle (oracle/risk6_lockstep.c, SIXPLAYER.md §2): with one descent per round it
is r6_mcts_search bit for bit; with K descents per round every simulation is backed up, every active_N mark is taken off again, the
active_N rule passes moves over, and a K that does not divide the simulation count is rejected."""
import numpy as np
import pytest

from oracle import pyoracle as po
from oracle.lockstep6 import Lockstep6Mcts

SEED = 0x5EED0001


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def positions(rules, n_games=12, every=9, plies=240):
    """positions reached by oracle random play: every `every`-th ply of `n_games` games (running games only)"""
    out = []
    for g in range(n_games):
        o = po.Oracle6Game(rules)
        o.new_game(SEED, g, 0)
        for ply in range(plies):
            if o.status() != -1:
                break
            if ply % every == 0:
                out.append((g, ply, o.image()))
            assert o.move(o.random_action(SEED, g, ply), SEED, g, ply) == 0
    return out


def lockstep_raw(tree, game_obj, seed, game, ply, K):
    return tree.search_rc(game_obj, seed, game, ply, K)


@pytest.mark.parametrize("sims", [16, 40])
def test_k1_equals_r6_mcts_search(sims):
    rules = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    pos = positions(rules)
    assert len(pos) >= 200
    a_tree, b_tree = po.Oracle6Mcts(rules), Lockstep6Mcts(rules)
    o = po.Oracle6Game(rules)
    for g, ply, img in pos:
        o.set_image(img)
        a = a_tree.search(o, SEED, g, ply)
        rc, b = lockstep_raw(b_tree, o, SEED, g, ply, 1)
        assert rc == 0
        for k in ("N", "Q", "P", "pi"):
            assert (bits(a[k]) == bits(b[k])).all(), (g, ply, k)
        assert a["sumN"] == b["sumN"] and np.float32(a["value"]) == np.float32(b["value"])
        assert a_tree.table_size() == b_tree.table_size(), (g, ply)
        for sample in (0, 1):    # both pick modes choose the same move from the same pi
            assert a_tree.pick(a["pi"], sample, SEED, g, ply) == b_tree.pick(b["pi"], sample, SEED, g, ply)
        assert b_tree.active_total() == 0
    assert b_tree.vl_counts() == (0, 0)


@pytest.mark.parametrize("K", [2, 4, 8, 16])
def test_k_descents_invariants(K):
    sims = 32
    rules = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    tree = Lockstep6Mcts(rules)
    o = po.Oracle6Game(rules)
    skipped = 0
    for g, ply, img in positions(rules, n_games=6, every=13):
        o.set_image(img)
        before = tree.vl_counts()[0]
        a = tree.search(o, SEED, g, ply, lockstep=K)
        assert a["sumN"] == sims and int(a["N"].sum()) == sims, (g, ply)
        assert tree.active_total() == 0, (g, ply)
        assert 1 <= tree.table_size() <= sims + 1
        assert abs(float(a["pi"].sum()) - 1.0) < 1e-5
        skipped += tree.vl_counts()[0] > before
    assert skipped > 0, "the active_N rule never passed a move over"


@pytest.mark.parametrize("K,sims", [(3, 16), (5, 32), (32, 16)])
def test_non_dividing_k_rejected(K, sims):
    rules = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    tree = Lockstep6Mcts(rules)
    o = po.Oracle6Game(rules)
    o.new_game(SEED, 0, 0)
    rc, _ = lockstep_raw(tree, o, SEED, 0, 0, K)
    assert rc != 0
