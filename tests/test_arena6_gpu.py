"""GPU suite of the six-player ARENA (az_arena6_*, SIXPLAYER.md §4).  Every match game is replayed on the oracle
(oracle/risk6_oracle.c through Oracle6Game / Oracle6Mcts) by the arena's semantics: deal of game id g - g % 6 (rotation) or g, seat
s played by seat_agent[(s + r) % 6], all randomness keyed by (seed, g, ply), searchers play argmax with their table cleared per
search, the random player is az_env6_rollout's rule.  Per-game status and plies are compared exactly, the tallies must add up."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
SEED = 0x5EED0006
EVAL_CB = C.CFUNCTYPE(None, C.POINTER(po.R6State), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p)


@pytest.fixture(scope="module")
def api():
    from alphazero_risk_b200 import api as a
    if a.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    return a


@EVAL_CB
def uniform_eval(sp, policy, value, user):
    p = float(np.float32(1.0) / np.float32(43.0))
    for i in range(43):
        policy[i] = p
    value[0] = 0.0


def net_eval(net, precision):
    """the oracle search's evaluator: the same CUDA forward at batch 1"""
    L = po.oracle_lib()
    L.r6_encode.argtypes = [C.POINTER(po.R6State), np.ctypeslib.ndpointer(np.float32, flags="C")]

    @EVAL_CB
    def fn(sp, policy, value, user):
        x = np.zeros(po.INPUT_FLOATS, np.float32)
        L.r6_encode(sp, x)
        p, v = net.forward(x.reshape(1, -1), precision)
        C.memmove(policy, p.ctypes.data, 43 * 4)
        value[0] = float(v[0])
    return fn


def replay(trees, seat_agent, rotate, first, n_games, rules_o):
    """the match on the oracle: trees[a] = Oracle6Mcts of searcher a or None (random player)"""
    status, plies, moves, win, win_seat = [], [], [0] * 6, [0] * 6, [0] * 6
    o = po.Oracle6Game(rules_o)
    for g in range(first, first + n_games):
        r = g % 6 if rotate else 0
        o.new_game(SEED, g - r, 0)
        ply = 0
        while o.status() == -1:
            agent = seat_agent[(o.s.cur + r) % 6]
            if trees[agent] is None:
                a = o.random_action(SEED, g, ply)
            else:
                a = trees[agent].pick(trees[agent].search(o, SEED, g, ply)["pi"], False, SEED, g, ply)
            assert o.move(a, SEED, g, ply) == 0
            ply += 1
            moves[agent] += 1
        st = o.status()
        status.append(st)
        plies.append(ply)
        if st >= 0:
            win[seat_agent[(st + r) % 6]] += 1
            win_seat[st] += 1
    return dict(status=np.array(status, np.int8), plies=np.array(plies, np.uint32), moves=moves, win=win, win_seat=win_seat)


def check_match(res, ref, n_games):
    assert (res["status"] == ref["status"]).all(), np.nonzero(res["status"] != ref["status"])
    assert (res["plies"] == ref["plies"]).all(), np.nonzero(res["plies"] != ref["plies"])
    assert res["count"] == n_games
    assert res["draw"] == int((ref["status"] == -2).sum())
    assert res["win"] == ref["win"] and res["win_seat"] == ref["win_seat"]
    assert res["draw"] + sum(res["win"]) == res["count"] and sum(res["win_seat"]) == sum(res["win"])
    assert res["moves"] == ref["moves"] and sum(res["moves"]) == int(res["plies"].sum())
    assert res["errors"] == 0


@pytest.mark.parametrize("rotate,first", [(True, 120), (False, 61)])
def test_random_players_match_oracle(api, rotate, first):
    n_games = 60
    env = api.Env6(7)
    ar = api.Arena6(env, [None, None, None], [0, 1, 2, 0, 1, 2], rotate_seats=rotate)
    res = ar.play(n_games, SEED, first_game=first)
    ref = replay([None, None, None], [0, 1, 2, 0, 1, 2], rotate, first, n_games, po.default_rules())
    check_match(res, ref, n_games)
    assert res["sims"] == 0 and res["evals"] == 0
    assert len(set(res["plies"].tolist())) > 1 and res["ticks"] == len(ar.active_slots())
    ar.close(); env.close()


@pytest.mark.parametrize("kinds,seat_agent", [(("pseudo", "uniform", None), (0, 1, 2, 0, 1, 2)),
                                              (("pseudo", "uniform"), (0, 1, 1, 1, 1, 1)),
                                              (("uniform", None), (0, 1, 1, 1, 1, 1))])
def test_searchers_and_random_player_match_oracle(api, kinds, seat_agent):
    sims, n_games, kw = 8, 12, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(5, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw))
    ev = {"pseudo": api.EVAL_PSEUDO, "uniform": api.EVAL_UNIFORM}
    agents = [api.Mcts6(env, evaluator=ev[k]) if k else None for k in kinds]
    trees = [None if k is None else po.Oracle6Mcts(rules_o, uniform_eval if k == "uniform" else None) for k in kinds]
    ar = api.Arena6(env, agents, seat_agent)
    res = ar.play(n_games, SEED, first_game=6)
    ref = replay(trees, seat_agent, True, 6, n_games, rules_o)
    check_match(res, ref, n_games)
    searched = sum(m for m, k in zip(res["moves"], kinds) if k)
    assert searched > 0 and res["sims"] == searched * sims
    ar.close()
    for a in agents:
        if a is not None:
            a.close()
    env.close()


def test_two_networks_match_oracle_and_lift_selection(api):
    """fp32 and bf16 networks of different weights: the compacted leaf batches of each searcher hold only its waiting slots, and
    as games of different lengths end and new ones are claimed the batches shrink and change composition"""
    sims, n_games, kw = 4, 6, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(4, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw))
    na, nb = api.Net(blocks=1, seed=11), api.Net(blocks=1, seed=12)
    ma = api.Mcts6(env, net=na, evaluator=api.EVAL_NN, precision=api.FP32)
    mb = api.Mcts6(env, net=nb, evaluator=api.EVAL_NN, precision=api.BF16)
    seat_agent = (0, 1, 1, 1, 1, 1)
    ar = api.Arena6(env, [ma, mb], seat_agent)
    res = ar.play(n_games, SEED, first_game=0)
    fa, fb = net_eval(na, api.FP32), net_eval(nb, api.BF16)
    ref = replay([po.Oracle6Mcts(rules_o, fa), po.Oracle6Mcts(rules_o, fb)], seat_agent, True, 0, n_games, rules_o)
    check_match(res, ref, n_games)
    assert res["sims"] == sum(res["moves"]) * sims
    assert len(set(res["plies"].tolist())) > 1
    active = ar.active_slots()
    assert active.max() == 4 and active.min() < 4 and res["ticks"] == len(active)
    # afterwards the handles search every game again, with their own game ids and full leaf batches
    env.reset(SEED + 1)
    env.rollout(300)
    fresh = api.Mcts6(env, net=nb, evaluator=api.EVAL_NN, precision=api.BF16)
    got, want = mb.search(), fresh.search()
    for k in ("N", "pi", "move", "status"):
        assert (np.asarray(got[k]).view(np.uint8) == np.asarray(want[k]).view(np.uint8)).all(), k
    ar.close(); fresh.close(); ma.close(); mb.close(); na.close(); nb.close(); env.close()


def test_after_a_match(api):
    """a pseudo searcher searches stand-alone exactly like a fresh handle after a match; a second play on the arena repeats the first"""
    sims, kw = 8, dict(max_game_rounds=20)
    rules = api.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(5, rules=rules, first_game_id=40)
    mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    ar = api.Arena6(env, [mc, None], (0, 1, 0, 1, 0, 1))
    r1 = ar.play(6, SEED)
    r2 = ar.play(6, SEED)
    for k in ("count", "draw", "win", "win_seat", "moves", "sims", "evals", "ticks", "errors"):
        assert r1[k] == r2[k], k
    assert (r1["status"] == r2["status"]).all() and (r1["plies"] == r2["plies"]).all()
    env.reset(SEED + 2)
    env.rollout(500)
    fresh = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    got, want = mc.search(), fresh.search()
    for k in ("N", "pi", "move", "status"):
        assert (np.asarray(got[k]).view(np.uint8) == np.asarray(want[k]).view(np.uint8)).all(), k
    ar.close(); fresh.close(); mc.close(); env.close()


def test_invariance_at_full_size(api):
    """configs[3]'s 16384 slots: a game's result depends only on (seed, g, agents) — not on the run, the slot, the env's size or a
    split of the match into first_game ranges"""
    sims, n_games, kw = 2, 16380, dict(max_game_rounds=20)
    rules = api.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    na, nb = api.Net(blocks=1, seed=21), api.Net(blocks=1, seed=22)
    seat_agent = (0, 1, 2, 0, 1, 2)

    def run(slots, parts):
        env = api.Env6(slots, rules=rules)
        ma = api.Mcts6(env, net=na, evaluator=api.EVAL_NN, precision=api.BF16)
        mb = api.Mcts6(env, net=nb, evaluator=api.EVAL_NN, precision=api.BF16)
        ar = api.Arena6(env, [ma, mb, None], seat_agent)
        out = [ar.play(count, SEED, first_game=first) for first, count in parts]
        ar.close(); ma.close(); mb.close(); env.close()
        return out

    (a,), (b,) = run(16384, [(0, n_games)]), run(16384, [(0, n_games)])
    assert a["count"] == n_games and a["errors"] == 0 and a["sims"] == (a["moves"][0] + a["moves"][1]) * sims
    for k in ("count", "draw", "win", "win_seat", "moves", "sims", "evals", "ticks"):
        assert a[k] == b[k], k
    assert (a["status"] == b["status"]).all() and (a["plies"] == b["plies"]).all()
    lo, hi = run(8192, [(0, 8190)])[0], run(8192, [(8190, 8190)])[0]
    assert (np.concatenate([lo["status"], hi["status"]]) == a["status"]).all()
    assert (np.concatenate([lo["plies"], hi["plies"]]) == a["plies"]).all()
    for k in ("win", "win_seat", "moves"):
        assert [x + y for x, y in zip(lo[k], hi[k])] == a[k], k
    (c,) = run(5000, [(0, n_games)])
    assert (c["status"] == a["status"]).all() and (c["plies"] == a["plies"]).all()
    assert c["win"] == a["win"] and c["moves"] == a["moves"] and c["ticks"] > a["ticks"]
    na.close(); nb.close()


def test_rejections(api):
    rules = api.default_rules(mcts_simulations=4, threads_per_mcts=1, max_game_rounds=20)
    env, other = api.Env6(6, rules=rules), api.Env6(6, rules=rules)
    mc, mc_other = api.Mcts6(env, evaluator=api.EVAL_PSEUDO), api.Mcts6(other, evaluator=api.EVAL_PSEUDO)
    for agents, seats in (([mc_other], [0] * 6),                 # a handle over another env
                          ([mc, mc], [0, 1, 0, 1, 0, 1]),        # the same handle twice
                          ([], [0] * 6),                         # n_agents outside 1..6
                          ([None] * 7, [0, 1, 2, 3, 4, 5]),
                          ([mc, None], [0, 1, 2, 0, 1, 0]),      # a seat_agent entry out of range
                          ([mc, None], [0] * 6)):                # an agent with no seat
        with pytest.raises(api.AzError):
            api.Arena6(env, agents, seats)
    ar = api.Arena6(env, [None, None], [0, 1, 0, 1, 0, 1])
    for n_games, first in ((7, 0), (6, 3)):                      # rotation: whole groups of six
        with pytest.raises(api.AzError):
            ar.play(n_games, SEED, first_game=first)
    with pytest.raises(api.AzError):                             # first_game + n_games > 2^32
        ar.play(6, SEED, first_game=2 ** 32 - 4)
    flat = api.Arena6(env, [None, None], [0, 1, 0, 1, 0, 1], rotate_seats=False)
    with pytest.raises(api.AzError):
        flat.play(2, SEED, first_game=2 ** 32 - 1)
    last = flat.play(1, SEED, first_game=2 ** 32 - 1)            # the last game id is playable
    assert last["count"] == 1 and last["plies"][0] > 0
    rec = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    rec.record(1000, 64)
    ar_rec = api.Arena6(env, [rec, None], [0, 1, 0, 1, 0, 1])   # recording is checked when the match starts
    with pytest.raises(api.AzError):
        ar_rec.play(6, SEED)
    for h in (ar_rec, flat, ar, rec, mc, mc_other, env, other):
        h.close()
