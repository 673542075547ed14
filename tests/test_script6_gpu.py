"""GPU suite of the six-player scripted agent (SIXPLAYER.md §5): az_env6_script_actions against the oracle (oracle/risk6_script.c)
bit for bit on rollout positions under every rule set and on hand-built positions, and arena matches with scripted agents replayed on
the oracle by the arena's semantics (test_arena6_gpu.py's replay with a script branch): per-game status and plies, tallies and moves
compared exactly."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as po
from oracle import script6 as s6
from oracle.lockstep6 import Lockstep6Mcts

pytestmark = pytest.mark.gpu
SEED = 0x5EED0006
SCRIPT = "script"
RULE_SETS = [dict(), dict(limit_attack=1), dict(limit_reinforcement=0), dict(allow_yield=0, max_game_rounds=30), dict(min_unit_move=1)]
RULE_IDS = ["default", "limit_attack", "no_limit_reinf", "no_yield_30_rounds", "min_unit_move_1"]
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


def oracle_actions(images, rules):
    o = po.Oracle6Game(rules)
    out = np.empty(len(images), np.uint8)
    for i, img in enumerate(images):
        o.set_image(img)
        out[i] = 0xff if o.status() != -1 else s6.script_action(o)
    return out


@pytest.mark.parametrize("kw", RULE_SETS, ids=RULE_IDS)
def test_script_actions_match_oracle_on_rollouts(api, kw):
    """2048 games exported at five points of a random rollout (set-up, early turns, eliminations, late game): 10240 positions"""
    n = 2048
    env = api.Env6(n, rules=api.default_rules(**kw), first_game_id=900)
    env.reset(SEED)
    rules_o = po.default_rules(**kw)
    checked, phases = 0, set()
    for steps in (0, 40, 300, 1200, 2500):
        env.rollout(steps)
        img, got = env.export(), env.script_actions()
        want = oracle_actions(img, rules_o)
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, (steps, bad[:5], got[bad[:5]], want[bad[:5]])
        valid, status = env.query()
        run = status == -1
        assert ((valid[run] >> got[run].astype(np.uint64)) & np.uint64(1)).all()
        checked += n
        phases |= set(img[:, 101].tolist())
    assert checked >= 10000 and phases == {0, 2, 3, 4, 5}
    env.close()


def test_script_actions_on_hand_built_and_finished_positions(api):
    """the hand-built positions of oracle/script6.py imported into an env of their rules; a finished game answers 0xff, and the
    host-driven scripted game (script_actions + step) stays on the oracle's trajectory"""
    by_rules = {}
    for name, kw, rules_kw, want in s6.HAND_CASES:
        by_rules.setdefault(tuple(sorted(rules_kw.items())), []).append((name, s6.position(**kw).image(), want))
    won = s6.position(own=set(range(42))).image()                # seat 0 owns every land: the game is over
    for rules_kw, cases in by_rules.items():
        env = api.Env6(len(cases) + 1, rules=api.default_rules(**dict(rules_kw)))
        env.import_images(np.stack([img for _, img, _ in cases] + [won]))
        got = env.script_actions()
        for (name, _, want), a in zip(cases, got):
            assert a == want, (name, a)
        assert got[-1] == 0xff
        env.close()
    n, first = 16, 40
    env = api.Env6(n, first_game_id=first)
    env.reset(SEED)
    games = [po.Oracle6Game() for _ in range(n)]
    for g, o in enumerate(games):
        o.new_game(SEED, first + g, 0)
    for ply in range(400):
        act = env.script_actions()
        assert (act == oracle_actions(np.stack([o.image() for o in games]), po.default_rules())).all(), ply
        st = env.step(act)
        for g, o in enumerate(games):
            if act[g] != 0xff:
                assert o.move(int(act[g]), SEED, first + g, ply) == 0
        assert (env.export() == np.stack([o.image() for o in games])).all(), ply
        assert (st[act != 0xff] == np.array([o.status() for o in games], np.int8)[act != 0xff]).all()
    env.close()


class _Tree:
    """an oracle searcher: the one-descent search (K = 1) or the lockstep search with K descents"""

    def __init__(self, rules_o, eval_fn, K):
        self.K, self.eval_fn = K, eval_fn                       # the C search calls eval_fn: keep the callback alive
        self.t = po.Oracle6Mcts(rules_o, eval_fn) if K == 1 else Lockstep6Mcts(rules_o, eval_fn)

    def action(self, o, g, ply):
        out = self.t.search(o, SEED, g, ply) if self.K == 1 else self.t.search(o, SEED, g, ply, lockstep=self.K)
        return self.t.pick(out["pi"], False, SEED, g, ply)


def replay(agents, seat_agent, rotate, first, n_games, rules_o):
    """the match on the oracle: agents[a] = a _Tree (searcher), SCRIPT (the scripted agent) or None (random player)"""
    status, plies, moves, win, win_seat = [], [], [0] * 6, [0] * 6, [0] * 6
    o = po.Oracle6Game(rules_o)
    for g in range(first, first + n_games):
        r = g % 6 if rotate else 0
        o.new_game(SEED, g - r, 0)
        ply = 0
        while o.status() == -1:
            agent = seat_agent[(o.s.cur + r) % 6]
            if agents[agent] is None:
                a = o.random_action(SEED, g, ply)
            elif agents[agent] is SCRIPT:
                a = s6.script_action(o)
            else:
                a = agents[agent].action(o, g, ply)
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
def test_script_vs_random_matches_oracle(api, rotate, first):
    n_games, seat_agent = 60, [0, 1, 1, 1, 1, 1]
    env = api.Env6(7)
    ar = api.Arena6(env, [api.SCRIPT6, None], seat_agent, rotate_seats=rotate)
    res = ar.play(n_games, SEED, first_game=first)
    ref = replay([SCRIPT, None], seat_agent, rotate, first, n_games, po.default_rules())
    check_match(res, ref, n_games)
    assert res["sims"] == 0 and res["evals"] == 0 and res["win"][0] > res["win"][1]
    ar.close(); env.close()


@pytest.mark.parametrize("K", [1, 2])
@pytest.mark.parametrize("kinds,seat_agent", [(("pseudo", "uniform", SCRIPT), (0, 1, 2, 0, 1, 2)),
                                              (("pseudo", SCRIPT, None), (0, 1, 2, 1, 2, 1))])
def test_script_vs_searchers_matches_oracle(api, kinds, seat_agent, K):
    sims, n_games, kw = 8, 12, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(5, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K, **kw))
    ev = {"pseudo": api.EVAL_PSEUDO, "uniform": api.EVAL_UNIFORM}
    agents = [api.Mcts6(env, evaluator=ev[k]) if k in ev else api.SCRIPT6 if k is SCRIPT else None for k in kinds]
    trees = [_Tree(rules_o, uniform_eval if k == "uniform" else None, K) if k in ev else k for k in kinds]
    ar = api.Arena6(env, agents, seat_agent)
    res = ar.play(n_games, SEED, first_game=6)
    ref = replay(trees, seat_agent, True, 6, n_games, rules_o)
    check_match(res, ref, n_games)
    searched = sum(m for m, k in zip(res["moves"], kinds) if k in ev)
    assert searched > 0 and res["sims"] == searched * sims
    assert res["moves"][kinds.index(SCRIPT)] > 0
    ar.close()
    for a in agents:
        if isinstance(a, api.Mcts6):
            a.close()
    env.close()


def test_script_vs_network_searcher_matches_oracle(api):
    sims, n_games, kw = 4, 6, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(4, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw))
    net = api.Net(blocks=1, seed=31)
    mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.FP32)
    seat_agent = (0, 1, 1, 1, 1, 1)
    ar = api.Arena6(env, [mc, api.SCRIPT6], seat_agent)
    res = ar.play(n_games, SEED, first_game=0)
    ref = replay([_Tree(rules_o, net_eval(net, api.FP32), 1), SCRIPT], seat_agent, True, 0, n_games, rules_o)
    check_match(res, ref, n_games)
    assert res["sims"] == res["moves"][0] * sims
    ar.close(); mc.close(); net.close(); env.close()


def test_script_match_invariance_at_full_size(api):
    """16384 slots, 1 script vs 5 random players: a game's result depends only on (seed, g, agents) — not on the run, the env's
    size or a split of the match over two envs"""
    n_games, seat_agent = 16380, (0, 1, 1, 1, 1, 1)

    def run(slots, parts):
        env = api.Env6(slots)
        ar = api.Arena6(env, [api.SCRIPT6, None], seat_agent)
        out = [ar.play(count, SEED, first_game=first) for first, count in parts]
        ar.close(); env.close()
        return out

    (a,), (b,) = run(16384, [(0, n_games)]), run(16384, [(0, n_games)])
    assert a["count"] == n_games and a["errors"] == 0 and a["sims"] == 0
    for k in ("count", "draw", "win", "win_seat", "moves", "ticks"):
        assert a[k] == b[k], k
    assert (a["status"] == b["status"]).all() and (a["plies"] == b["plies"]).all()
    assert a["win"][0] > 0.8 * n_games
    lo, hi = run(8192, [(0, 8190)])[0], run(8192, [(8190, 8190)])[0]
    assert (np.concatenate([lo["status"], hi["status"]]) == a["status"]).all()
    assert (np.concatenate([lo["plies"], hi["plies"]]) == a["plies"]).all()
    for k in ("win", "win_seat", "moves"):
        assert [x + y for x, y in zip(lo[k], hi[k])] == a[k], k
    (c,) = run(5000, [(0, n_games)])
    assert (c["status"] == a["status"]).all() and (c["plies"] == a["plies"]).all()
    assert c["win"] == a["win"] and c["moves"] == a["moves"]


def test_create_agents_rejections_and_create_equivalence(api):
    L = api.lib()
    rules = api.default_rules(mcts_simulations=4, threads_per_mcts=1, max_game_rounds=20)
    env = api.Env6(6, rules=rules)
    mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    seats = np.array([0, 1, 0, 1, 0, 1], np.uint8)

    def create(handles, kinds):
        hs = (C.c_void_p * 2)(*handles)
        ks = np.array(kinds, np.int32)
        h = C.c_void_p()
        rc = L.az_arena6_create_agents(env.h, hs, C.c_void_p(ks.ctypes.data), 2, C.c_void_p(seats.ctypes.data), 1, C.byref(h))
        if rc == 0:
            L.az_arena6_destroy(h)
        return rc

    S, R, X = api.AGENT6_SEARCHER, api.AGENT6_RANDOM, api.AGENT6_SCRIPT
    assert create([mc.h, None], [S, R]) == 0 and create([mc.h, None], [S, X]) == 0 and create([None, None], [X, R]) == 0
    for handles, kinds in (([None, None], [S, R]),               # a searcher without a handle
                           ([mc.h, mc.h], [S, X]),               # a handle for the scripted agent
                           ([mc.h, mc.h], [S, R]),               # a handle for the random player
                           ([None, None], [3, R]),               # unknown kinds
                           ([None, None], [R, -1]),
                           ([mc.h, None], [S, 255])):
        assert create(handles, kinds) != 0, (handles, kinds)
    h = C.c_void_p()
    assert L.az_arena6_create_agents(env.h, (C.c_void_p * 1)(None), None, 1, C.c_void_p(seats.ctypes.data), 1, C.byref(h)) != 0
    # az_arena6_create derives the kinds from the handles: the same match as the kinds spelled out
    h = C.c_void_p()
    assert L.az_arena6_create(env.h, (C.c_void_p * 2)(mc.h, None), 2, C.c_void_p(seats.ctypes.data), 1, C.byref(h)) == 0
    r1 = api.AzArena6Results()
    st1, pl1 = np.empty(6, np.int8), np.empty(6, np.uint32)
    assert L.az_arena6_play(h, 0, 6, SEED, C.byref(r1), C.c_void_p(st1.ctypes.data), C.c_void_p(pl1.ctypes.data), None) == 0
    L.az_arena6_destroy(h)
    ar = api.Arena6(env, [mc, None], seats)
    r2 = ar.play(6, SEED)
    assert r1.as_dict() == {k: v for k, v in r2.items() if k not in ("status", "plies")}
    assert (st1 == r2["status"]).all() and (pl1 == r2["plies"]).all()
    ar.close(); mc.close(); env.close()


def test_searcher_after_a_match_with_scripts(api):
    """a pseudo searcher searches stand-alone exactly like a fresh handle after a match against scripts; a second play repeats the
    first"""
    sims, kw = 8, dict(max_game_rounds=20)
    env = api.Env6(5, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw), first_game_id=40)
    mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    ar = api.Arena6(env, [mc, api.SCRIPT6], (0, 1, 1, 1, 1, 1))
    r1, r2 = ar.play(12, SEED), ar.play(12, SEED)
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
