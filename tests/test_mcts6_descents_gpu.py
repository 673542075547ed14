"""GPU suite of the six-player search with several descents per tree (az_rules.concurrent_descents = K on an Env6, SIXPLAYER.md §2).
The checker is the oracle's lockstep search (oracle/risk6_lockstep.c, Lockstep6Mcts.search(lockstep=K)): visit counts, Q, P, pi, table sizes, chosen
moves and env images are compared as bit patterns, with the oracle's own evaluators or, for the network path, the same CUDA forward at
batch 1.  Arena matches are replayed game by game on the oracle, self-play records against oracle/samples6.py."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as po
from oracle.lockstep6 import Lockstep6Mcts
from oracle.samples6 import SAMPLE6_BYTES, sample_record

pytestmark = pytest.mark.gpu
SEED = 0x5EED0007
EVAL_CB = C.CFUNCTYPE(None, C.POINTER(po.R6State), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p)


@pytest.fixture(scope="module")
def api():
    from alphazero_risk_b200 import api as a
    if a.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    return a


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


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


def run_descents(api, K, n, first, sims, play_mode, max_moves, rules_kw=None, net=None, precision=None, evaluator=None,
                 start_rollout=0):
    """device search with K descents per tree against the oracle's lockstep search, move by move; returns (moves, skips, duplicates)"""
    rules_kw = rules_kw or {}
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **rules_kw)
    env = api.Env6(n, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K, **rules_kw),
                   first_game_id=first)
    env.reset(SEED)
    if start_rollout:
        env.rollout(start_rollout)
    if net is not None:
        eval_fn, ev = net_eval(net, precision), api.EVAL_NN
    elif evaluator == "uniform":
        eval_fn, ev = uniform_eval, api.EVAL_UNIFORM
    else:
        eval_fn, ev = None, api.EVAL_PSEUDO
    mc = api.Mcts6(env, net=net, evaluator=ev, precision=api.FP32 if precision is None else precision)
    img = env.export()
    games = [po.Oracle6Game(rules_o) for _ in range(n)]
    trees = [Lockstep6Mcts(rules_o, eval_fn) for _ in range(n)]
    for g, o in enumerate(games):
        o.set_image(img[g])
    ply = np.full(n, start_rollout, int)
    moves_done = 0
    for step in range(max_moves):
        res = mc.search(pick_mode=api.PICK_ARGMAX if play_mode else api.PICK_SELFPLAY, apply_move=True)
        rs = mc.root_stats()
        for g, o in enumerate(games):
            if o.status() != -1:
                assert res["move"][g] == 43 and res["status"][g] == o.status()
                continue
            a = trees[g].search(o, SEED, first + g, int(ply[g]), lockstep=K)
            assert (res["N"][g] == a["N"]).all(), (step, g, res["N"][g], a["N"])
            assert (bits(rs["Q"][g]) == bits(a["Q"])).all(), (step, g)
            assert (bits(rs["P"][g]) == bits(a["P"])).all(), (step, g)
            assert (bits(res["pi"][g]) == bits(a["pi"])).all(), (step, g)
            assert rs["sumN"][g] == a["sumN"] == sims and rs["table"][g] == trees[g].table_size(), (step, g)
            assert trees[g].active_total() == 0
            sample = (not play_mode) and o.s.round <= rules_o.temperature_threshold
            mv = trees[g].pick(a["pi"], sample, SEED, first + g, int(ply[g]))
            assert res["move"][g] == mv, (step, g)
            assert o.move(mv, SEED, first + g, int(ply[g])) == 0
            ply[g] += 1
            moves_done += 1
            assert res["status"][g] == o.status()
        if step % 16 == 0 or step == max_moves - 1:
            dev = env.export()
            for g, o in enumerate(games):
                assert (dev[g] == o.image()).all(), (step, g)
    cnt = mc.counters()
    assert cnt["errors"] == 0 and cnt["sims"] == moves_done * sims and cnt["steps"] == moves_done
    mc.close(); env.close()
    vl = [t.vl_counts() for t in trees]
    return moves_done, sum(s for s, _ in vl), sum(d for _, d in vl)


@pytest.mark.parametrize("K,sims,play_mode,start,kw", [
    (2, 16, False, 0, {}),
    (4, 32, True, 600, {}),
    (8, 64, False, 900, {}),
    (16, 48, True, 0, {}),
    (4, 20, False, 800, dict(cpuct=2.5, dir_noise_epsi=0.5, dir_noise_value=0.05, temperature_threshold=20, limit_attack=1,
                             limit_reinforcement=0, min_unit_move=1, allow_yield=0, max_game_rounds=40)),
])
def test_descents_pseudo_vs_oracle(api, K, sims, play_mode, start, kw):
    moves, skips, dups = run_descents(api, K, n=6, first=50 + K, sims=sims, play_mode=play_mode, max_moves=40, rules_kw=kw,
                                      start_rollout=start)
    assert moves > 100 and skips > 0
    if K == 16:    # set-up from the deal: 7 legal moves and 16 descents in the first round, so the rule must request one again
        assert dups > 0


def test_descents_uniform_evaluator(api):
    moves, skips, _ = run_descents(api, 8, n=5, first=7, sims=32, play_mode=False, max_moves=30, evaluator="uniform", start_rollout=400)
    assert moves > 60 and skips > 0


@pytest.mark.parametrize("blocks,prec", [(1, "fp32"), (2, "bf16")])
def test_descents_network_matches_oracle_given_same_outputs(api, blocks, prec):
    net = api.Net(blocks=blocks, seed=4321 + blocks)
    moves, skips, _ = run_descents(api, 4, n=4, first=70, sims=12, play_mode=False, max_moves=24, net=net,
                                   precision=api.FP32 if prec == "fp32" else api.BF16, start_rollout=700)
    assert moves > 50 and skips > 0
    net.close()


def test_descents_full_size_self_play(api):
    """16384 games, K = 4, a 1-block bf16 network: counters add up, the run is reproducible, a half-size shard with the second half's
    game ids reproduces the second half"""
    n, sims, moves, K = 16384, 8, 3, 4
    net = api.Net(blocks=1, seed=5)
    rules = api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K)

    def run(count, first):
        env = api.Env6(count, rules=rules, first_game_id=first)
        env.reset(SEED)
        mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
        mc.selfplay(moves)
        cnt, img = mc.counters(), env.export().copy()
        mc.close(); env.close()
        return cnt, img

    cnt, img = run(n, 0)
    assert cnt["errors"] == 0 and cnt["sims"] == n * sims * moves and cnt["steps"] == n * moves and cnt["evals"] >= n * moves
    cnt2, img2 = run(n, 0)
    assert cnt2 == cnt and (img2 == img).all()
    _, half = run(n // 2, n // 2)
    assert (half == img[n // 2:]).all()
    net.close()


# ------------------------------------------------------------------ arena
def replay(trees, seat_agent, rotate, first, n_games, rules_o, K):
    """the match on the oracle: trees[a] = Lockstep6Mcts of searcher a (lockstep search with K descents) or None (random player)"""
    status, plies = [], []
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
                a = trees[agent].pick(trees[agent].search(o, SEED, g, ply, lockstep=K)["pi"], False, SEED, g, ply)
            assert o.move(a, SEED, g, ply) == 0
            ply += 1
        status.append(o.status())
        plies.append(ply)
    return np.array(status, np.int8), np.array(plies, np.uint32)


@pytest.mark.parametrize("K", [2, 4])
def test_arena_searchers_and_random_player_match_oracle(api, K):
    sims, n_games, kw = 8, 12, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(5, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K, **kw))
    agents = [api.Mcts6(env, evaluator=api.EVAL_PSEUDO), api.Mcts6(env, evaluator=api.EVAL_UNIFORM), None]
    trees = [Lockstep6Mcts(rules_o), Lockstep6Mcts(rules_o, uniform_eval), None]
    seat_agent = (0, 1, 2, 0, 1, 2)
    ar = api.Arena6(env, agents, seat_agent)
    res = ar.play(n_games, SEED, first_game=6)
    status, plies = replay(trees, seat_agent, True, 6, n_games, rules_o, K)
    assert (res["status"] == status).all() and (res["plies"] == plies).all()
    assert res["errors"] == 0 and res["sims"] == (res["moves"][0] + res["moves"][1]) * sims
    ar.close()
    for a in agents:
        if a is not None:
            a.close()
    env.close()


@pytest.mark.parametrize("K", [2, 4])
def test_arena_two_networks_match_oracle(api, K):
    """compacted leaf batches of K * count positions, position j * count + k = descent slot j * n + games[k]"""
    sims, n_games, kw = 4, 6, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(4, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K, **kw))
    na, nb = api.Net(blocks=1, seed=11), api.Net(blocks=1, seed=12)
    ma = api.Mcts6(env, net=na, evaluator=api.EVAL_NN, precision=api.FP32)
    mb = api.Mcts6(env, net=nb, evaluator=api.EVAL_NN, precision=api.BF16)
    seat_agent = (0, 1, 1, 1, 1, 1)
    ar = api.Arena6(env, [ma, mb], seat_agent)
    res = ar.play(n_games, SEED, first_game=0)
    trees = [Lockstep6Mcts(rules_o, net_eval(na, api.FP32)), Lockstep6Mcts(rules_o, net_eval(nb, api.BF16))]
    status, plies = replay(trees, seat_agent, True, 0, n_games, rules_o, K)
    assert (res["status"] == status).all() and (res["plies"] == plies).all()
    assert res["errors"] == 0 and res["sims"] == sum(res["moves"]) * sims
    active = ar.active_slots()
    assert active.max() == 4 and active.min() < 4
    ar.close(); ma.close(); mb.close(); na.close(); nb.close(); env.close()


def test_arena_16384_slots_invariance(api):
    """K = 4 at 16384 slots: two runs agree, and a split of the games over two envs gives the same per-game results"""
    sims, K, n_games, kw = 4, 4, 16380, dict(max_game_rounds=12)
    rules = api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K, **kw)
    net = api.Net(blocks=1, seed=21)

    def play(slots, first, count):
        env = api.Env6(slots, rules=rules)
        mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.BF16)
        ar = api.Arena6(env, [mc, None], (0, 1, 1, 1, 1, 1))
        res = ar.play(count, SEED, first_game=first)
        ar.close(); mc.close(); env.close()
        return res

    a, b = play(16384, 0, n_games), play(16384, 0, n_games)
    assert (a["status"] == b["status"]).all() and (a["plies"] == b["plies"]).all() and a["ticks"] == b["ticks"]
    assert a["errors"] == 0 and a["sims"] == a["moves"][0] * sims
    half = n_games // 2
    lo, hi = play(8192, 0, half), play(8192, half, n_games - half)
    assert (np.concatenate([lo["status"], hi["status"]]) == a["status"]).all()
    assert (np.concatenate([lo["plies"], hi["plies"]]) == a["plies"]).all()
    net.close()


# ------------------------------------------------------------------ recording
def test_recording_with_descents(api):
    """K = 4: recording changes nothing the search computes, and the records are oracle/samples6.py's records of the oracle's self-play
    with the lockstep search (finished games re-dealt, as az_selfplay6_run does)"""
    n, first, sims, K, moves = 8, 40, 8, 4, 1000
    kw = dict(mcts_simulations=sims, threads_per_mcts=1, max_game_rounds=20)

    def run(record):
        env = api.Env6(n, rules=api.default_rules(concurrent_descents=K, **kw), first_game_id=first)
        env.reset(SEED)
        mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
        if record:
            mc.record(capacity_samples=n * moves, max_moves_per_game=2048)
        mc.selfplay(moves)
        res, rs = mc.search(pick_mode=api.PICK_SELFPLAY), mc.root_stats()
        recs = mc.samples()[0] if record else None
        cnt, img = mc.counters(), env.export().copy()
        mc.close(); env.close()
        return (res, rs), cnt, img, recs

    (o0, c0, i0, _), (o1, c1, i1, recs) = run(False), run(True)
    assert c0 == c1 and c0["games"] > 0 and c0["errors"] == 0 and (i0 == i1).all()
    for d0, d1 in zip(o0, o1):
        for k in d0:
            assert (np.ascontiguousarray(d0[k]).view(np.uint8) == np.ascontiguousarray(d1[k]).view(np.uint8)).all(), k
    rules = po.default_rules(**kw)
    expected = []
    for g in range(n):
        o, t = po.Oracle6Game(rules), Lockstep6Mcts(rules)
        o.new_game(SEED, first + g, 0)
        cur = []
        for ply in range(moves):
            a = t.search(o, SEED, first + g, ply, lockstep=K)
            cur.append((o.image(), a["pi"].copy()))
            mv = t.pick(a["pi"], o.s.round <= rules.temperature_threshold, SEED, first + g, ply)
            assert o.move(mv, SEED, first + g, ply) == 0
            st = o.status()
            if st != -1:
                expected.append(np.stack([sample_record(img, pi, st) for img, pi in cur]).tobytes())
                cur = []
                o.new_game(SEED, first + g, ply + 1)
    assert len(expected) >= n // 2 and recs.shape[1] == SAMPLE6_BYTES
    assert sum(len(e) for e in expected) == recs.size
    blob, pos = recs.tobytes(), 0
    left = sorted(expected, key=len, reverse=True)
    while pos < len(blob):
        hit = [e for e in left if blob.startswith(e, pos)]
        assert hit, "record stream at byte %d matches no expected game" % pos
        left.remove(hit[0]); pos += len(hit[0])
    assert not left


# ------------------------------------------------------------------ rejections
@pytest.mark.parametrize("K", [3, 17])
def test_invalid_descents_rejected(api, K):
    env = api.Env6(4, rules=api.default_rules(mcts_simulations=16, threads_per_mcts=1, concurrent_descents=K))
    with pytest.raises(api.AzError):
        api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    env.close()
