"""GPU suite of the six-seat value vector (SIXPLAYER.md §2): a network with six value outputs (az_nn_create_value), its training on
[n][6] targets and on six-player records, and the six-player search's per-seat backup.  Checkers: oracle/nn_oracle.py (forward, fp64
Trainer; a dense_2/kernel of shape [256, 6] gives the value as [n * 6] and the mean squared error over all n * 6 elements) and
oracle/risk6_vector.c (Vector6Mcts): visit counts, Q, P, pi, table sizes, chosen moves and env images are compared as bit patterns, with
the pseudo6 evaluator or, for the network path, the same CUDA forward at batch 1.  Arena matches are replayed game by game on the
oracles, self-play records against oracle/samples6.py."""
import ctypes as C

import numpy as np
import pytest

from oracle import nn_oracle as no
from oracle import pyoracle as po
from oracle.lockstep6 import Lockstep6Mcts
from oracle.samples6 import SAMPLE6_BYTES, sample_record
from oracle.vector6 import EVAL6_CB, Vector6Mcts

pytestmark = pytest.mark.gpu
SEED = 0x5EED0066
LOSS = np.float32(-1.0) / np.float32(5.0)
GRAD_TOL, LOSS_TOL = 2e-4, 2e-5                 # tests/test_train_gpu.py
BF16_POLICY_TOL, BF16_VALUE_TOL = 2e-3, 1e-2    # tests/test_nn_gpu.py
EVAL_CB = C.CFUNCTYPE(None, C.POINTER(po.R6State), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p)


@pytest.fixture(scope="module")
def api():
    from alphazero_risk_b200 import api as a
    if a.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    return a


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def perturbed_net(api, blocks, seed, value_outputs=6):
    net = api.Net(blocks=blocks, seed=seed, value_outputs=value_outputs)
    rng = np.random.default_rng(seed)
    for name, shape in net.variables():       # make BN parameters non-trivial
        if name.endswith("/gamma"):
            net.load(name, rng.uniform(0.8, 1.2, shape))
        elif name.endswith("/beta") or name.endswith("/bias"):
            net.load(name, rng.uniform(-0.1, 0.1, shape))
    return net


def env6_inputs(api, n, rollout=300):
    env = api.Env6(n)
    env.reset(SEED)
    env.rollout(rollout)
    x = env.encode()
    env.close()
    return x


def train_data(api, n, seed=0xC0FFEE):
    rng = np.random.default_rng(seed)
    x = env6_inputs(api, n, 200 + seed % 97)
    tp = rng.random((n, 43)).astype(np.float32)
    tp /= tp.sum(1, keepdims=True)
    tv = rng.choice([1.0, float(LOSS), 0.0], (n, 6)).astype(np.float32)
    return x, tp, tv


# ------------------------------------------------------------------ network
def test_inventory_and_glorot(api):
    net = api.Net(blocks=1, seed=3, value_outputs=6)
    shapes = dict(net.variables())
    assert net.value_outputs == 6 and shapes["dense_2/kernel"] == (256, 6) and shapes["dense_2/bias"] == (6,)
    one = dict(api.Net(blocks=1, value_outputs=1).variables())
    assert {k: v for k, v in shapes.items() if not k.startswith("dense_2")} == {k: v for k, v in one.items() if not k.startswith("dense_2")}
    w = net.get("dense_2/kernel", (256, 6))
    lim = np.float32(np.sqrt(np.float32(6.0) / np.float32(262.0)))
    assert np.abs(w).max() <= lim and np.abs(w).max() > 0.9 * lim
    with pytest.raises(api.AzError):
        api.Net(blocks=1, value_outputs=2)
    net.close()


@pytest.mark.parametrize("blocks,n", [(2, 37), (1, 1), (3, 130)])
def test_forward_matches_oracle_and_policy_is_the_one_output_policy(api, blocks, n):
    net6 = perturbed_net(api, blocks, 1234 + n)
    net1 = api.Net(blocks=blocks, value_outputs=1)
    for name, shape in net6.variables():
        if not name.startswith("dense_2"):
            net1.load(name, net6.get(name, shape))
    x = env6_inputs(api, n)
    p32, v32 = net6.forward(x, api.FP32)
    assert v32.shape == (n, 6)
    rp, rv = no.forward(net6.weights(), x, blocks)
    assert np.abs(p32 - rp).max() <= 1e-5 and np.abs(v32.reshape(-1) - rv).max() <= 1e-5
    p16, v16 = net6.forward(x, api.BF16)
    assert np.abs(p32 - p16).max() <= BF16_POLICY_TOL and np.abs(v32 - v16).max() <= BF16_VALUE_TOL
    for prec, pol6 in ((api.FP32, p32), (api.BF16, p16)):
        pol1, val1 = net1.forward(x, prec)
        assert val1.shape == (n,) and (bits(pol1) == bits(pol6)).all()
    p1, v1 = net6.forward(x[:1], api.FP32)                            # batch invariance
    assert (bits(p1[0]) == bits(p32[0])).all() and (bits(v1[0]) == bits(v32[0])).all()
    net6.close(); net1.close()


# ------------------------------------------------------------------ training
@pytest.mark.parametrize("blocks,n", [(2, 16), (1, 5)])
def test_one_step_matches_trainer(api, blocks, n):
    net = perturbed_net(api, blocks, 77)
    ref = no.Trainer(net.weights(), blocks)
    x, tp, tv = train_data(api, n)
    lp, lv = net.train_step(x, tp, tv)
    rp, rv = ref.step(x, tp, tv.reshape(-1))
    assert abs(lp - rp) <= LOSS_TOL * max(1.0, abs(rp)) and abs(lv - rv) <= LOSS_TOL * max(1.0, abs(rv)), (lp, rp, lv, rv)
    shapes = dict(net.variables())
    for name in no.trainable_names(blocks):
        g, gr = net.grad(name, shapes[name]), ref.grads[name].numpy()
        err = np.abs(g - gr).max() / max(np.abs(gr).max(), 1e-12)
        assert err <= GRAD_TOL, (name, err)
    w, wr = net.weights(), ref.weights()
    for name in no.trainable_names(blocks):
        clear = np.abs(ref.grads[name].numpy()) > 1e-6
        assert np.abs(w[name] - wr[name])[clear].max(initial=0.0) <= 2e-5, name
    net.close()


def test_bf16_training_step_close_to_trainer(api):
    blocks, n = 1, 64
    net = perturbed_net(api, blocks, 78)
    net.train_precision(api.BF16)
    ref = no.Trainer(net.weights(), blocks)
    x, tp, tv = train_data(api, n, seed=31)
    lp, lv = net.train_step(x, tp, tv)
    rp, rv = ref.step(x, tp, tv.reshape(-1))
    assert abs(lp - rp) <= 1e-2 * max(1.0, abs(rp)) and abs(lv - rv) <= 1e-2 * max(1.0, abs(rv)), (lp, rp, lv, rv)
    shapes = dict(net.variables())
    for name in no.trainable_names(blocks):
        g = net.grad(name, shapes[name]).ravel().astype(np.float64)
        gx = ref.grads[name].numpy().ravel()
        cos = float(g @ gx / max(np.linalg.norm(g) * np.linalg.norm(gx), 1e-30))
        assert cos >= 0.98 or gx.size <= 64, (name, cos)
    g2 = net.grad("dense_2/kernel", (256, 6)).astype(np.float64).ravel()
    gx2 = ref.grads["dense_2/kernel"].numpy().ravel()
    assert float(g2 @ gx2 / (np.linalg.norm(g2) * np.linalg.norm(gx2))) >= 0.98
    net.close()


def test_several_steps_track_the_trainer(api):
    blocks, n = 2, 24
    net = perturbed_net(api, blocks, 5)
    ref = no.Trainer(net.weights(), blocks)
    x, tp, tv = train_data(api, n, seed=99)
    first = None
    for step in range(4):
        lp, lv = net.train_step(x, tp, tv)
        rp, rv = ref.step(x, tp, tv.reshape(-1))
        assert abs(lp - rp) <= 2e-3 * max(1.0, abs(rp)) and abs(lv - rv) <= 2e-3 * max(1.0, abs(rv)), (step, lp, rp, lv, rv)
        first = first if first is not None else (lp, lv)
    assert lp < first[0] and lv < first[1]
    w, wr = net.weights(), ref.weights()
    for name in w:
        d = np.abs(w[name] - wr[name])
        assert d.max() <= 8.1e-3 and (d.size < 256 or np.median(d) <= 2e-5), (name, np.median(d), d.max())
    p, v = net.forward(x, api.FP32)
    pr, vr = no.forward(w, x, blocks)
    assert np.abs(p - pr).max() <= 1e-5 and np.abs(v.reshape(-1) - vr).max() <= 1e-5
    net.close()


def test_train6_equals_manual_batches(api):
    """az_nn_train6 with six value outputs: target k = the value of seat (cur + k) % 6 under the record's status, built on the
    device; equal, bit for bit, to az_nn_train_step on the same batches with the targets derived on the host"""
    rules = po.default_rules()
    o, enc, rng = po.Oracle6Game(rules), po.Oracle6Mcts(rules), np.random.default_rng(6)
    recs, xs, tps, tvs = [], [], [], []
    g = 0
    while len(recs) < 150:
        o.new_game(0xABCE, g, 0)
        ply = 0
        while o.status() == -1 and len(recs) < 150:
            if ply % 11 == 0:
                valid = o.valid()
                t = np.array([rng.random() if (valid >> i) & 1 else 0.0 for i in range(43)], np.float32)
                t /= t.sum()
                status = int(rng.choice([0, 1, 2, 3, 4, 5, -2]))
                recs.append(sample_record(o.image(), t, status)); xs.append(enc.encode(o)); tps.append(t)
                tvs.append([0.0 if status == -2 else (1.0 if status == (o.s.cur + k) % 6 else LOSS) for k in range(6)])
            o.move(o.random_action(0xABCE, g, ply), 0xABCE, g, ply)
            ply += 1
        g += 1
    recs = np.stack(recs); xs = np.array(xs, np.float32); tps = np.array(tps, np.float32); tvs = np.array(tvs, np.float32)
    assert (bits(recs[:, 108:112].copy().view(np.float32).reshape(-1)) == bits(tvs[:, 0])).all()    # component 0 = the stored float
    epochs, batch, seed = 2, 32, 43
    a, b = perturbed_net(api, 1, 9), perturbed_net(api, 1, 9)
    lp, lv = a.train6(recs, epochs, batch, seed)
    order, st, M = np.arange(len(recs)), seed, (1 << 64) - 1
    for e in range(epochs):
        for i in range(len(recs) - 1, 0, -1):                       # the library's Fisher-Yates on splitmix64
            st = (st + 0x9E3779B97F4A7C15) & M
            z = st; z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M; z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M; z ^= z >> 31
            j = z % (i + 1)
            order[i], order[j] = order[j], order[i]
        losses = []
        for k in range(len(recs) // batch):
            idx = order[k * batch:(k + 1) * batch]
            losses.append(b.train_step(xs[idx], tps[idx], tvs[idx]))
        assert abs(np.mean([l[0] for l in losses]) - lp[e]) < 1e-5 and abs(np.mean([l[1] for l in losses]) - lv[e]) < 1e-5
    wa, wb = a.weights(), b.weights()
    for name in wa:
        assert (bits(wa[name]) == bits(wb[name])).all(), name
    with pytest.raises(api.AzError):                                # two-player records hold one value target
        a.train(np.zeros((64, api.SAMPLE_BYTES), np.uint8), 1, 32, 0)
    a.close(); b.close()


def test_checkpoints_and_cross_width_rejections(api, tmp_path):
    a = perturbed_net(api, 1, 12)
    x, tp, tv = train_data(api, 8, seed=5)
    a.train_step(x, tp, tv)
    a.save_checkpoint(tmp_path / "six")
    b = api.Net(blocks=1, value_outputs=6)
    b.load_checkpoint(tmp_path / "six")
    wa, wb = a.weights(), b.weights()
    for name in wa:
        assert (bits(wa[name]) == bits(wb[name])).all(), name
    assert b.optimizer_powers()[:2] == a.optimizer_powers()[:2]
    for name in ("dense_2/kernel", "dense_2/bias"):
        shape = dict(a.variables())[name]
        for which in (0, 1):
            assert (bits(a.optimizer_slot(name, which, shape)) == bits(b.optimizer_slot(name, which, shape))).all()
    assert (bits(a.forward(x, api.FP32)[1]) == bits(b.forward(x, api.FP32)[1])).all()
    one = api.Net(blocks=1, seed=1, value_outputs=1)
    one.save_checkpoint(tmp_path / "one")
    with pytest.raises(api.AzError):
        b.load_checkpoint(tmp_path / "one")
    with pytest.raises(api.AzError):
        one.load_checkpoint(tmp_path / "six")
    with pytest.raises(api.AzError):
        one.copy_state_from(a)
    with pytest.raises(api.AzError):
        a.copy_state_from(one)
    env = api.Env(4)
    with pytest.raises(api.AzError):
        api.Mcts(env, net=a, evaluator=api.EVAL_NN)
    with pytest.raises(api.AzError):
        api.Mcts(env, evaluator=api.EVAL_PSEUDO6)
    env.close(); a.close(); b.close(); one.close()


# ------------------------------------------------------------------ search
def net_eval6(net, precision):
    """the oracle search's evaluator: the same CUDA forward at batch 1"""
    L = po.oracle_lib()
    L.r6_encode.argtypes = [C.POINTER(po.R6State), np.ctypeslib.ndpointer(np.float32, flags="C")]

    @EVAL6_CB
    def fn(sp, policy, value, user):
        x = np.zeros(po.INPUT_FLOATS, np.float32)
        L.r6_encode(sp, x)
        p, v = net.forward(x.reshape(1, -1), precision)
        C.memmove(policy, p.ctypes.data, 43 * 4)
        C.memmove(value, np.ascontiguousarray(v[0]).ctypes.data, 6 * 4)
    return fn


def net_eval1(net, precision):
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


def run_vector(api, K, n, first, sims, play_mode, max_moves, net=None, precision=None, start_rollout=0):
    """device search with a value vector against Vector6Mcts, move by move; returns the moves made"""
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    env = api.Env6(n, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K), first_game_id=first)
    env.reset(SEED)
    if start_rollout:
        env.rollout(start_rollout)
    if net is not None:
        eval_fn, ev = net_eval6(net, precision), api.EVAL_NN
    else:
        eval_fn, ev = None, api.EVAL_PSEUDO6
    mc = api.Mcts6(env, net=net, evaluator=ev, precision=api.FP32 if precision is None else precision)
    img = env.export()
    games = [po.Oracle6Game(rules_o) for _ in range(n)]
    trees = [Vector6Mcts(rules_o, eval_fn) for _ in range(n)]
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
    return moves_done


@pytest.mark.parametrize("K,sims,play_mode,start", [(1, 24, False, 0), (2, 16, True, 600), (8, 64, False, 900), (16, 48, True, 0),
                                                    (1, 16, True, 1200)])
def test_pseudo6_search_matches_oracle(api, K, sims, play_mode, start):
    moves = run_vector(api, K, n=6, first=30 + K, sims=sims, play_mode=play_mode, max_moves=40, start_rollout=start)
    assert moves > 100


@pytest.mark.parametrize("blocks,prec,K", [(1, "fp32", 1), (2, "bf16", 4)])
def test_network_search_matches_oracle_given_same_outputs(api, blocks, prec, K):
    net = perturbed_net(api, blocks, 4321 + blocks)
    moves = run_vector(api, K, n=4, first=70, sims=12, play_mode=False, max_moves=24, net=net,
                       precision=api.FP32 if prec == "fp32" else api.BF16, start_rollout=700)
    assert moves > 50
    net.close()


def test_full_size_self_play(api):
    """16384 games, a 1-block bf16 six-output network, K = 2: counters add up, the run is reproducible, a half-size shard with the
    second half's game ids reproduces the second half"""
    n, sims, moves, K = 16384, 8, 3, 2
    net = api.Net(blocks=1, seed=6, value_outputs=6)
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


def test_arena_vector_scalar_and_random_match_oracles(api):
    """a six-output searcher, a one-output searcher and the random player, seat-rotated; every game replayed on the oracles"""
    sims, n_games, K, kw = 4, 12, 2, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(5, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K, **kw))
    n6, n1 = api.Net(blocks=1, seed=31, value_outputs=6), api.Net(blocks=1, seed=32)
    m6 = api.Mcts6(env, net=n6, evaluator=api.EVAL_NN, precision=api.FP32)
    m1 = api.Mcts6(env, net=n1, evaluator=api.EVAL_NN, precision=api.BF16)
    seat_agent = (0, 1, 2, 0, 1, 2)
    ar = api.Arena6(env, [m6, m1, None], seat_agent)
    res = ar.play(n_games, SEED, first_game=6)
    trees = [Vector6Mcts(rules_o, net_eval6(n6, api.FP32)), Lockstep6Mcts(rules_o, net_eval1(n1, api.BF16)), None]
    status, plies = [], []
    o = po.Oracle6Game(rules_o)
    for g in range(6, 6 + n_games):
        r = g % 6
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
        status.append(o.status()); plies.append(ply)
    assert (res["status"] == np.array(status, np.int8)).all() and (res["plies"] == np.array(plies, np.uint32)).all()
    assert res["errors"] == 0 and res["sims"] == (res["moves"][0] + res["moves"][1]) * sims
    ar.close(); m6.close(); m1.close(); n6.close(); n1.close(); env.close()


def test_pseudo6_selfplay_records_match_oracle_replay(api):
    """recording with the value vector: the records are oracle/samples6.py's records of the oracle's self-play with Vector6Mcts
    (finished games re-dealt, as az_selfplay6_run does)"""
    n, first, sims, K, moves = 8, 20, 4, 2, 1000
    kw = dict(mcts_simulations=sims, threads_per_mcts=1, max_game_rounds=20)
    env = api.Env6(n, rules=api.default_rules(concurrent_descents=K, **kw), first_game_id=first)
    env.reset(SEED)
    mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO6)
    mc.record(capacity_samples=n * moves, max_moves_per_game=2048)
    mc.selfplay(moves)
    recs, dropped = mc.samples()
    assert dropped == 0 and mc.counters()["errors"] == 0
    mc.close(); env.close()
    rules = po.default_rules(**kw)
    expected = []
    for g in range(n):
        o, t = po.Oracle6Game(rules), Vector6Mcts(rules)
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
