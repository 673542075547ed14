"""GPU suite of the six-player training samples (az_selfplay6_record / az_selfplay6_samples, AZ_SAMPLE6_BYTES records) and of
az_nn_train6.  The checker is oracle/risk6_oracle.c: every record must equal, byte for byte, the oracle's replay of the same game
(r6_mcts_search with the pseudo evaluator, the same move choice) turned into records by oracle/samples6.py."""
import numpy as np
import pytest

from oracle import pyoracle as po
from oracle.samples6 import sample_record

pytestmark = pytest.mark.gpu
SEED = 0x5EED0001
REC = 288
LOSS = np.float32(-1.0) / np.float32(5.0)


@pytest.fixture(scope="module")
def api():
    from alphazero_risk_b200 import api as a
    if a.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    return a


def rules_kw(sims):
    return dict(mcts_simulations=sims, threads_per_mcts=1, max_game_rounds=20)


def replay(n, first, sims, moves, seed=SEED, images=None, ply0=0):
    """the oracle's self-play of games first .. first + n - 1 for `moves` moves (finished games re-dealt, as az_selfplay6_run does):
    the records of every game that finished, one bytes blob per game, in finishing order per slot"""
    rules = po.default_rules(**rules_kw(sims))
    done = []
    for g in range(n):
        o, t = po.Oracle6Game(rules), po.Oracle6Mcts(rules)
        if images is None:
            o.new_game(seed, first + g, 0)
        else:
            o.set_image(images[g])
        cur, ply = [], ply0
        for _ in range(moves):
            a = t.search(o, seed, first + g, ply)
            cur.append((o.image(), a["pi"].copy()))
            mv = t.pick(a["pi"], o.s.round <= rules.temperature_threshold, seed, first + g, ply)
            assert o.move(mv, seed, first + g, ply) == 0
            ply += 1
            st = o.status()
            if st != -1:
                done.append(np.stack([sample_record(img, pi, st) for img, pi in cur]).tobytes())
                cur = []
                o.new_game(seed, first + g, ply)
    return done


def match_whole_games(recs, expected):
    """the queue = whole expected games back to back (in any order); returns the games found"""
    blob, left, pos, found = recs.tobytes(), sorted(expected, key=len, reverse=True), 0, []
    while pos < len(blob):
        hit = [e for e in left if blob.startswith(e, pos)]
        assert hit, "record stream at byte %d matches no expected game" % pos
        left.remove(hit[0]); found.append(hit[0]); pos += len(hit[0])
    return found


N1, FIRST1, SIMS1, MOVES1 = 12, 3, 4, 1000


@pytest.fixture(scope="module")
def expected1():
    return replay(N1, FIRST1, SIMS1, MOVES1)


def selfplay_recorded(api, n, first, sims, moves, capacity, max_moves, seed=SEED):
    env = api.Env6(n, rules=api.default_rules(**rules_kw(sims)), first_game_id=first)
    env.reset(seed)
    mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    mc.record(capacity_samples=capacity, max_moves_per_game=max_moves)
    mc.selfplay(moves)
    recs, dropped = mc.samples()
    again, dropped2 = mc.samples()
    assert mc.counters()["errors"] == 0
    mc.close(); env.close()
    return recs, dropped, again, dropped2


def test_selfplay_records_match_oracle_replay(api, expected1):
    recs, dropped, again, dropped2 = selfplay_recorded(api, N1, FIRST1, SIMS1, MOVES1, N1 * MOVES1, 2048)
    assert len(expected1) >= N1 // 2, "too few finished games for a meaningful check"
    assert dropped == 0 and recs.shape[1] == REC
    assert sum(len(e) for e in expected1) == recs.size
    assert len(match_whole_games(recs, expected1)) == len(expected1)
    z = recs[:, 108:112].copy().view(np.float32).reshape(-1)
    assert set(np.unique(z).tolist()) <= {1.0, float(LOSS), 0.0} and (z == 1.0).any() and (z == LOSS).any()
    pi = recs[:, 112:284].copy().view(np.float32)
    assert np.allclose(pi.sum(1), 1.0, atol=1e-5)
    assert (recs[:, 285:] == 0).all()
    assert len(again) == 0 and dropped2 == 0


def test_recording_changes_nothing_the_search_computes(api):
    n, sims = 8, 6

    def run(record):
        env = api.Env6(n, rules=api.default_rules(**rules_kw(sims)), first_game_id=40)
        env.reset(SEED)
        mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
        if record:
            mc.record(capacity_samples=100000, max_moves_per_game=2048)
        outs = []
        for step in range(40):
            res = mc.search(pick_mode=step % 2, apply_move=True)
            outs.append((res, mc.root_stats()))
        mc.selfplay(600)
        res = mc.search(pick_mode=api.PICK_SELFPLAY, apply_move=True)
        outs.append((res, mc.root_stats()))
        cnt, img = mc.counters(), env.export().copy()
        if record:
            assert len(mc.samples()[0]) > 0
        mc.close(); env.close()
        return outs, cnt, img

    (o0, c0, i0), (o1, c1, i1) = run(False), run(True)
    assert c0 == c1 and c0["games"] > 0 and (i0 == i1).all()
    for (r0, s0), (r1, s1) in zip(o0, o1):
        for k in r0:
            assert (np.ascontiguousarray(r0[k]).view(np.uint8) == np.ascontiguousarray(r1[k]).view(np.uint8)).all(), k
        for k in s0:
            assert (np.ascontiguousarray(s0[k]).view(np.uint8) == np.ascontiguousarray(s1[k]).view(np.uint8)).all(), k


def test_small_queue_returns_whole_games_and_counts_the_rest(api, expected1):
    total = sum(len(e) for e in expected1) // REC
    cap = total // 3
    recs, dropped, _, _ = selfplay_recorded(api, N1, FIRST1, SIMS1, MOVES1, cap, 2048)
    assert 0 < len(recs) <= cap
    found = match_whole_games(recs, expected1)
    assert sum(len(f) for f in found) == recs.size
    assert len(recs) + dropped == total


def test_game_longer_than_staging_is_dropped_whole(api, expected1):
    lengths = sorted(len(e) // REC for e in expected1)
    limit = lengths[len(lengths) // 2]
    recs, dropped, _, _ = selfplay_recorded(api, N1, FIRST1, SIMS1, MOVES1, N1 * MOVES1, limit)
    kept = [e for e in expected1 if len(e) // REC <= limit]
    assert 0 < len(kept) < len(expected1)
    assert sorted(match_whole_games(recs, expected1)) == sorted(kept)
    assert dropped == sum(len(e) // REC for e in expected1 if len(e) // REC > limit)


def test_search_apply_move_flushes_each_game_once(api):
    """az_mcts6_search(apply_move = 1) without re-deals: a game's records appear when it ends, and a finished game records nothing more"""
    n, first, sims = 6, 20, 4
    rules = po.default_rules(**rules_kw(sims))
    env = api.Env6(n, rules=api.default_rules(**rules_kw(sims)), first_game_id=first)
    env.reset(SEED)
    mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    mc.record(capacity_samples=20000, max_moves_per_game=2048)
    got, steps = [], 0
    while steps < 4000:
        res = mc.search(pick_mode=api.PICK_SELFPLAY, apply_move=True)
        steps += 1
        r, dropped = mc.samples()
        assert dropped == 0
        if len(r):
            got.append(r)
        if (res["status"] != -1).all():
            break
    assert (res["status"] != -1).all(), "games did not finish"
    for _ in range(3):
        res = mc.search(pick_mode=api.PICK_SELFPLAY, apply_move=True)
        assert (res["move"] == 43).all() and (res["status"] != -1).all()
    assert len(mc.samples()[0]) == 0
    recs = np.concatenate(got)
    expected = []
    for g in range(n):
        o, t = po.Oracle6Game(rules), po.Oracle6Mcts(rules)
        o.new_game(SEED, first + g, 0)
        cur, ply = [], 0
        while o.status() == -1:
            a = t.search(o, SEED, first + g, ply)
            cur.append((o.image(), a["pi"].copy()))
            mv = t.pick(a["pi"], o.s.round <= rules.temperature_threshold, SEED, first + g, ply)
            assert o.move(mv, SEED, first + g, ply) == 0
            ply += 1
        st = o.status()
        assert st == res["status"][g]
        blob = [sample_record(img, pi, st) for img, pi in cur]
        expected.append(np.stack(blob).tobytes())
    assert sum(len(e) for e in expected) == recs.size
    assert len(match_whole_games(recs, expected)) == n
    mc.close(); env.close()


@pytest.mark.parametrize("how", ["reset", "import"])
def test_reset_or_import_discards_staged_samples(api, how):
    n, first, sims, pre, moves = 8, 60, 4, 30, 900
    seed2 = SEED + 7 if how == "reset" else SEED
    env = api.Env6(n, rules=api.default_rules(**rules_kw(sims)), first_game_id=first)
    env.reset(SEED)
    mc = api.Mcts6(env, evaluator=api.EVAL_PSEUDO)
    mc.record(capacity_samples=n * moves, max_moves_per_game=2048)
    mc.selfplay(pre)
    assert len(mc.samples()[0]) == 0
    if how == "reset":
        env.reset(seed2)
        images, ply0 = None, 0
    else:
        images, ply0 = env.export().copy(), pre
        env.import_images(images)
    mc.selfplay(moves)
    recs, dropped = mc.samples()
    assert dropped == 0
    expected = replay(n, first, sims, moves, seed=seed2, images=images, ply0=ply0)
    assert len(expected) >= n // 2
    assert sum(len(e) for e in expected) == recs.size
    assert len(match_whole_games(recs, expected)) == len(expected)
    mc.close(); env.close()


def test_shard_records_are_contained_in_the_full_run(api):
    n, sims, moves = 16, 4, 700
    full, d0, _, _ = selfplay_recorded(api, n, 0, sims, moves, n * moves, 2048)
    half, d1, _, _ = selfplay_recorded(api, n // 2, n // 2, sims, moves, n * moves, 2048)
    assert d0 == 0 and d1 == 0 and len(half) > 0 and len(half) < len(full)
    rows, counts = np.unique(full, axis=0, return_counts=True)
    have = {r.tobytes(): c for r, c in zip(rows, counts)}
    hrows, hcounts = np.unique(half, axis=0, return_counts=True)
    for r, c in zip(hrows, hcounts):
        assert have.get(r.tobytes(), 0) >= c


def perturbed_net(api, blocks, seed):
    net = api.Net(blocks=blocks, seed=seed)
    rng = np.random.default_rng(seed)
    for name, shape in net.variables():
        if name.endswith("/gamma"):
            net.load(name, rng.uniform(0.8, 1.2, shape))
        elif name.endswith("/beta") or name.endswith("/bias"):
            net.load(name, rng.uniform(-0.1, 0.1, shape))
    return net


def test_train6_equals_manual_batches(api):
    """az_nn_train6: records -> six-seat planes / targets on the device, shuffled whole batches per epoch == az_nn_train_step on the
    same batches built on the host from the oracle's r6_encode"""
    rules = po.default_rules()
    o, enc, rng = po.Oracle6Game(rules), po.Oracle6Mcts(rules), np.random.default_rng(5)
    recs, xs, tps, tvs = [], [], [], []
    g = 0
    while len(recs) < 150:
        o.new_game(0xABCD, g, 0)
        ply = 0
        while o.status() == -1 and len(recs) < 150:
            if ply % 11 == 0:
                valid = o.valid()
                t = np.array([rng.random() if (valid >> i) & 1 else 0.0 for i in range(43)], np.float32)
                t /= t.sum()
                status = int(rng.choice([0, 1, 2, 3, 4, 5, -2]))
                recs.append(sample_record(o.image(), t, status)); xs.append(enc.encode(o)); tps.append(t)
                tvs.append(0.0 if status == -2 else (1.0 if status == o.s.cur else LOSS))
            o.move(o.random_action(0xABCD, g, ply), 0xABCD, g, ply)
            ply += 1
        g += 1
    recs = np.stack(recs); xs = np.array(xs, np.float32); tps = np.array(tps, np.float32); tvs = np.array(tvs, np.float32)
    epochs, batch, seed = 2, 32, 42
    a, b = perturbed_net(api, 1, 8), perturbed_net(api, 1, 8)
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
        assert (wa[name].view(np.uint32) == wb[name].view(np.uint32)).all(), name
    assert lp[1] < lp[0]
    bad = recs[:batch].copy()
    bad[3, 42 + 7] = 6                                              # an owner byte outside the six seats
    with pytest.raises(api.AzError):
        a.train6(bad, 1, batch, seed)
    a.close(); b.close()


def test_selfplay6_train6_loop(api):
    """six-player self-play with the network evaluator -> records -> az_nn_train6: the network learns its own samples, and a searcher
    built before the training call evaluates with the new weights"""
    blocks, games, sims = 2, 96, 8
    rules = api.default_rules(**rules_kw(sims))
    gen_net, train_net = api.Net(blocks=blocks, seed=21), api.Net(blocks=blocks, seed=21)
    env = api.Env6(games, rules=rules)
    env.reset(SEED)
    gen = api.Mcts6(env, net=gen_net, evaluator=api.EVAL_NN, precision=api.BF16)
    gen.record(capacity_samples=200000, max_moves_per_game=4096)
    recs = np.zeros((0, REC), np.uint8)
    for _ in range(20):
        gen.selfplay(100)
        r, dropped = gen.samples()
        assert dropped == 0
        recs = np.concatenate([recs, r])
        if len(recs) >= 4096:
            break
    assert len(recs) >= 4096 and gen.counters()["errors"] == 0
    z = recs[:, 108:112].copy().view(np.float32).reshape(-1)
    assert set(np.unique(z).tolist()) <= {1.0, float(LOSS), 0.0}
    train_net.train_precision(api.BF16)
    lp, lv = train_net.train6(recs, epochs=6, batch_size=512, seed=1)
    assert np.isfinite(lp).all() and np.isfinite(lv).all()
    assert lp[-1] < lp[0] and lv[-1] < lv[0], (lp, lv)
    # a searcher built BEFORE the training call sees the new weights: its root priors are the new forward's masked, normalised policy
    env2 = api.Env6(8, rules=rules, first_game_id=500)
    env2.reset(SEED)
    env2.rollout(200)
    mc = api.Mcts6(env2, net=train_net, evaluator=api.EVAL_NN, precision=api.FP32)
    x = env2.encode()
    p_before, _ = train_net.forward(x, api.FP32)
    train_net.train6(recs[:1024], epochs=1, batch_size=512, seed=2)
    p_after, _ = train_net.forward(x, api.FP32)
    valid, status = env2.query()
    mask = np.array([[(int(v) >> i) & 1 for i in range(43)] for v in valid], bool)

    def priors(p):
        q = np.where(mask, p, 0.0).astype(np.float32)
        return q / q.sum(1, keepdims=True)

    mc.search(pick_mode=api.PICK_ARGMAX, apply_move=False)
    P = mc.root_stats()["P"]
    live = status == -1
    assert live.any()
    assert np.abs(priors(p_after) - priors(p_before))[live].max() > 1e-4
    assert np.allclose(P[live], priors(p_after)[live], atol=1e-6), "the search still evaluates with the weights from before the training call"
    print("six-player loop: %d samples, policy loss %.3f -> %.3f, value loss %.4f -> %.4f" % (len(recs), lp[0], lp[-1], lv[0], lv[-1]))
    for h in (mc, env2, gen, env, train_net, gen_net):
        h.close()
