"""GPU suite of the six-player seat planes (SIXPLAYER.md §2, "seat planes"): a network with 16 input planes (az_nn_create_planes), the
16-plane encoding of az_env6_encode_planes, the six-player search's leaf batches, training, checkpoints and the arena.  Checkers:
oracle/risk6_planes.c (r6_encode16), oracle/nn_planes.py (nn_oracle.py's forward and fp64 Trainer with the plane count read from conv/kernel),
oracle/risk6_lockstep.c and oracle/risk6_vector.c (the searches, evaluated by r6_encode16 plus the same CUDA forward at batch 1), and a
13-plane network mapped onto 16 planes, which must compute the 13-plane network's outputs."""
import ctypes as C

import numpy as np
import pytest

from oracle import nn_oracle as no
from oracle import nn_planes as npl
from oracle import planes6
from oracle import pyoracle as po
from oracle.lockstep6 import Lockstep6Mcts
from oracle.samples6 import SAMPLE6_BYTES, sample_record
from oracle.vector6 import EVAL6_CB, Vector6Mcts

pytestmark = pytest.mark.gpu
SEED = 0x5EED0616
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


def perturbed_net(api, blocks, seed, value_outputs=1, input_planes=16):
    net = api.Net(blocks=blocks, seed=seed, value_outputs=value_outputs, input_planes=input_planes)
    rng = np.random.default_rng(seed)
    for name, shape in net.variables():       # make BN parameters non-trivial
        if name.endswith("/gamma"):
            net.load(name, rng.uniform(0.8, 1.2, shape))
        elif name.endswith("/beta") or name.endswith("/bias"):
            net.load(name, rng.uniform(-0.1, 0.1, shape))
    return net


def env6_inputs(api, n, rollout=300, planes=16):
    env = api.Env6(n)
    env.reset(SEED)
    env.rollout(rollout)
    x = env.encode(planes=planes)
    env.close()
    return x


def train_data(api, n, vo, seed=0xC0FFEE):
    rng = np.random.default_rng(seed)
    x = env6_inputs(api, n, 200 + seed % 97)
    tp = rng.random((n, 43)).astype(np.float32)
    tp /= tp.sum(1, keepdims=True)
    tv = rng.choice([1.0, float(LOSS), 0.0], (n, vo)).astype(np.float32)
    return x, tp, (tv[:, 0] if vo == 1 else tv)


def rel(a, b):
    a, b = np.asarray(a, np.float64).ravel(), np.asarray(b, np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ------------------------------------------------------------------ encoding
def test_encode16_matches_oracle(api):
    """dealt positions, mid-game and positions with eliminated seats: az_env6_encode_planes(16) is r6_encode16 bit for bit, and the
    13-plane call is still r6_encode"""
    n = 96
    env = api.Env6(n)
    env.reset(SEED)
    o = po.Oracle6Game()
    eliminated = 0
    for steps in (0, 400, 3000, 6000):
        env.rollout(steps)
        x16, x13, img = env.encode(planes=16), env.encode(), env.export()
        assert x16.shape == (n, 7, 6, 16) and x13.shape == (n, 7, 6, 13)
        for g in range(n):
            o.set_image(img[g])
            assert (bits(x16[g].reshape(-1)) == bits(planes6.encode16(o))).all(), (steps, g)
            assert (bits(x13[g].reshape(-1)) == bits(planes6.encode13(o))).all(), (steps, g)
            eliminated += len(set(int(v) for v in o.s.owner)) < 6
    assert eliminated > 20
    for bad in (0, 12, 14, 15, 17):
        with pytest.raises(api.AzError):
            env.encode(planes=bad)
        with pytest.raises(api.AzError):
            api.Net(blocks=1, input_planes=bad)
    env.close()


# ------------------------------------------------------------------ network
def test_inventory_and_glorot(api):
    net = api.Net(blocks=1, seed=3, input_planes=16)
    shapes = dict(net.variables())
    assert net.input_planes == 16 and shapes["conv/kernel"] == (3, 3, 16, 256)
    thirteen = api.Net(blocks=1)
    assert thirteen.input_planes == 13
    t = dict(thirteen.variables())
    assert {k: v for k, v in shapes.items() if k != "conv/kernel"} == {k: v for k, v in t.items() if k != "conv/kernel"}
    assert net.num_params() - thirteen.num_params() == 9 * 3 * 256
    w = net.get("conv/kernel", (3, 3, 16, 256))
    lim = np.float32(np.sqrt(np.float32(6.0) / np.float32(9 * 16 + 9 * 256)))
    assert abs(float(lim) - 0.049507) < 1e-6
    assert np.abs(w).max() <= lim and np.abs(w).max() > 0.99 * lim
    net.close(); thirteen.close()


@pytest.mark.parametrize("blocks,n,vo", [(2, 37, 1), (1, 1, 6), (3, 130, 6)])
def test_forward_matches_oracle(api, blocks, n, vo):
    net = perturbed_net(api, blocks, 1600 + n, vo)
    x = env6_inputs(api, n)
    p32, v32 = net.forward(x, api.FP32)
    assert v32.shape == ((n,) if vo == 1 else (n, 6))
    rp, rv = npl.forward(net.weights(), x, blocks)
    assert np.abs(p32 - rp).max() <= 1e-5 and np.abs(v32.reshape(-1) - rv).max() <= 1e-5
    p16, v16 = net.forward(x, api.BF16)
    assert np.abs(p32 - p16).max() <= BF16_POLICY_TOL and np.abs(v32 - v16).max() <= BF16_VALUE_TOL
    for prec, p, v in ((api.FP32, p32, v32), (api.BF16, p16, v16)):         # batch invariance
        p1, v1 = net.forward(x[:1], prec)
        assert (bits(p1[0]) == bits(p[0])).all() and (bits(v1[0]) == bits(v[0])).all()
    net.close()


def map_to_16(k13):
    """W16[..., 0] = W13[..., 0], W16[..., 1] = W13[..., 1], W16[..., 2..5] = W13[..., 2], W16[..., 6..15] = W13[..., 3..12]"""
    return np.concatenate([k13[:, :, :2], np.repeat(k13[:, :, 2:3], 4, axis=2), k13[:, :, 3:]], axis=2)


@pytest.mark.parametrize("vo", [1, 6])
def test_mapped_network_equals_the_13_plane_network(api, vo):
    """where all six seats own land, plane 1 is the next seat's in both encodings and planes 2..5 split plane 2 by owner, one non-zero
    per cell: the 16-plane fp32 stem adds exact zeros at the same step of the accumulation order, so the outputs are equal bit for bit"""
    blocks = 2
    net13 = perturbed_net(api, blocks, 616 + vo, vo, input_planes=13)
    net16 = api.Net(blocks=blocks, value_outputs=vo, input_planes=16)
    for name, shape in net13.variables():
        w = net13.get(name, shape)
        net16.load(name, map_to_16(w) if name == "conv/kernel" else w)
    env = api.Env6(512)
    env.reset(SEED)
    env.rollout(900)
    keep = [g for g, im in enumerate(env.export()) if len(set(im[42:84].tolist())) == 6]
    assert len(keep) >= 100
    x13, x16 = env.encode()[keep], env.encode(planes=16)[keep]
    env.close()
    p13, v13 = net13.forward(x13, api.FP32)
    p16, v16 = net16.forward(x16, api.FP32)
    assert (bits(p13) == bits(p16)).all() and (bits(v13) == bits(v16)).all()
    b13, c13 = net13.forward(x13, api.BF16)
    b16, c16 = net16.forward(x16, api.BF16)
    assert np.abs(b16 - b13).max() <= BF16_POLICY_TOL and np.abs(c16 - c13).max() <= BF16_VALUE_TOL
    assert np.abs(b16 - p16).max() <= BF16_POLICY_TOL and np.abs(c16 - v16).max() <= BF16_VALUE_TOL
    net13.close(); net16.close()


# ------------------------------------------------------------------ training
# seeds whose fp64 forward keeps every ReLU input at least 3e-6 away from zero on this batch (8.4e-6 and 3.2e-6): fp32 rounding can put
# an input within ~1e-6 of zero on the other side, and that one element of the mask moves its channel's gradients by ~1e-2 relative
@pytest.mark.parametrize("blocks,n,vo,seed", [(2, 16, 1, 96), (1, 5, 6, 77)])
def test_one_step_matches_trainer(api, blocks, n, vo, seed):
    net = perturbed_net(api, blocks, seed, vo)
    ref = npl.Trainer(net.weights(), blocks)
    x, tp, tv = train_data(api, n, vo)
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


@pytest.mark.parametrize("vo", [1, 6])
def test_bf16_training_step_against_trainer_and_emulation(api, vo):
    """the 16-channel stem on the k_tc_gemm route: its convolution output is the bf16 emulation's (Trainer(bf16=True)) to 1e-6, as in
    tests/test_train_gpu.py; losses and gradients against the exact fp64 Trainer with that file's bounds"""
    blocks, n = 1, 64
    net = perturbed_net(api, blocks, 78, vo)
    net.train_precision(api.BF16)
    w0 = net.weights()
    exact, emu = npl.Trainer(w0, blocks), npl.Trainer(w0, blocks, bf16=True)
    x, tp, tv = train_data(api, n, vo, seed=31)
    lp, lv = net.train_step(x, tp, tv)
    rp, rv = exact.step(x, tp, tv.reshape(-1))
    no.TRACE = {}
    try:
        emu.step(x, tp, tv.reshape(-1))
        trace = no.TRACE
    finally:
        no.TRACE = None
    assert abs(lp - rp) <= 1e-2 * max(1.0, abs(rp)) and abs(lv - rv) <= 1e-2 * max(1.0, abs(rv)), (lp, rp, lv, rv)
    assert rel(net.layer(0, 0, n), trace["conv_bn"]) <= 1e-6
    shapes = dict(net.variables())
    for name in no.trainable_names(blocks):
        g = net.grad(name, shapes[name]).ravel().astype(np.float64)
        gx = exact.grads[name].numpy().ravel()
        cos = float(g @ gx / max(np.linalg.norm(g) * np.linalg.norm(gx), 1e-30))
        assert cos >= 0.98 or gx.size <= 64, (name, cos)
    net.close()


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_several_steps_track_the_trainer(api, prec):
    blocks, n, vo = 2, 24, 6
    net = perturbed_net(api, blocks, 5, vo)
    if prec == "bf16":
        net.train_precision(api.BF16)
    ref = npl.Trainer(net.weights(), blocks)
    x, tp, tv = train_data(api, n, vo, seed=99)
    tol = 2e-3 if prec == "fp32" else 1e-2
    first = None
    for step in range(4):
        lp, lv = net.train_step(x, tp, tv)
        rp, rv = ref.step(x, tp, tv.reshape(-1))
        assert abs(lp - rp) <= tol * max(1.0, abs(rp)) and abs(lv - rv) <= tol * max(1.0, abs(rv)), (step, lp, rp, lv, rv)
        first = first if first is not None else (lp, lv)
    assert lp < first[0] and lv < first[1]
    w = net.weights()
    if prec == "fp32":
        wr = ref.weights()
        for name in w:
            d = np.abs(w[name] - wr[name])
            assert d.max() <= 8.1e-3 and (d.size < 256 or np.median(d) <= 2e-5), (name, np.median(d), d.max())
    p, v = net.forward(x, api.FP32)
    pr, vr = npl.forward(w, x, blocks)
    assert np.abs(p - pr).max() <= 1e-5 and np.abs(v.reshape(-1) - vr).max() <= 1e-5
    net.close()


@pytest.mark.parametrize("vo", [1, 6])
def test_train6_equals_manual_batches(api, vo):
    """az_nn_train6 on a 16-plane network: the records' images are encoded with the seat planes on the device; equal, bit for bit, to
    az_nn_train_step on the same batches with r6_encode16 inputs"""
    rules = po.default_rules()
    o, rng = po.Oracle6Game(rules), np.random.default_rng(16)
    recs, xs, tps, tvs = [], [], [], []
    g = 0
    while len(recs) < 150:
        o.new_game(0xABCF, g, 0)
        ply = 0
        while o.status() == -1 and len(recs) < 150:
            if ply % 17 == 0:
                valid = o.valid()
                t = np.array([rng.random() if (valid >> i) & 1 else 0.0 for i in range(43)], np.float32)
                t /= t.sum()
                status = int(rng.choice([0, 1, 2, 3, 4, 5, -2]))
                recs.append(sample_record(o.image(), t, status)); xs.append(planes6.encode16(o)); tps.append(t)
                tvs.append([0.0 if status == -2 else (1.0 if status == (o.s.cur + k) % 6 else LOSS) for k in range(vo)])
            o.move(o.random_action(0xABCF, g, ply), 0xABCF, g, ply)
            ply += 1
        g += 1
    recs = np.stack(recs); xs = np.array(xs, np.float32); tps = np.array(tps, np.float32); tvs = np.array(tvs, np.float32)
    if vo == 1:
        tvs = tvs[:, 0]
    epochs, batch, seed = 2, 32, 47
    a, b = perturbed_net(api, 1, 9, vo), perturbed_net(api, 1, 9, vo)
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
    a.close(); b.close()


def test_checkpoints_and_cross_plane_rejections(api, tmp_path):
    a = perturbed_net(api, 1, 12)
    x, tp, tv = train_data(api, 8, 1, seed=5)
    a.train_step(x, tp, tv)
    a.save_checkpoint(tmp_path / "sixteen")
    b = api.Net(blocks=1, input_planes=16)
    b.load_checkpoint(tmp_path / "sixteen")
    wa, wb = a.weights(), b.weights()
    for name in wa:
        assert (bits(wa[name]) == bits(wb[name])).all(), name
    assert b.optimizer_powers()[:2] == a.optimizer_powers()[:2]
    for which in (0, 1):
        assert (bits(a.optimizer_slot("conv/kernel", which, (3, 3, 16, 256))) == bits(b.optimizer_slot("conv/kernel", which, (3, 3, 16, 256)))).all()
    assert (bits(a.forward(x, api.FP32)[0]) == bits(b.forward(x, api.FP32)[0])).all()
    thirteen = api.Net(blocks=1, seed=1)
    thirteen.save_checkpoint(tmp_path / "thirteen")
    with pytest.raises(api.AzError):                               # conv/kernel [3, 3, 13, 256] against [3, 3, 16, 256]
        b.load_checkpoint(tmp_path / "thirteen")
    with pytest.raises(api.AzError):
        thirteen.load_checkpoint(tmp_path / "sixteen")
    with pytest.raises(api.AzError):                               # the blobs differ in size
        thirteen.copy_state_from(a)
    with pytest.raises(api.AzError):
        a.copy_state_from(thirteen)
    env = api.Env(4)
    with pytest.raises(api.AzError):                               # the two-player search encodes 13 planes
        api.Mcts(env, net=a, evaluator=api.EVAL_NN)
    with pytest.raises(api.AzError):                               # two-player records encode 13 planes
        a.train(np.zeros((64, api.SAMPLE_BYTES), np.uint8), 1, 32, 0)
    env.close(); a.close(); b.close(); thirteen.close()


# ------------------------------------------------------------------ search
def net_eval16(net, precision):
    """the oracle search's evaluator: r6_encode16 and the same CUDA forward at batch 1 (EVAL6_CB for six outputs, else the scalar one)"""
    if net.value_outputs == 6:
        @EVAL6_CB
        def fn6(sp, policy, value, user):
            p, v = net.forward(planes6.encode16_state(sp).reshape(1, -1), precision)
            C.memmove(policy, p.ctypes.data, 43 * 4)
            C.memmove(value, np.ascontiguousarray(v[0]).ctypes.data, 6 * 4)
        return fn6

    @EVAL_CB
    def fn1(sp, policy, value, user):
        p, v = net.forward(planes6.encode16_state(sp).reshape(1, -1), precision)
        C.memmove(policy, p.ctypes.data, 43 * 4)
        value[0] = float(v[0])
    return fn1


def net_eval13(net, precision):
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


def oracle_tree(net, precision, rules_o):
    fn = net_eval16(net, precision)
    return Vector6Mcts(rules_o, fn) if net.value_outputs == 6 else Lockstep6Mcts(rules_o, fn)


@pytest.mark.parametrize("vo,prec,K", [(1, "fp32", 1), (1, "bf16", 8), (6, "fp32", 2), (6, "bf16", 1), (6, "bf16", 8)])
def test_search_matches_oracle(api, vo, prec, K):
    """the device search over a 16-plane network against r6l_search (one output) / r6v_search (six), move by move, bit for bit"""
    n, first, sims, max_moves, start = 4, 80 + K, 16, 24, 700
    precision = api.FP32 if prec == "fp32" else api.BF16
    net = perturbed_net(api, 1 + (K == 8), 4600 + vo + K, vo)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    env = api.Env6(n, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K), first_game_id=first)
    env.reset(SEED)
    env.rollout(start)
    mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=precision)
    img = env.export()
    games = [po.Oracle6Game(rules_o) for _ in range(n)]
    trees = [oracle_tree(net, precision, rules_o) for _ in range(n)]
    for g, o in enumerate(games):
        o.set_image(img[g])
    ply = np.full(n, start, int)
    moves_done = 0
    for step in range(max_moves):
        res = mc.search(pick_mode=api.PICK_SELFPLAY, apply_move=True)
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
            mv = trees[g].pick(a["pi"], o.s.round <= rules_o.temperature_threshold, SEED, first + g, int(ply[g]))
            assert res["move"][g] == mv, (step, g)
            assert o.move(mv, SEED, first + g, int(ply[g])) == 0
            ply[g] += 1
            moves_done += 1
            assert res["status"][g] == o.status()
    dev = env.export()
    for g, o in enumerate(games):
        assert (dev[g] == o.image()).all(), g
    cnt = mc.counters()
    assert cnt["errors"] == 0 and cnt["sims"] == moves_done * sims and moves_done > 50
    mc.close(); env.close(); net.close()


def test_full_size_self_play(api):
    """16384 games, a 1-block bf16 16-plane six-output network, K = 2: counters add up, the run is reproducible, a half-size shard
    with the second half's game ids reproduces the second half"""
    n, sims, moves, K = 16384, 8, 3, 2
    net = api.Net(blocks=1, seed=16, value_outputs=6, input_planes=16)
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


def test_selfplay_records_match_oracle_replay(api):
    """recording with a 16-plane network: the records are oracle/samples6.py's records of the oracle's self-play with the same
    evaluator (finished games re-dealt, as az_selfplay6_run does)"""
    n, first, sims, K, moves = 4, 40, 4, 2, 500
    kw = dict(mcts_simulations=sims, threads_per_mcts=1, max_game_rounds=17)
    net = perturbed_net(api, 1, 1616, 6)
    env = api.Env6(n, rules=api.default_rules(concurrent_descents=K, **kw), first_game_id=first)
    env.reset(SEED)
    mc = api.Mcts6(env, net=net, evaluator=api.EVAL_NN, precision=api.FP32)
    mc.record(capacity_samples=n * moves, max_moves_per_game=2048)
    mc.selfplay(moves)
    recs, dropped = mc.samples()
    assert dropped == 0 and mc.counters()["errors"] == 0
    mc.close(); env.close()
    rules = po.default_rules(**kw)
    expected = []
    for g in range(n):
        o, t = po.Oracle6Game(rules), oracle_tree(net, api.FP32, rules)
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
    assert len(expected) >= n and recs.shape[1] == SAMPLE6_BYTES
    assert sum(len(e) for e in expected) == recs.size
    blob, pos = recs.tobytes(), 0
    left = sorted(expected, key=len, reverse=True)
    while pos < len(blob):
        hit = [e for e in left if blob.startswith(e, pos)]
        assert hit, "record stream at byte %d matches no expected game" % pos
        left.remove(hit[0]); pos += len(hit[0])
    assert not left
    net.close()


def test_arena_16_plane_13_plane_and_random_match_oracles(api):
    """a 16-plane searcher, a 13-plane searcher and the random player, seat-rotated; every game replayed on the oracles"""
    sims, n_games, K, kw = 4, 12, 2, dict(max_game_rounds=20)
    rules_o = po.default_rules(mcts_simulations=sims, threads_per_mcts=1, **kw)
    env = api.Env6(5, rules=api.default_rules(mcts_simulations=sims, threads_per_mcts=1, concurrent_descents=K, **kw))
    n16, n13 = api.Net(blocks=1, seed=61, value_outputs=6, input_planes=16), api.Net(blocks=1, seed=62)
    m16 = api.Mcts6(env, net=n16, evaluator=api.EVAL_NN, precision=api.BF16)
    m13 = api.Mcts6(env, net=n13, evaluator=api.EVAL_NN, precision=api.FP32)
    seat_agent = (0, 1, 2, 0, 1, 2)
    ar = api.Arena6(env, [m16, m13, None], seat_agent)
    res = ar.play(n_games, SEED, first_game=12)
    trees = [oracle_tree(n16, api.BF16, rules_o), Lockstep6Mcts(rules_o, net_eval13(n13, api.FP32)), None]
    status, plies = [], []
    o = po.Oracle6Game(rules_o)
    for g in range(12, 12 + n_games):
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
    ar.close(); m16.close(); m13.close(); n16.close(); n13.close(); env.close()
