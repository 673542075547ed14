"""GPU suite: every bf16 tensor-core contraction against an fp64 reference on the operands the kernel actually read.

The forward runs through the ordinary API (Net.forward(x, BF16)); az_nn_tc_probe then copies its work buffers back: the stem operand,
the three activation buffers and the per-cell head sums.  Each layer is recomputed in fp64 (oracle/tc_operands.py) from its own input
buffer, its bf16-rounded weights and the BatchNorm fold az_nn_tc_prepare computes, and held to a bound that only fp32 accumulation order
can reach (half a bf16 ulp + 2 K 2^-24 sum |a w| + the epilogue's fp32 roundings).  The training step's contractions are checked the
same way: its per-layer forward through az_nn_train_get_layer, and the forward / data gradient / weight gradient through az_tc_conv_test.
Each check prints the largest err / bound it measured and, for bf16 outputs, the share of elements that did not round as the exact
reference rounds."""
import ctypes as C

import numpy as np
import pytest

from oracle import pyoracle as po
from oracle import tc_operands as to

pytestmark = pytest.mark.gpu

SIZES = [1, 2, 3, 8, 37, 600, 1000, 2048]
MISMATCH_MAX = 0.01          # truncation instead of round-to-nearest-even would put this near one half of the non-zero outputs
TAIL_TOL = 1e-5


@pytest.fixture(scope="module")
def api():
    from alphazero_risk_b200 import api as a
    if a.lib().az_device_count() == 0:
        pytest.fail("no CUDA device visible: the gpu suite must run on a B200")
    L = a.lib()
    L.az_nn_tc_probe.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_int)]
    L.az_tc_conv_test.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
    return a


def report(what, ratio, mismatch=None):
    print("%-58s max err/bound %.3e%s" % (what, ratio, "" if mismatch is None else "  mismatch share %.2e" % mismatch))


def game_inputs(n, seed=0xBEEF):
    """encoded positions from seeded random play (as tests/test_nn_gpu.py builds them)"""
    xs, o, g = [], po.OracleGame(), 0
    while len(xs) < n:
        o.new_game(seed, g, 0)
        ply = 0
        while o.status() == -1 and len(xs) < n:
            if ply % 9 == 0:
                xs.append(o.encode())
            o.move(o.random_action(seed, g, ply), seed, g, ply)
            ply += 1
        g += 1
    return np.array(xs, np.float32).reshape(n, 7, 6, 13)


def inputs(n, planes=13, uniform=False):
    if uniform:
        return np.random.default_rng(n).random((n, 7, 6, planes)).astype(np.float32)
    x = game_inputs(n)
    if planes == 16:                                  # three more live planes
        x = np.concatenate([x, np.random.default_rng(n + 1).random((n, 7, 6, 3)).astype(np.float32)], 3)
    return x


def perturb(net, seed):
    """non-trivial BatchNorm (as tests/test_nn_gpu.py): identity statistics would hide indexing mistakes"""
    rng = np.random.default_rng(seed)
    for name, shape in net.variables():
        if name.endswith("/gamma"):
            net.load(name, rng.uniform(0.8, 1.2, shape))
        elif name.endswith("/beta") or name.endswith("/moving_mean") or name.endswith("/bias"):
            net.load(name, rng.uniform(-0.1, 0.1, shape))
        elif name.endswith("/moving_variance"):
            net.load(name, rng.uniform(0.7, 1.3, shape))


def probe(api, net, which, n):
    ra = C.c_int()
    api.check(api.lib().az_nn_tc_probe(net.h, 0, which, n, None, 0, C.byref(ra)))
    r = ra.value
    buf = np.empty((3, 2, r, 8) if which == 0 else (n, 42, 4) if which == 4 else (32, r, 8), np.uint16 if which < 4 else np.float32)
    api.check(api.lib().az_nn_tc_probe(net.h, 0, which, n, buf.ctypes.data, buf.nbytes, None))
    return buf


def layer_name(i, h):
    return "%d%s_branch2%s" % (i, chr(97 + i), "ab"[h])


def tower(w, i, h):
    """bf16 weights and the folded BatchNorm of tower layer (block i, branch 2a / 2b)"""
    sfx = layer_name(i, h)
    s, sh = to.fold_bn(*(w["bn" + sfx + "/" + k] for k in ("gamma", "beta", "moving_mean", "moving_variance")))
    return to.bf16_rn(w["res" + sfx + "/kernel"]), s, sh


def stem(w, planes):
    k = np.zeros((3, 3, 16, 256), np.float32)
    k[:, :, :planes] = w["conv/kernel"]
    s, sh = to.fold_bn(*(w["conv_bn/" + k2] for k2 in ("gamma", "beta", "moving_mean", "moving_variance")))
    return to.bf16_rn(k), s[None, :, None, None], sh[None, :, None, None]      # BatchNorm per board row


def head_w(w):
    return np.concatenate([w["pi/kernel"].reshape(256, 2), w["v/kernel"].reshape(256, 1)], 1)


def check_stem_operand(din, x, n):
    """the stem's three operand copies bit for bit: bf16_rn(x) (channels past the planes zero), the x = 5 / x = 0 cells zeroed in
    copies 1 / 2, every other row zero"""
    planes = x.shape[3]
    xx = np.zeros((n, 7, 6, 16), np.float32)
    xx[..., :planes] = x
    want = to.bf16_bits(xx).reshape(n * 42, 16)
    cx = np.tile(np.arange(42) % 6, n)
    rows = to.cell_rows(np.arange(n)).ravel()
    for v, masked in ((0, None), (1, 5), (2, 0)):
        got = din[v][:, rows, :].transpose(1, 0, 2).reshape(n * 42, 16)
        exp = want.copy()
        if masked is not None:
            exp[cx == masked] = 0
        assert (got == exp).all(), ("stem operand copy", v)
    assert not din[:, :, to.invalid_rows(n, din.shape[2]), :].any(), "stem operand: halo / padding rows"


def check_padding(buf, n, what):
    assert not buf[:, to.invalid_rows(n, buf.shape[1]), :].any(), what + ": padding rows are not zero"


def check_layer(what, out_buf, in_cells, W, s, sh, boards, res_cells=None):
    acc, ab = to.conv3x3(in_cells, W)
    ratio, mism = to.check_bf16(to.decode_cells(out_buf, boards), acc, ab, 9 * W.shape[2], s, sh, res_cells)
    report(what, ratio, mism)
    assert ratio <= 1.0 and mism < MISMATCH_MAX, (what, ratio, mism)


def check_heads(what, hz, in_cells, W, s, sh, res_cells, hw, boards):
    acc, ab = to.conv3x3(in_cells, W)
    f, tol = to.bf16_tol(acc, ab, 9 * 256, s, sh, res_cells)
    ratio = to.check_head_sums(hz[boards, :, :3].reshape(len(boards), 7, 6, 3), f, tol, hw)
    report(what, ratio)
    assert ratio <= 1.0, (what, ratio)


def check_tails(what, hz, w, pol, val, value_outputs=1):
    rp, rv = to.heads_tail(hz[:, :, :3], w, value_outputs)
    ep, ev = np.abs(pol - rp).max(), np.abs(val - rv).max()
    print("%-58s max |policy err| %.2e  max |value err| %.2e" % (what, ep, ev))
    assert ep <= TAIL_TOL and ev <= TAIL_TOL, (what, ep, ev)


def two_nets(api, seed):
    """a two-block network and a one-block network with the same stem, block 0 and heads: the one-block forward keeps block 0's 2a
    output in d_act[1], which the two-block forward overwrites with block 1's"""
    net2 = api.Net(blocks=2, seed=seed)
    perturb(net2, seed)
    w = net2.weights()
    net1 = api.Net(blocks=1, seed=seed + 1)
    for name, _ in net1.variables():
        net1.load(name, w[name])
    return net1, net2, w


def forward_and_check(api, net1, net2, w, x, tag):
    n = x.shape[0]
    boards = to.sample_boards(n, seed=n)
    p1, v1 = net1.forward(x, api.BF16)
    din = probe(api, net1, 0, n)
    a0, a1, hz1 = probe(api, net1, 1, n), probe(api, net1, 2, n), probe(api, net1, 4, n)
    p2, v2 = net2.forward(x, api.BF16)
    b0, b1, b2, hz2 = probe(api, net2, 1, n), probe(api, net2, 2, n), probe(api, net2, 3, n), probe(api, net2, 4, n)
    check_stem_operand(din, x, n)
    assert (a0 == b0).all(), "the two networks' stem outputs differ"
    for buf, what in ((a0, "stem"), (a1, "block 0 2a"), (b1, "block 1 2a"), (b2, "block 0 2b")):
        check_padding(buf, n, what)
    xin = to.decode_cells(din[0], boards)
    c0, c1 = to.decode_cells(a0, boards), to.decode_cells(a1, boards)
    d1, d2 = to.decode_cells(b1, boards), to.decode_cells(b2, boards)
    check_layer("%s n %d: stem (row BN)" % (tag, n), a0, xin, *stem(w, 13), boards)
    check_layer("%s n %d: block 0 2a" % (tag, n), a1, c0, *tower(w, 0, 0), boards)
    check_heads("%s n %d: block 0 2b + heads (1 block)" % (tag, n), hz1, c1, *tower(w, 0, 1), c0, head_w(w), boards)
    check_layer("%s n %d: block 0 2b + residual" % (tag, n), b2, c1, *tower(w, 0, 1), boards, res_cells=c0)
    check_layer("%s n %d: block 1 2a" % (tag, n), b1, d2, *tower(w, 1, 0), boards)
    check_heads("%s n %d: block 1 2b + heads (2 blocks)" % (tag, n), hz2, d1, *tower(w, 1, 1), d2, head_w(w), boards)
    check_tails("%s n %d: heads tail (1 block)" % (tag, n), hz1, w, p1, v1)
    check_tails("%s n %d: heads tail (2 blocks)" % (tag, n), hz2, w, p2, v2)


@pytest.mark.parametrize("n", SIZES)
def test_forward_layers_on_their_own_operands(api, n):
    """n = 1, 2, 3, 8, 37: odd tile counts (the peer CTA's duplicated last tile); 600: more than one item per CTA pair; 1000: three or
    more items per pair (TMEM accumulators reused, the stem's persistent loop past j = 2); 2048: a self-play cohort"""
    net1, net2, w = two_nets(api, 300 + n)
    forward_and_check(api, net1, net2, w, inputs(n), "positions")
    net1.close(); net2.close()


def test_forward_on_uniform_random_input(api):
    net1, net2, w = two_nets(api, 17)
    forward_and_check(api, net1, net2, w, inputs(37, uniform=True), "uniform input")
    net1.close(); net2.close()


@pytest.mark.parametrize("n", [3, 600])
def test_sixteen_input_planes(api, n):
    """az_nn_tc_forward_planes16: channels 13..15 of the stem operand are live; the stem, tower and heads are the same kernels"""
    net = api.Net(blocks=1, seed=5 + n, input_planes=16)
    perturb(net, 5 + n)
    w = net.weights()
    x = inputs(n, planes=16)
    pol, val = net.forward(x, api.BF16)
    boards = to.sample_boards(n, seed=n)
    din, a0, a1, hz = probe(api, net, 0, n), probe(api, net, 1, n), probe(api, net, 2, n), probe(api, net, 4, n)
    check_stem_operand(din, x, n)
    check_padding(a0, n, "stem"); check_padding(a1, n, "2a")
    c0, c1 = to.decode_cells(a0, boards), to.decode_cells(a1, boards)
    check_layer("16 planes n %d: stem (row BN)" % n, a0, to.decode_cells(din[0], boards), *stem(w, 16), boards)
    check_layer("16 planes n %d: block 0 2a" % n, a1, c0, *tower(w, 0, 0), boards)
    check_heads("16 planes n %d: block 0 2b + heads" % n, hz, c1, *tower(w, 0, 1), c0, head_w(w), boards)
    check_tails("16 planes n %d: heads tail" % n, hz, w, pol, val)
    net.close()


@pytest.mark.parametrize("n", [37, 1000])
def test_six_value_outputs_tail(api, n):
    """k_nn_value6_tail from the kernel's own head sums; the policy comes from k_nn_heads_tail as for one output"""
    net = api.Net(blocks=1, seed=11 + n, value_outputs=6)
    perturb(net, 11 + n)
    w = net.weights()
    pol, val = net.forward(inputs(n), api.BF16)
    check_tails("six value outputs n %d" % n, probe(api, net, 4, n), w, pol, val, value_outputs=6)
    net.close()


def test_smaller_batch_after_a_larger_one_equals_a_fresh_network(api):
    """n = 1000 then n = 37 on the same buffers: the 37 boards' operand rows and every row of the tiles the second forward computes
    (activations, padding, halo) are bit for bit what a fresh network writes, and so are its head sums and outputs"""
    dirty, other, w = two_nets(api, 41)
    other.close()
    fresh = api.Net(blocks=1)
    for name, _ in fresh.variables():
        fresh.load(name, w[name])
    dirty.forward(inputs(1000, uniform=True), api.BF16)
    x = inputs(37)
    pd, vd = dirty.forward(x, api.BF16)
    pf, vf = fresh.forward(x, api.BF16)
    assert (pd == pf).all() and (vd == vf).all()
    upto = to.computed_rows(37)
    for which in (1, 2):
        assert (probe(api, dirty, which, 37)[:, :upto] == probe(api, fresh, which, 37)[:, :upto]).all(), which
    rows = slice(to.HALO, to.HALO + 37 * to.RPB)
    assert (probe(api, dirty, 0, 37)[:, :, rows] == probe(api, fresh, 0, 37)[:, :, rows]).all()
    assert (probe(api, dirty, 4, 37) == probe(api, fresh, 4, 37)).all()
    dirty.close(); fresh.close()


def unit_bn(net):
    """BatchNorm whose fp32 fold is exactly scale 1, shift 0"""
    var = np.float32(1) - to.EPS
    while np.float32(var + to.EPS) != np.float32(1):
        var = np.nextafter(var, np.float32(2))
    for name, shape in net.variables():
        if name.startswith(("conv_bn", "bn0a")):
            value = {"gamma": 1.0, "beta": 0.0, "moving_mean": 0.0, "moving_variance": var}[name.split("/")[1]]
            net.load(name, np.full(shape, value, np.float32))
    s, h = to.fold_bn(np.ones(256), np.zeros(256), np.zeros(256), np.full(256, var))
    assert (s == 1).all() and (h == 0).all()


def test_structured_operands_exact(api):
    """one-hot inputs, small-integer weights, BatchNorm folded to exactly (1, 0): every output is an exact integer that depends on
    which (cell, tap, channel) produced it, so the stem, 2a, 2b (+ residual) and head sums must equal the fp64 reference exactly"""
    n = 37
    rng = np.random.default_rng(23)
    x = np.zeros((n, 7, 6, 13), np.float32)
    b, y, xx = np.meshgrid(np.arange(n), np.arange(7), np.arange(6), indexing="ij")
    x[b, y, xx, (b * 5 + y * 6 + xx) % 13] = 1.0
    ws = rng.integers(0, 2, (3, 3, 13, 256)).astype(np.float32)                       # stem outputs 0..9
    t = np.arange(9).reshape(3, 3, 1, 1)
    ci, co = np.arange(256).reshape(1, 1, 256, 1), np.arange(256).reshape(1, 1, 1, 256)
    sign = rng.choice([-1.0, 1.0], (3, 3, 1, 256))
    w2a = np.where(ci == (co * 11 + t * 29) % 256, sign, 0.0).astype(np.float32)      # |2a| <= 81
    w2b = np.where((ci == (co * 13 + t * 7) % 256) & ((t == co % 9) | (t == (co + 4) % 9)), 1.0, 0.0).astype(np.float32)   # 2b <= 171
    hw = rng.integers(-1, 2, (256, 3)).astype(np.float32)
    nets = [api.Net(blocks=1, seed=1), api.Net(blocks=2, seed=2)]
    for net in nets:
        unit_bn(net)
        net.load("conv/kernel", ws)
        net.load("res0a_branch2a/kernel", w2a)
        net.load("res0a_branch2b/kernel", w2b)
        net.load("pi/kernel", hw[:, :2].reshape(1, 1, 256, 2))
        net.load("v/kernel", hw[:, 2:].reshape(1, 1, 256, 1))
        net.forward(x, api.BF16)
    ref0 = np.maximum(to.conv3x3(x, ws)[0], 0)
    ref1 = np.maximum(to.conv3x3(ref0, w2a)[0], 0)
    ref2 = np.maximum(to.conv3x3(ref1, w2b)[0] + ref0, 0)
    assert ref2.max() < 256 and np.abs(ref1).max() < 256
    allb = np.arange(n)
    assert (to.decode_cells(probe(api, nets[0], 1, n), allb) == ref0).all(), "stem"
    assert (to.decode_cells(probe(api, nets[0], 2, n), allb) == ref1).all(), "2a"
    assert (probe(api, nets[0], 4, n)[:, :, :3].reshape(n, 7, 6, 3) == ref2 @ hw).all(), "2b + heads"
    assert (to.decode_cells(probe(api, nets[1], 3, n), allb) == ref2).all(), "2b + residual"
    for net in nets:
        net.close()


# ---------------------------------------------------------------- training step
def train_layer_name(L):
    return "conv/kernel" if L == 0 else "res%s/kernel" % layer_name((L - 1) // 2, 1 - L % 2)


@pytest.mark.parametrize("blocks,n,planes", [(2, 5, 13), (3, 64, 13), (2, 131, 16), (3, 512, 13), (2, 64, 16)])
def test_training_forward_layers_on_their_own_operands(api, blocks, n, planes):
    """train_precision(BF16): z[L] against the fp64 convolution of bf16_rn(a[L - 1]) (k_tr_bn_apply_rpb rounds the fp32 value it
    stores) and bf16_rn of the weights before the step; L = 0 is the stem (im2col + k_tc_gemm), L >= 1 the tower kernel (T3_RAW)"""
    net = api.Net(blocks=blocks, seed=77, input_planes=planes)
    perturb(net, 77)
    net.train_precision(api.BF16)
    w0 = net.weights()
    x = inputs(n, planes=planes)
    rng = np.random.default_rng(n)
    tp = rng.random((n, 43)).astype(np.float32)
    tp /= tp.sum(1, keepdims=True)
    net.train_step(x, tp, rng.choice([-1.0, 1.0], n).astype(np.float32))
    boards = to.sample_boards(n, seed=n)
    prev = x
    for L in range(2 * blocks + 1):
        z = net.layer(L, 0, n)
        W = to.bf16_rn(w0[train_layer_name(L)])
        acc, ab = to.conv3x3(to.bf16_rn(prev[boards]), W)
        ratio = to.check_fp32(z[boards], acc, ab, 9 * (16 if L == 0 else 256))
        report("training forward blocks %d n %d planes %d: layer %d" % (blocks, n, planes, L), ratio)
        assert ratio <= 1.0, (L, ratio)
        prev = net.layer(L, 1, n)
    net.close()


def conv_test(api, mode, a, b, n, n_warm=0, max_splits=1):
    out = np.empty((3, 3, 256, 256) if mode == 2 else (n, 7, 6, 256), np.float32)
    api.check(api.lib().az_tc_conv_test(mode, np.ascontiguousarray(a, np.float32).ctypes.data, np.ascontiguousarray(b, np.float32).ctypes.data,
                                          n, n_warm, max_splits, out.ctypes.data))
    return out


CONV_CASES = [(0, n, 0, 1) for n in (1, 5, 37, 131, 512, 1000)] + [(0, 37, 600, 1)] + \
             [(1, n, 0, 1) for n in (1, 5, 37, 131, 512, 1000)] + [(1, 37, 1000, 1)] + \
             [(2, 1, 0, 1), (2, 5, 0, 16), (2, 37, 0, 1), (2, 37, 0, 16), (2, 131, 0, 16), (2, 512, 0, 1), (2, 512, 0, 16), (2, 1000, 0, 16),
              (2, 5, 600, 16), (2, 131, 1000, 1)]


@pytest.mark.parametrize("mode,n,n_warm,max_splits", CONV_CASES)
def test_training_contractions(api, mode, n, n_warm, max_splits):
    """az_tc_conv_test: forward (az_tc_conv_raw), data gradient (az_tc_dz_prepare + az_tc_dgrad_prepared), weight gradient
    (az_tc_wgrad_prepared, K splits, az_tg_reduce) on bf16-representable operands; n_warm > n first dirties the same scratch"""
    rng = np.random.default_rng(1000 * mode + n)
    a = to.bf16_rn(rng.standard_normal((n, 7, 6, 256)).astype(np.float32))
    b = to.bf16_rn((rng.standard_normal((n, 7, 6, 256)) if mode == 2 else rng.standard_normal((3, 3, 256, 256)) * 0.05).astype(np.float32))
    out = conv_test(api, mode, a, b, n, n_warm, max_splits)
    if mode == 2:
        ref, ab = to.conv3x3_wgrad(a, b)
        ratio = to.check_fp32(out, ref, ab, n * to.RPB + max_splits)
    else:
        boards = to.sample_boards(n, seed=n)
        ref, ab = (to.conv3x3 if mode == 0 else to.conv3x3_dgrad)(a[boards], b)
        ratio = to.check_fp32(out[boards], ref, ab, 9 * 256)
    report("%s n %d n_warm %d max_splits %d" % (("forward", "data gradient", "weight gradient")[mode], n, n_warm, max_splits), ratio)
    assert ratio <= 1.0, ratio


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_training_contractions_structured_exact(api, mode):
    """one-hot activations (mode 0 / 2) or gradients (mode 1) and small-integer weights or gradients: every output is an exact
    integer, so the kernel must equal the fp64 reference exactly"""
    n = 5
    rng = np.random.default_rng(mode)
    onehot = np.zeros((n, 7, 6, 256), np.float32)
    b, y, x = np.meshgrid(np.arange(n), np.arange(7), np.arange(6), indexing="ij")
    onehot[b, y, x, (b * 42 + y * 6 + x) * 37 % 256] = 1.0
    if mode == 2:
        other = rng.integers(-2, 3, (n, 7, 6, 256)).astype(np.float32)
        ref = to.conv3x3_wgrad(onehot, other)[0]
    else:
        other = rng.integers(-2, 3, (3, 3, 256, 256)).astype(np.float32)
        ref = (to.conv3x3 if mode == 0 else to.conv3x3_dgrad)(onehot, other)[0]
    out = conv_test(api, mode, onehot, other, n, 0, 16)
    assert (out == ref).all(), np.argwhere(out != ref)[:8]
