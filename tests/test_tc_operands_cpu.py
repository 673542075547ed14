"""CPU suite: the checkers of tests/test_tc_operands_gpu.py (oracle/tc_operands.py) accept the exact reference rounded the way the
kernels round, and reject the kernel-free result of each deliberately wrong operation: one tap dropped, the x masks swapped, the residual
omitted, truncation instead of round-to-nearest-even, the wrong stem BatchNorm row, a weight gradient with one K split missing."""
import numpy as np
import pytest

from oracle import tc_operands as to


@pytest.fixture(scope="module")
def case():
    rng = np.random.default_rng(5)
    n, cin, cout = 3, 16, 24
    x = to.bf16_rn(rng.standard_normal((n, 7, 6, cin)).astype(np.float32))
    w = to.bf16_rn((rng.standard_normal((3, 3, cin, cout)) * 0.3).astype(np.float32))
    res = to.bf16_rn(np.abs(rng.standard_normal((n, 7, 6, cout))).astype(np.float32))
    scale, shift = to.fold_bn(rng.uniform(0.8, 1.2, cout), rng.uniform(-0.1, 0.1, cout), rng.uniform(-0.1, 0.1, cout), rng.uniform(0.7, 1.3, cout))
    acc, ab = to.conv3x3(x, w)
    return dict(x=x, w=w, res=res, scale=scale, shift=shift, acc=acc, ab=ab, K=9 * cin)


def kernel_like(acc, scale, shift, res=None, rnd=to.bf16_rn):
    """what the epilogue stores for an accumulator acc: fp32 fma with the folded BatchNorm, + residual, ReLU, bf16"""
    f = (acc.astype(np.float32) * scale + shift).astype(np.float32)
    if res is not None:
        f = (f + res).astype(np.float32)
    return rnd(np.maximum(f, 0.0).astype(np.float32))


def test_layout_conv_is_the_convolution(case):
    assert np.abs(to.layout_conv(case["x"], case["w"]) - case["acc"]).max() < 1e-12


def test_true_reference_passes(case):
    c = case
    out = kernel_like(c["acc"], c["scale"], c["shift"], c["res"])
    ratio, mism = to.check_bf16(out, c["acc"], c["ab"], c["K"], c["scale"], c["shift"], c["res"])
    assert ratio <= 1.0 and mism < 0.01, (ratio, mism)
    assert to.check_fp32(c["acc"].astype(np.float32), c["acc"], c["ab"], c["K"]) <= 1.0


@pytest.mark.parametrize("tap", range(9))
def test_a_dropped_tap_fails(case, tap):
    c = case
    out = kernel_like(to.layout_conv(c["x"], c["w"], drop_tap=tap), c["scale"], c["shift"])
    assert to.check_bf16(out, c["acc"], c["ab"], c["K"], c["scale"], c["shift"])[0] > 10.0
    assert to.check_fp32(to.layout_conv(c["x"], c["w"], drop_tap=tap), c["acc"], c["ab"], c["K"]) > 10.0


def test_swapped_x_masks_fail(case):
    c = case
    wrong = to.layout_conv(c["x"], c["w"], variants=(2, 0, 1))
    assert to.check_bf16(kernel_like(wrong, c["scale"], c["shift"]), c["acc"], c["ab"], c["K"], c["scale"], c["shift"])[0] > 10.0
    assert to.check_fp32(wrong, c["acc"], c["ab"], c["K"]) > 10.0


def test_omitted_residual_fails(case):
    c = case
    out = kernel_like(c["acc"], c["scale"], c["shift"])
    assert to.check_bf16(out, c["acc"], c["ab"], c["K"], c["scale"], c["shift"], c["res"])[0] > 10.0


def test_truncation_fails(case):
    c = case
    out = kernel_like(c["acc"], c["scale"], c["shift"], c["res"], rnd=to.bf16_trunc)
    ratio, mism = to.check_bf16(out, c["acc"], c["ab"], c["K"], c["scale"], c["shift"], c["res"])
    assert ratio > 1.5 and mism > 0.2, (ratio, mism)          # about half of the non-zero outputs


def test_wrong_stem_bn_row_fails(case):
    c = case
    rng = np.random.default_rng(6)
    srow, hrow = to.fold_bn(rng.uniform(0.8, 1.2, 7), rng.uniform(-0.1, 0.1, 7), rng.uniform(-0.1, 0.1, 7), rng.uniform(0.7, 1.3, 7))
    s, h = srow[None, :, None, None], hrow[None, :, None, None]
    ok = kernel_like(c["acc"], s, h)
    assert to.check_bf16(ok, c["acc"], c["ab"], c["K"], s, h)[0] <= 1.0
    wrong = kernel_like(c["acc"], np.roll(srow, 1)[None, :, None, None], np.roll(hrow, 1)[None, :, None, None])
    assert to.check_bf16(wrong, c["acc"], c["ab"], c["K"], s, h)[0] > 10.0


def test_weight_gradient_with_a_split_missing_fails():
    rng = np.random.default_rng(7)
    n = 4
    a = to.bf16_rn(rng.standard_normal((n, 7, 6, 16)).astype(np.float32))
    dz = to.bf16_rn(rng.standard_normal((n, 7, 6, 8)).astype(np.float32))
    ref, ab = to.conv3x3_wgrad(a, dz)
    assert to.check_fp32(ref.astype(np.float32), ref, ab, n * 48) <= 1.0
    # k_tc_wgrad's K splits are blocks of 64 rows of the 48-row layout: drop the dz rows of the second one
    rows = (np.arange(n)[:, None] * to.RPB + np.arange(42)[None, :]).reshape(n, 7, 6)
    part = dz * ((rows // 64) != 1)[..., None]
    wrong, _ = to.conv3x3_wgrad(a, part)
    assert to.check_fp32(wrong.astype(np.float32), ref, ab, n * 48) > 10.0


def test_head_sums_checker(case):
    c = case
    hw = to.bf16_rn(np.random.default_rng(8).standard_normal((c["acc"].shape[3], 3)).astype(np.float32))
    f, tol = to.bf16_tol(c["acc"], c["ab"], c["K"], c["scale"], c["shift"], c["res"])
    act = kernel_like(c["acc"], c["scale"], c["shift"], c["res"])
    hz = np.zeros(act.shape[:3] + (3,), np.float32)
    for ch in range(act.shape[3]):                                    # the epilogue's fp32 fma chain in channel order
        hz = (hz + act[..., ch:ch + 1] * hw[ch]).astype(np.float32)
    assert to.check_head_sums(hz, f, tol, hw) <= 1.0
    trunc = kernel_like(c["acc"], c["scale"], c["shift"], c["res"], rnd=to.bf16_trunc).astype(np.float64) @ hw
    assert to.check_head_sums(trunc, f, tol, hw) > 1.0
    nores = kernel_like(c["acc"], c["scale"], c["shift"]).astype(np.float64) @ hw
    assert to.check_head_sums(nores, f, tol, hw) > 10.0


def test_tails_reference_matches_the_oracle_network():
    """heads_tail on exact head sums equals oracle/nn_oracle.forward of a one-block network"""
    import torch
    from oracle import nn_oracle as no
    rng = np.random.default_rng(9)
    w = {}
    shapes = {"conv/kernel": (3, 3, 13, 256), "pi/kernel": (1, 1, 256, 2), "v/kernel": (1, 1, 256, 1), "dense/kernel": (84, 43),
              "dense/bias": (43,), "dense_1/kernel": (42, 256), "dense_1/bias": (256,), "dense_2/kernel": (256, 1), "dense_2/bias": (1,)}
    for name in no.variable_names(1):
        shape = shapes.get(name, (3, 3, 256, 256) if name.endswith("kernel") else (7,) if name.startswith("conv_bn") else
                           (2,) if name.startswith("bn_pi") else (1,) if name.startswith("bn_v") else (256,))
        w[name] = rng.uniform(0.7, 1.3, shape) if "variance" in name or "gamma" in name else rng.standard_normal(shape) * 0.05
    x = rng.random((3, 7, 6, 13))
    pol, val = no.forward(w, x, 1, dtype=torch.float64)
    t = torch.as_tensor(x).permute(0, 3, 1, 2)
    t = torch.relu(no._bn(no._conv(t, torch.as_tensor(w["conv/kernel"])), {k: torch.as_tensor(v) for k, v in w.items()}, "conv_bn", 2))
    wt = {k: torch.as_tensor(v) for k, v in w.items()}
    r = torch.relu(no._bn(no._conv(t, wt["res0a_branch2a/kernel"]), wt, "bn0a_branch2a", 1))
    t = torch.relu(no._bn(no._conv(r, wt["res0a_branch2b/kernel"]), wt, "bn0a_branch2b", 1) + t).permute(0, 2, 3, 1).numpy()
    hw = np.concatenate([w["pi/kernel"].reshape(256, 2), w["v/kernel"].reshape(256, 1)], 1)
    p2, v2 = to.heads_tail((t @ hw).reshape(3, 42, 3), w)
    assert np.abs(p2 - pol).max() < 1e-12 and np.abs(v2 - val).max() < 1e-12
