"""TEST INFRASTRUCTURE — fp64 references and error bounds for the bf16 tensor-core contractions, checked on the operands each kernel
actually read (tests/test_tc_operands_gpu.py; the checkers' own power is shown without a GPU in tests/test_tc_operands_cpu.py).

A bf16 x bf16 product is exact in fp32, so given a contraction's operands the kernel differs from an fp64 reference only by the order
and rounding of its fp32 accumulation.  For K accumulated terms that error is at most A = 2 K 2^-24 sum |a w| in any order, even with
truncating adds.  On top of that come the epilogue's fp32 roundings (fma with the folded BatchNorm, the residual add) and, for bf16
outputs, half a bf16 ulp.  These bounds cannot fail on a correct kernel, and one missing tap, a wrong mask, a wrong BatchNorm row or a
missing residual exceeds them by orders of magnitude.

Layout of the tensor-core buffers (az_nn.cuh): [channel chunk of 8][row][8 channels] bf16, AZ_TC_HALO zero rows in front, then
AZ_TC_RPB = 48 rows per board: cell (y, x) at row y * 6 + x, rows 42..47 zero."""
import numpy as np
import torch
import torch.nn.functional as F

HALO, RPB, TILE = 8, 48, 128
U = 2.0 ** -24                       # unit roundoff of fp32
EPS = np.float32(0.001)              # AZ_NN_BN_EPS


# ---------------------------------------------------------------- bf16 helpers
def bf16_rn(x):
    """round fp32 to bf16, nearest even (what __float2bfloat16_rn does to finite values), returned as fp32"""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7fff + ((u >> 16) & 1)) & 0xffff0000
    return u.astype(np.uint32).view(np.float32)


def bf16_trunc(x):
    """round fp32 to bf16 toward zero (a deliberately wrong rounding for the checkers' power)"""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32) & np.uint32(0xffff0000)
    return u.view(np.float32)


def bf16_bits(x):
    return (bf16_rn(x).view(np.uint32) >> 16).astype(np.uint16)


def from_bits(b):
    return (np.asarray(b, np.uint16).astype(np.uint32) << 16).view(np.float32)


def ulp_bf16(v):
    """spacing of bf16 numbers at |v| (8 significant bits); the subnormal spacing at 0"""
    _, e = np.frexp(np.abs(np.asarray(v, np.float64)))
    return np.maximum(np.ldexp(1.0, e - 8), 2.0 ** -133)


def fold_bn(gamma, beta, mean, var):
    """az_nn_tc_prepare's fp32 fold: scale = gamma / sqrtf(var + eps), shift = beta - mean * scale"""
    g, b, m, v = (np.asarray(a, np.float32) for a in (gamma, beta, mean, var))
    scale = g / np.sqrt(v + EPS)
    return scale.astype(np.float32), (b - m * scale).astype(np.float32)


# ---------------------------------------------------------------- buffer decoding
def cell_rows(boards):
    """rows of the chunked layout that hold the 42 cells of each board in `boards` -> [len(boards), 42]"""
    return HALO + np.asarray(boards)[:, None] * RPB + np.arange(42)[None, :]


def decode_cells(buf, boards):
    """chunked bf16 bits [chunks][rows][8] -> fp32 [len(boards), 7, 6, chunks * 8]"""
    rows = cell_rows(boards).ravel()
    v = from_bits(buf[:, rows, :])                                    # [chunks, B * 42, 8]
    return np.ascontiguousarray(v.transpose(1, 0, 2)).reshape(len(boards), 7, 6, -1)


def invalid_rows(n, upto):
    """rows below `upto` that hold no board cell of a batch of n boards (halo, six padding rows per board, rows past the batch)"""
    r = np.arange(upto)
    b, p = (r - HALO) // RPB, (r - HALO) % RPB
    return r[(r < HALO) | (b >= n) | (p >= 42)]


def computed_rows(n):
    """rows of the tiles a forward of n boards computes (the halo in front included)"""
    return HALO + -(-n * RPB // TILE) * TILE


def sample_boards(n, seed=0):
    """every board up to 37; above: first and last, boards straddling 128-row tile boundaries, every board of the last tile and 32 seeded
    random boards"""
    if n <= 37:
        return np.arange(n)
    b = np.arange(n)
    straddle = b[(b * RPB) // TILE != (b * RPB + RPB - 1) // TILE]
    last_tile = (n * RPB - 1) // TILE
    in_last = b[(b * RPB + RPB - 1) // TILE >= last_tile]
    rnd = np.random.default_rng(seed).choice(n, 32, replace=False)
    return np.unique(np.concatenate([[0, n - 1], straddle[:6], straddle[-6:], in_last, rnd]))


# ---------------------------------------------------------------- fp64 references (torch on the CPU, as oracle/nn_oracle._ConvBf16)
def _nchw(x):
    return torch.as_tensor(np.asarray(x, np.float64)).permute(0, 3, 1, 2)


def _oihw(w):
    return torch.as_tensor(np.asarray(w, np.float64)).permute(3, 2, 0, 1)


def conv3x3(x, w):
    """forward: x [n, 7, 6, cin], w HWIO [3, 3, cin, cout] -> (out, sum |x w|) [n, 7, 6, cout]"""
    out = F.conv2d(_nchw(x), _oihw(w), padding=1).permute(0, 2, 3, 1).numpy()
    ab = F.conv2d(_nchw(np.abs(x)), _oihw(np.abs(w)), padding=1).permute(0, 2, 3, 1).numpy()
    return out, ab


def conv3x3_dgrad(dz, w):
    """data gradient: dz [n, 7, 6, cout], w HWIO [3, 3, cin, cout] -> (da, sum |dz w|) [n, 7, 6, cin]"""
    shape = (dz.shape[0], w.shape[2], 7, 6)
    out = torch.nn.grad.conv2d_input(shape, _oihw(w), _nchw(dz), padding=1).permute(0, 2, 3, 1).numpy()
    ab = torch.nn.grad.conv2d_input(shape, _oihw(np.abs(w)), _nchw(np.abs(dz)), padding=1).permute(0, 2, 3, 1).numpy()
    return out, ab


def conv3x3_wgrad(a, dz):
    """weight gradient: a [n, 7, 6, cin], dz [n, 7, 6, cout] -> (dW, sum |a dz|) HWIO [3, 3, cin, cout]"""
    shape = (dz.shape[3], a.shape[3], 3, 3)
    out = torch.nn.grad.conv2d_weight(_nchw(a), shape, _nchw(dz), padding=1).permute(2, 3, 1, 0).numpy()
    ab = torch.nn.grad.conv2d_weight(_nchw(np.abs(a)), shape, _nchw(np.abs(dz)), padding=1).permute(2, 3, 1, 0).numpy()
    return out, ab


def layout_conv(x, w, variants=(1, 0, 2), drop_tap=None):
    """the tensor-core kernels' algorithm on the 48-row board layout, in fp64: tap (ky, kx) reads the row (ky - 1) * 6 + (kx - 1) away in
    operand copy variants[kx] (0 plain, 1 the x = 5 cells zeroed, 2 the x = 0 cells zeroed).  With the default variants it equals
    conv3x3; other variants or a dropped tap give the wrong operations the checkers must reject."""
    n, cin = x.shape[0], x.shape[3]
    flat = np.zeros((HALO + n * RPB + HALO, cin))
    flat[cell_rows(np.arange(n)).ravel()] = np.asarray(x, np.float64).reshape(n * 42, cin)
    xs = (np.arange(flat.shape[0]) - HALO) % RPB % 6
    copies = [flat, np.where((xs == 5)[:, None], 0.0, flat), np.where((xs == 0)[:, None], 0.0, flat)]
    rows = cell_rows(np.arange(n)).ravel()
    out = np.zeros((n * 42, w.shape[3]))
    for t in range(9):
        if t == drop_tap:
            continue
        ky, kx = divmod(t, 3)
        out += copies[variants[kx]][rows + (ky - 1) * 6 + (kx - 1)] @ np.asarray(w[ky, kx], np.float64)
    return out.reshape(n, 7, 6, -1)


# ---------------------------------------------------------------- checkers
def check_bf16(out, acc, absum, K, scale, shift, res=None):
    """a bf16 output relu(acc * scale + shift [+ res]) against the exact contraction acc (sum |a w| = absum over K terms).
    Returns (max err / bound, share of elements != bf16_rn(reference)).  bound = half a bf16 ulp + A + the epilogue's fp32 roundings"""
    acc = np.asarray(acc, np.float64)
    s, h = np.asarray(scale, np.float64), np.asarray(shift, np.float64)
    r = 0.0 if res is None else np.asarray(res, np.float64)
    f = acc * s + h + r
    ref = np.maximum(f, 0.0)
    tol = 2 * K * U * np.abs(s) * absum + 4 * U * (np.abs(acc * s) + np.abs(h) + np.abs(r) + np.abs(f))
    bound = 0.5 * ulp_bf16(ref + tol) + tol
    out = np.asarray(out, np.float64)
    ratio = float((np.abs(out - ref) / bound).max())
    mismatch = float(np.mean(out != bf16_rn(ref.astype(np.float32))))
    return ratio, mismatch


def bf16_tol(acc, absum, K, scale, shift, res=None):
    """the fp32 error bound of acc * scale + shift [+ res] before its bf16 rounding (see check_bf16)"""
    acc = np.asarray(acc, np.float64)
    s, h = np.asarray(scale, np.float64), np.asarray(shift, np.float64)
    r = 0.0 if res is None else np.asarray(res, np.float64)
    f = acc * s + h + r
    return f, 2 * K * U * np.abs(s) * absum + 4 * U * (np.abs(acc * s) + np.abs(h) + np.abs(r) + np.abs(f))


def check_fp32(out, ref, absum, K):
    """an fp32 contraction output against the exact one: |out - ref| <= A = 2 K 2^-24 sum |a w|; returns max err / bound"""
    err = np.abs(np.asarray(out, np.float64) - ref)
    bound = 2 * K * U * np.asarray(absum, np.float64)
    if (err[bound == 0] != 0).any():
        return float("inf")
    return float((err[bound > 0] / bound[bound > 0]).max(initial=0.0))


def check_head_sums(hz, f, tol, head_w):
    """the T3_HEADS epilogue's per-cell sums hz [..., 3] = sum_c bf16(relu(f_c)) * head_w[c] against fp64 sums on bf16_rn of the
    reference activation f (tolerance tol per channel).  A channel whose reference lies within tol of a bf16 rounding boundary or of 0
    may round the other way: it is allowed |w_c| (ulp + tol); every other channel must round exactly as the reference.  The fp32 fma
    chain over 256 channels adds 2 * 256 * 2^-24 sum |act w|.  Returns max err / bound."""
    v = np.maximum(f, 0.0)
    tw = tol + 4 * U * np.abs(f)
    lo = bf16_rn(np.maximum(f - tw, 0.0).astype(np.float32))
    hi = bf16_rn(np.maximum(f + tw, 0.0).astype(np.float32))
    ambiguous = (lo != hi) | (np.abs(f) <= tw)
    act = bf16_rn(v.astype(np.float32)).astype(np.float64)
    hw = np.asarray(head_w, np.float64)                               # [256, 3]
    ref = act @ hw
    slack = np.where(ambiguous, ulp_bf16(v + tw) + tw, 0.0) @ np.abs(hw)
    bound = slack + 2 * 256 * U * (np.abs(act) @ np.abs(hw)) + 2.0 ** -126
    return float((np.abs(np.asarray(hz, np.float64) - ref) / bound).max())


def heads_tail(hz, w, value_outputs=1):
    """policy [n, 43] and value ([n] or [n, 6]) in fp64 from the per-cell head sums hz [n, 42, >= 3] (k_nn_heads_tail /
    k_nn_value6_tail: BatchNorm + ReLU per cell, the dense layers, softmax / tanh)"""
    hz = np.asarray(hz, np.float64)
    g = {k: np.asarray(v, np.float64) for k, v in w.items()}

    def bn(x, p):
        return np.maximum((x - g[p + "/moving_mean"]) * (g[p + "/gamma"] / np.sqrt(g[p + "/moving_variance"] + float(EPS))) + g[p + "/beta"], 0.0)

    p = bn(hz[:, :, 0:2], "bn_pi").reshape(-1, 84)
    logits = p @ g["dense/kernel"] + g["dense/bias"]
    e = np.exp(logits - logits.max(1, keepdims=True))
    policy = e / e.sum(1, keepdims=True)
    v = bn(hz[:, :, 2:3], "bn_v").reshape(-1, 42)
    hdn = np.maximum(v @ g["dense_1/kernel"] + g["dense_1/bias"], 0.0)
    value = np.tanh(hdn @ g["dense_2/kernel"].reshape(256, value_outputs) + g["dense_2/bias"])
    return policy, (value.reshape(-1) if value_outputs == 1 else value)
