"""CPU checks of the six-player seat planes (SIXPLAYER.md §2, "seat planes") on the oracle: r6_encode16 (oracle/risk6_planes.c) against
r6_encode on rollouts with eliminations, the binding's constants against the C header, and oracle/nn_planes.py (nn_oracle.py's network
with the plane count read from conv/kernel): nn_oracle itself at 13 planes, and a 13-plane network mapped onto 16 planes computes the
same function."""
import ctypes as C
import os
import re

import numpy as np
import torch

from oracle import graphdef_oracle as go
from oracle import nn_oracle as no
from oracle import nn_planes as npl
from oracle import planes6
from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0x5EED0016


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def rollout_positions(n_games=6, every=13):
    """positions of whole random games (to the end, so later positions have eliminated seats)"""
    rules = po.default_rules()
    out = []
    for g in range(n_games):
        o = po.Oracle6Game(rules)
        o.new_game(SEED, g, 0)
        ply = 0
        while o.status() == -1:
            if ply % every == 0:
                out.append(o.image())
            assert o.move(o.random_action(SEED, g, ply), SEED, g, ply) == 0
            ply += 1
        out.append(o.image())
    return out


def test_seat_planes_against_the_13_plane_encoding():
    o = po.Oracle6Game()
    eliminated_seen = 0
    for img in rollout_positions():
        o.set_image(img)
        x16 = planes6.encode16(o).reshape(42, 16)
        x13 = planes6.encode13(o).reshape(42, 13)
        assert (bits(x16[:, 0]) == bits(x13[:, 0])).all()
        assert (bits(x16[:, 6:]) == bits(x13[:, 3:])).all()
        assert (bits(x16[:, 1:6].sum(1)) == bits(x13[:, 1] + x13[:, 2])).all()       # one owner per land: one non-zero term
        cur = int(o.s.cur)
        owners = set(int(v) for v in o.s.owner)
        alive = [k for k in range(1, 6) if (cur + k) % 6 in owners]
        if alive:
            assert (bits(x16[:, alive[0]]) == bits(x13[:, 1])).all()                     # k*: the first seat alive after cur
        for k in range(6):
            seat_lands = np.array([int(v) == (cur + k) % 6 for v in o.s.owner])
            assert (x16[~seat_lands, k] == 0).all() and (x16[seat_lands, k] > 0).all()
            if not seat_lands.any():
                eliminated_seen += 1
                assert (bits(x16[:, k]) == 0).all()
    assert eliminated_seen > 100


def test_binding_agrees_with_header():
    from alphazero_risk_b200 import api
    text = open(os.path.join(ROOT, "include", "az_b200.h")).read()
    floats = int(re.search(r"#define AZ_INPUT6_FLOATS\s+(\d+)", text).group(1))
    assert floats == api.INPUT6_FLOATS == planes6.INPUT6_FLOATS == 42 * 16
    assert C.c_int.in_dll(planes6.lib(), "r6_input16_floats").value == floats
    assert re.search(r"AZ_API int az_nn_create_planes\(int blocks, int value_outputs, int input_planes, int device, az_nn\*\* out\);", text)
    assert re.search(r"AZ_API int az_nn_input_planes\(const az_nn\* nn\);", text)
    assert re.search(r"AZ_API int az_env6_encode_planes\(az_env6\* env, int input_planes, float\* h_x, void\* stream\);", text)
    L = api.lib()
    assert L.az_nn_create_planes.argtypes == [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    assert L.az_nn_input_planes.argtypes == [C.c_void_p] and L.az_nn_input_planes.restype == C.c_int
    assert L.az_env6_encode_planes.argtypes == [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]


def test_nn_planes_is_nn_oracle_at_13_planes(golden_dir):
    """forward, train_losses and a Trainer step at 13 planes: bit for bit nn_oracle's, and the golden forward vectors"""
    sl = go.load_slice()
    g = np.load(os.path.join(golden_dir, "graph_forward_V2_5.npz"))
    w = go.golden_weights(sl, int(g["seed"]))
    pr, vr = npl.forward(w, g["x"], 5, dtype=torch.float64)
    assert np.abs(pr - g["policy"]).max() < 1e-12 and np.abs(vr - g["value"]).max() < 1e-12
    for dtype in (torch.float64, torch.float32):
        p0, v0 = no.forward(w, g["x"], 5, dtype=dtype)
        p1, v1 = npl.forward(w, g["x"], 5, dtype=dtype)
        assert (p0 == p1).all() and (v0 == v1).all()
    rng = np.random.default_rng(13)
    tp = rng.random((len(g["x"]), 43)); tp /= tp.sum(1, keepdims=True)
    tv = rng.choice([1.0, -1.0, 0.0], len(g["x"]))
    a, b = no.Trainer(w, 5), npl.Trainer(w, 5)
    assert a.step(g["x"], tp, tv) == b.step(g["x"], tp, tv)
    wa, wb = a.weights(), b.weights()
    assert all((wa[k] == wb[k]).all() for k in wa) and all((a.grads[k] == b.grads[k]).all() for k in a.grads)
    assert no.train_losses is not npl.train_losses            # the 13-plane loss is restored after the step


def map_to_16(w13):
    """W16[..., 0] = W13[..., 0], W16[..., 1] = W13[..., 1], W16[..., 2..5] = W13[..., 2], W16[..., 6..15] = W13[..., 3..12]"""
    k = w13["conv/kernel"]
    w16 = dict(w13)
    w16["conv/kernel"] = np.concatenate([k[:, :, :2], np.repeat(k[:, :, 2:3], 4, axis=2), k[:, :, 3:]], axis=2)
    return w16


def test_mapped_network_is_the_13_plane_function():
    """on positions where all six seats own land, a 13-plane network and its 16-plane mapping compute the same outputs (fp64), in the
    forward and in the training losses"""
    sl = go.load_slice()
    w13 = go.golden_weights(sl, 5)
    w16 = map_to_16(w13)
    assert w16["conv/kernel"].shape == (3, 3, 16, 256)
    o, x13, x16 = po.Oracle6Game(), [], []
    for img in rollout_positions(n_games=2, every=29):
        o.set_image(img)
        if len(set(int(v) for v in o.s.owner)) == 6:
            x13.append(planes6.encode13(o)); x16.append(planes6.encode16(o))
    assert len(x13) >= 20
    x13, x16 = np.array(x13), np.array(x16)
    p13, v13 = npl.forward(w13, x13, 5, dtype=torch.float64)
    p16, v16 = npl.forward(w16, x16, 5, dtype=torch.float64)
    assert np.abs(p13 - p16).max() < 1e-12 and np.abs(v13 - v16).max() < 1e-12
    tp = np.full((len(x13), 43), 1.0 / 43)
    tv = np.zeros(len(x13))
    losses = []
    for w, x in ((w13, x13), (w16, x16)):
        t = {k: torch.as_tensor(np.asarray(v), dtype=torch.float64) for k, v in w.items()}
        lp, lv, _ = npl.train_losses(t, torch.as_tensor(x, dtype=torch.float64), torch.as_tensor(tp), torch.as_tensor(tv), 5, {})
        losses.append((float(lp), float(lv)))
    assert abs(losses[0][0] - losses[1][0]) < 1e-12 and abs(losses[0][1] - losses[1][1]) < 1e-12
