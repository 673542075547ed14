"""CPU checks of the six-seat value vector (SIXPLAYER.md §2) on the oracle (oracle/risk6_vector.c): with an evaluator that spreads the
scalar rule into a vector, [v, -v/5, ..., -v/5], the vector search is the scalar lockstep search (oracle/risk6_lockstep.c) bit for bit;
with the pseudo6 evaluator every simulation is backed up, no active_N mark is left and the root Q differs from the scalar search's.
The Python binding's new constants and signatures agree with the C header."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import pyoracle as po
from oracle.lockstep6 import Lockstep6Mcts
from oracle.vector6 import EVAL6_CB, Vector6Mcts, lib, pseudo6

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 0x5EED0061


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def scalar_pseudo():
    """r6_eval_pseudo of the vector oracle's library (risk6_oracle.c's own evaluator)"""
    f = lib().r6_eval_pseudo
    f.argtypes = [C.POINTER(po.R6State), C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p]
    return f


@EVAL6_CB
def spread_eval(sp, policy, value, user):
    """r6_eval_pseudo's policy and value v, spread as [v, -v/5, ..., -v/5] (-v/5 a correctly rounded float division)"""
    v = C.c_float(0)
    scalar_pseudo()(sp, policy, C.byref(v), None)
    value[0] = v.value
    other = np.float32(-np.float32(v.value)) / np.float32(5.0)
    for k in range(1, 6):
        value[k] = float(other)


def positions(rules, n_games=6, every=23, plies=600):
    out = []
    for g in range(n_games):
        o = po.Oracle6Game(rules)
        o.new_game(SEED, g, 0)
        for ply in range(plies):
            if o.status() != -1:
                break
            if ply % every == 0:
                out.append((g, ply, o.image()))
            assert o.move(o.random_action(SEED, g, ply), SEED, g, ply) == 0
    return out


def test_pseudo6_component0_is_the_scalar_value():
    rules = po.default_rules()
    differ = 0
    for g, ply, img in positions(rules, n_games=2, every=37):
        o = po.Oracle6Game(rules)
        o.set_image(img)
        p6, v6 = pseudo6(o)
        p, v = np.zeros(43, np.float32), C.c_float(0)
        scalar_pseudo()(C.byref(o.s), p.ctypes.data_as(C.POINTER(C.c_float)), C.byref(v), None)
        assert (bits(p6) == bits(p)).all() and bits(v6[:1])[0] == bits(np.float32([v.value]))[0]
        assert ((v6 * 128).astype(np.int64) == v6 * 128).all() and (np.abs(v6) <= 1).all()    # dyadic, like az_pn_value
        differ += int((v6[1:] != -v6[0] / 5).any())
    assert differ > 0


@pytest.mark.parametrize("K,sims", [(1, 16), (2, 16), (4, 32), (8, 32), (16, 48)])
def test_spread_vector_equals_scalar_lockstep(K, sims):
    rules = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    pos = positions(rules)
    assert len(pos) >= 60
    vec, sca = Vector6Mcts(rules, spread_eval), Lockstep6Mcts(rules)
    for g, ply, img in pos:
        o = po.Oracle6Game(rules)
        o.set_image(img)
        a = vec.search(o, SEED, g, ply, lockstep=K)
        b = sca.search(o, SEED, g, ply, lockstep=K)
        assert (a["N"] == b["N"]).all(), (g, ply)
        for k in ("Q", "P", "pi"):
            assert (bits(a[k]) == bits(b[k])).all(), (k, g, ply)
        assert a["sumN"] == b["sumN"] == sims and bits(np.float32([a["value"]]))[0] == bits(np.float32([b["value"]]))[0]
        assert vec.table_size() == sca.table_size() and vec.active_total() == 0


@pytest.mark.parametrize("K", [1, 4, 16])
def test_pseudo6_backs_up_every_simulation(K):
    sims = 48
    rules = po.default_rules(mcts_simulations=sims, threads_per_mcts=1)
    vec, sca = Vector6Mcts(rules), Lockstep6Mcts(rules)
    q_differs = 0
    for g, ply, img in positions(rules):
        o = po.Oracle6Game(rules)
        o.set_image(img)
        a = vec.search(o, SEED, g, ply, lockstep=K)
        b = sca.search(o, SEED, g, ply, lockstep=K)
        assert a["sumN"] == sims and int(a["N"].sum()) == sims and vec.active_total() == 0
        assert bits(np.float32([a["value"]]))[0] == bits(np.float32([b["value"]]))[0]     # the stored value is component 0
        assert (bits(a["P"]) == bits(b["P"])).all()
        q_differs += int((bits(a["Q"]) != bits(b["Q"])).any())
    assert q_differs > 0
    if K > 1:
        assert vec.vl_skips() > 0


def test_vector_search_rejects_k_not_dividing():
    rules = po.default_rules(mcts_simulations=16, threads_per_mcts=1)
    o = po.Oracle6Game(rules)
    o.new_game(SEED, 0, 0)
    rc, _ = Vector6Mcts(rules).search_rc(o, SEED, 0, 0, 3)
    assert rc != 0


def test_binding_agrees_with_header():
    from alphazero_risk_b200 import api
    text = open(os.path.join(ROOT, "include", "az_b200.h")).read()
    consts = dict((k, int(v)) for k, v in re.findall(r"#define (AZ_EVAL_\w+)\s+(\d+)", text))
    assert consts["AZ_EVAL_PSEUDO6"] == api.EVAL_PSEUDO6 == 3
    assert (consts["AZ_EVAL_NN"], consts["AZ_EVAL_PSEUDO"], consts["AZ_EVAL_UNIFORM"]) == (api.EVAL_NN, api.EVAL_PSEUDO, api.EVAL_UNIFORM)
    assert re.search(r"AZ_API int az_nn_create_value\(int blocks, int value_outputs, int device, az_nn\*\* out\);", text)
    assert re.search(r"AZ_API int az_nn_value_outputs\(const az_nn\* nn\);", text)
    L = api.lib()
    assert L.az_nn_create_value.argtypes == [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
    assert L.az_nn_value_outputs.argtypes == [C.c_void_p] and L.az_nn_value_outputs.restype == C.c_int
