"""CPU suite: the network restatement (oracle/nn_oracle.py, the checker of the CUDA forward) against the reference's own shipped
GraphDef.  tests/golden/graph_V2_5_inference.json is the inference slice of python/model/model_txt_V2_5.pb (extracted by
tests/golden/gen_graph_slice.py); oracle/graphdef_oracle.py executes it op by op.  The TensorFlow kernels behind the ops are restated
(un-vendored dependency), everything else — wiring, variables, shapes, data formats, epsilon, the inference branch of every
BatchNorm — is the reference's artifact."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import graphdef_oracle as go
from oracle import nn_oracle as no

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.environ.get("AZ_REFERENCE_DIR")          # a checkout of the original project, as oracle/ref/build_ref.sh reads it
REF_PB = os.path.join(REF_DIR, "python", "model", "model_txt_V2_5.pb") if REF_DIR else ""


@pytest.fixture(scope="module")
def sl():
    return go.load_slice()


def test_slice_reads_exactly_the_variables_of_the_restatement(sl, golden_dir):
    got = dict(go.variables(sl))
    assert sorted(got) == sorted(no.variable_names(5))
    inv = json.load(open(os.path.join(golden_dir, "ckpt_tensors_V2_5.json")))          # the Saver's inventory of the same GraphDef
    shapes = {name: tuple(shape) for name, shape in inv["tensors"]}
    for name, shape in got.items():
        assert shapes[name] == shape, name
    assert got["conv/kernel"] == (3, 3, 13, 256) and got["conv_bn/gamma"] == (7,) and got["dense/kernel"] == (84, 43)
    assert got["dense_1/kernel"] == (42, 256) and got["pi/kernel"] == (1, 1, 256, 2) and got["v/kernel"] == (1, 1, 256, 1)


def test_structural_facts_the_cuda_path_relies_on(sl):
    bns = [n for n in sl["nodes"] if n["op"] == "FusedBatchNormV3"]
    assert len(bns) == 13
    for n in bns:
        stem = n["name"].startswith("conv_bn/")
        assert n["attr"]["data_format"]["s"] == ("NCHW" if stem else "NHWC")        # the stem normalises over the board-row axis
        assert n["attr"]["is_training"]["b"] is False
        assert np.float32(n["attr"]["epsilon"]["f"]) == np.float32(0.001)
    convs = [n for n in sl["nodes"] if n["op"] == "Conv2D"]
    assert len(convs) == 13 and all(n["attr"]["padding"]["s"] == "SAME" and n["attr"]["data_format"]["s"] == "NHWC" for n in convs)
    ifs = [n for n in sl["nodes"] if n["op"] == "IfElseOutput"]
    assert len(ifs) == 13                                                            # every BatchNorm branches on input_training
    assert sum(n["op"] == "Add" for n in sl["nodes"]) == 5 and sum(n["op"] == "Relu" for n in sl["nodes"]) == 14


def test_restatement_equals_the_graphdef(sl):
    for seed, n in ((1, 3), (2, 9)):
        w = go.golden_weights(sl, seed)
        x = np.random.default_rng(100 + seed).random((n, 7, 6, 13)).astype(np.float32)
        p, v = go.run(sl, w, x)
        pr, vr = no.forward(w, x, 5, dtype=torch.float64)
        assert np.abs(p - pr).max() < 1e-12 and np.abs(v - vr).max() < 1e-12
        p32, v32 = no.forward(w, x, 5, dtype=torch.float32)
        assert np.abs(p - p32).max() < 1e-5 and np.abs(v - v32).max() < 1e-5


def test_golden_forward_vectors(sl, golden_dir):
    g = np.load(os.path.join(golden_dir, "graph_forward_V2_5.npz"))
    w = go.golden_weights(sl, int(g["seed"]))
    p, v = go.run(sl, w, g["x"])
    assert np.abs(p - g["policy"]).max() < 1e-12 and np.abs(v - g["value"]).max() < 1e-12
    pr, vr = no.forward(w, g["x"], 5, dtype=torch.float32)
    assert np.abs(pr - g["policy"]).max() < 1e-5 and np.abs(vr - g["value"]).max() < 1e-5
    assert np.allclose(g["policy"].sum(1), 1.0, atol=1e-12) and g["policy"].std(0).max() > 1e-3


def test_training_forward_of_the_graphdef_equals_the_restatement(sl):
    """input_training = true: the two losses, the minimised total (add_6 = loss_pi + loss_v + total_regularization_loss) and the amount
    every moving statistic is decreased by, evaluated from the reference's own nodes, against nn_oracle.train_losses.  The optimizer
    differentiates exactly this forward (tf.gradients of add_6), so pinning it pins what nn_oracle.Trainer's autograd differentiates."""
    ts = go.load_slice(go.TRAINING_SLICE)
    upd = ts["moving_average_updates"]
    assert len(upd) == 26 and ts["adam"]["minimised"] == "add_6"
    for seed, n in ((5, 6), (6, 17)):
        w = go.golden_weights(sl, seed)
        rng = np.random.default_rng(seed)
        x = rng.random((n, 7, 6, 13)).astype(np.float32)
        tp = rng.random((n, 43))
        tp /= tp.sum(1, keepdims=True)
        tv = rng.choice([-1.0, 0.0, 1.0], n)
        out = go.run(ts, w, x, training=True, targets=(tp, tv),
                     fetch=["softmax_cross_entropy_loss/value", "mean_squared_error/value", "add_6"] + [u[1] for u in upd])
        wt = {k: torch.as_tensor(v, dtype=torch.float64) for k, v in w.items()}
        stats = {}
        lp, lv, l2 = no.train_losses(wt, torch.as_tensor(x, dtype=torch.float64), torch.as_tensor(tp), torch.as_tensor(tv), 5, stats)
        assert abs(float(out[0]) - float(lp)) < 1e-11 and abs(float(out[1]) - float(lv)) < 1e-11
        assert abs(float(out[2]) - float(lp + lv + l2)) < 1e-11
        for (var, _), val in zip(upd, out[3:]):
            prefix, which = var.rsplit("/", 1)
            mean, var_unbiased = stats[prefix]
            target = (mean if which == "moving_mean" else var_unbiased).numpy()
            ref = (w[var].astype(np.float64) - target) * (1.0 - no.BN_MOMENTUM)          # Trainer.step: moving -= (moving - batch) * (1 - momentum)
            assert np.abs(val - ref).max() < 1e-12, var


def test_optimizer_wiring_and_constants(sl):
    """the 45 ResourceApplyAdam ops of the graph: which variables they update, their slots, hyper-parameters and beta-power inputs"""
    ts = go.load_slice(go.TRAINING_SLICE)
    ad = ts["adam"]
    assert ad["variables"] == sorted(no.trainable_names(5)) and len(ad["variables"]) == 45
    assert np.float32(ad["learning_rate"]) == np.float32(no.ADAM["lr"]) and np.float32(ad["beta1"]) == np.float32(no.ADAM["beta1"])
    assert np.float32(ad["beta2"]) == np.float32(no.ADAM["beta2"]) and np.float32(ad["epsilon"]) == np.float32(no.ADAM["eps"])
    assert ad["use_nesterov"] is False and ad["slots"] == ["<variable>/optimize", "<variable>/optimize_1"]
    regularised = sorted(n["name"].split("/Regularizer/")[0] for n in ts["nodes"] if n["name"].endswith("/Regularizer/Square"))
    assert regularised == sorted(n for n in no.variable_names(5) if n.endswith("/kernel")) and len(regularised) == 16


@pytest.mark.skipif(not os.path.exists(REF_PB), reason="AZ_REFERENCE_DIR does not name a checkout of the original project")
def test_committed_slices_are_what_the_extractor_produces(tmp_path, golden_dir):
    a, b = str(tmp_path / "inference.json"), str(tmp_path / "training.json")
    subprocess.check_call([sys.executable, os.path.join(golden_dir, "gen_graph_slice.py"), REF_PB, a, b], stdout=subprocess.DEVNULL)
    assert json.load(open(a)) == json.load(open(os.path.join(golden_dir, "graph_V2_5_inference.json")))
    assert json.load(open(b)) == json.load(open(os.path.join(golden_dir, "graph_V2_5_training.json")))
