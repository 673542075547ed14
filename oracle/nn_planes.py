"""TEST INFRASTRUCTURE — oracle/nn_oracle.py's restatement of the network for any input plane count: 13 (the reference graph) or the 16
six-player seat planes (SIXPLAYER.md §2, "seat planes"), read from conv/kernel's third dimension.  Everything but the input's reshape is
nn_oracle's own code: its BatchNorm, convolution (with the bf16 contraction mode) and trace helpers here, its Adam step in Trainer.
At 13 planes forward() and train_losses() compute what nn_oracle.forward() and nn_oracle.train_losses() compute.
Only tests/ may import it."""
from unittest import mock

import numpy as np
import torch

from oracle import nn_oracle as no


def planes(weights):
    return int(weights["conv/kernel"].shape[2])


def forward(weights, x, blocks, dtype=torch.float32):
    """nn_oracle.forward with the input [n, 7, 6, P], P = conv/kernel's input channels"""
    w = {k: torch.as_tensor(np.asarray(v), dtype=dtype) for k, v in weights.items()}
    t = torch.as_tensor(np.asarray(x), dtype=dtype).reshape(-1, 7, 6, planes(w)).permute(0, 3, 1, 2)   # NCHW: [n,P,7,6]
    t = no._conv(t, w["conv/kernel"])
    t = torch.relu(no._bn(t, w, "conv_bn", axis=2))
    for i in range(blocks):
        sfx = "%d%s" % (i, chr(ord("a") + i))
        r = torch.relu(no._bn(no._conv(t, w["res%s_branch2a/kernel" % sfx]), w, "bn%s_branch2a" % sfx, axis=1))
        r = no._bn(no._conv(r, w["res%s_branch2b/kernel" % sfx]), w, "bn%s_branch2b" % sfx, axis=1)
        t = torch.relu(r + t)
    p = torch.relu(no._bn(no._conv(t, w["pi/kernel"]), w, "bn_pi", axis=1))
    p = p.permute(0, 2, 3, 1).reshape(-1, 84)
    policy = torch.softmax(p @ w["dense/kernel"] + w["dense/bias"], dim=1)
    v = torch.relu(no._bn(no._conv(t, w["v/kernel"]), w, "bn_v", axis=1))
    v = v.permute(0, 2, 3, 1).reshape(-1, 42)
    v = torch.relu(v @ w["dense_1/kernel"] + w["dense_1/bias"])
    v = torch.tanh(v @ w["dense_2/kernel"] + w["dense_2/bias"]).reshape(-1)
    return policy.numpy(), v.numpy()


def train_losses(w, x, target_policy, target_value, blocks, batch_stats):
    """nn_oracle.train_losses with the input [n, 7, 6, P], P = conv/kernel's input channels"""
    t = x.reshape(-1, 7, 6, planes(w)).permute(0, 3, 1, 2)
    t = torch.relu(no._bn_train(no._conv(t, w["conv/kernel"]), w, "conv_bn", 2, batch_stats))
    for i in range(blocks):
        sfx = "%d%s" % (i, chr(ord("a") + i))
        r = torch.relu(no._bn_train(no._conv(t, w["res%s_branch2a/kernel" % sfx]), w, "bn%s_branch2a" % sfx, 1, batch_stats))
        r = no._bn_train(no._conv(r, w["res%s_branch2b/kernel" % sfx]), w, "bn%s_branch2b" % sfx, 1, batch_stats)
        t = torch.relu(r + t)
    p = torch.relu(no._bn_train(no._conv(t, w["pi/kernel"]), w, "bn_pi", 1, batch_stats))
    logits = p.permute(0, 2, 3, 1).reshape(-1, 84) @ w["dense/kernel"] + w["dense/bias"]
    loss_pi = -(target_policy * torch.log_softmax(logits, dim=1)).sum(dim=1).mean()
    v = torch.relu(no._bn_train(no._conv(t, w["v/kernel"]), w, "bn_v", 1, batch_stats))
    v = torch.relu(v.permute(0, 2, 3, 1).reshape(-1, 42) @ w["dense_1/kernel"] + w["dense_1/bias"])
    v = torch.tanh(v @ w["dense_2/kernel"] + w["dense_2/bias"]).reshape(-1)
    loss_v = ((v - target_value) ** 2).mean()
    l2 = sum((w[n] ** 2).sum() for n in w if n.endswith("/kernel")) * no.L2_C
    return loss_pi, loss_v, l2


class Trainer(no.Trainer):
    """nn_oracle.Trainer (the graph's variables, Adam slots, moving statistics) with the loss of train_losses above: its step() is
    nn_oracle's, run with this module's train_losses in place of the 13-plane one"""

    def step(self, x, target_policy, target_value):
        with mock.patch.object(no, "train_losses", train_losses):
            return super().step(x, target_policy, target_value)
