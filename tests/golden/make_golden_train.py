"""Fixtures that pin oracle/train_oracle.py (and, on the GPU box, csrc/train.cu) to the reference's own loss class.

Needs a checkout of the reference: imports libs/ft.py's WeightedL2Loss2d through the
`galerkin_transformer` alias package (which stubs the plotting imports), evaluates it on seeded inputs the way
train_batch_darcy does (libs/utils_ft.py:672-674: loss_func(u_pred, u, targets_prime=gradu, K=a)), and records the
outputs and the autograd gradients of the loss and of the regulariser w.r.t. preds in tests/golden/train/<case>.pt.

    GALERKIN_REFERENCE=/path/to/reference python tests/golden/make_golden_train.py"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from galerkin_transformer import load_reference_module                         # noqa: E402

CASES = [dict(name="loss_h1_k", B=3, n=17, regularizer=True, gamma=0.5, use_K=True, use_tp=True, dilation=2, return_norm=True),
         dict(name="loss_l2_only", B=2, n=12, regularizer=False, gamma=0.1, use_K=False, use_tp=False, dilation=2, return_norm=True),
         dict(name="loss_h1_dil4_mean", B=2, n=21, regularizer=True, gamma=0.1, use_K=True, use_tp=True, dilation=4, return_norm=False),
         dict(name="loss_h1_nok", B=4, n=33, regularizer=True, gamma=0.1, use_K=False, use_tp=True, dilation=2, return_norm=True)]


def main():
    ft = load_reference_module("ft")
    assert ft is not None, "set GALERKIN_REFERENCE to the root of a checkout of the reference"
    os.makedirs(os.path.join(HERE, "train"), exist_ok=True)
    for i, c in enumerate(CASES):
        g = torch.Generator().manual_seed(4100 + i)
        B, n = c["B"], c["n"]
        h = 1.0 / n
        targets = torch.randn(B, n, n, generator=g)
        preds = (targets + 0.3 * torch.randn(B, n, n, generator=g)).requires_grad_(True)
        tp = torch.randn(B, n, n, 2, generator=g) * 3.0 if c["use_tp"] else None
        K = (0.5 + torch.rand(B, n, n, 1, generator=g)) if c["use_K"] else None
        lf = ft.WeightedL2Loss2d(regularizer=c["regularizer"], h=h, gamma=c["gamma"], dilation=c["dilation"],
                                 return_norm=c["return_norm"])
        loss, reg, metric, _ = lf(preds, targets, targets_prime=tp, K=K)
        dloss, = torch.autograd.grad(loss, preds, retain_graph=True)
        if c["regularizer"] and tp is not None:
            dreg, = torch.autograd.grad(reg, preds)
        else:
            dreg = torch.zeros_like(preds)
        fix = dict(case=c, h=h, preds=preds.detach(), targets=targets, targets_prime=tp, K=K, loss=loss.detach().reshape(()),
                   reg=reg.detach().reshape(()), metric=float(metric), dloss=dloss, dreg=dreg)
        torch.save(fix, os.path.join(HERE, "train", c["name"] + ".pt"))
        print(c["name"], float(loss), float(reg), float(metric))


if __name__ == "__main__":
    main()
