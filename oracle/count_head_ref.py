"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the instance-count branch of isa_b200.archs.ReSeg(count_head=True).

The reference tree has no code for this branch (reseg.py:13-40 names a count head; the shipped tree never builds it),
so this is not reference code: it restates this project's own layer list with stock torch modules, and is the oracle
the kernels and the wired branch are compared against.

    ins_cls_cnn:  max_pool2d 2x2 -> conv1 3x3 C->64 +ReLU -> conv2 3x3 +ReLU -> max_pool2d 2x2 -> conv3 3x3 +ReLU
                  -> conv4 3x3 +ReLU
    ins_cls_out:  AdaptiveAvgPool2d(1) -> linear 64->1 -> sigmoid = s
    loss = MSELoss(s, n_objects / K);   n_pred = clamp(round(s * K), 1, K)  (round half to even)

Parameter names match the product's (`ins_cls_cnn.conv{1..4}`, `ins_cls_out.linear`), so one state_dict loads into both.
"""
from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F


class CountBranchRef(nn.Module):
    def __init__(self, n_input=224, n_filters=64):
        super().__init__()
        self.ins_cls_cnn = nn.Sequential(OrderedDict([
            ("pool1", nn.MaxPool2d(2, 2)),
            ("conv1", nn.Conv2d(n_input, n_filters, 3, padding=1)), ("relu1", nn.ReLU()),
            ("conv2", nn.Conv2d(n_filters, n_filters, 3, padding=1)), ("relu2", nn.ReLU()),
            ("pool2", nn.MaxPool2d(2, 2)),
            ("conv3", nn.Conv2d(n_filters, n_filters, 3, padding=1)), ("relu3", nn.ReLU()),
            ("conv4", nn.Conv2d(n_filters, n_filters, 3, padding=1)), ("relu4", nn.ReLU()),
        ]))
        self.ins_cls_out = nn.Sequential(OrderedDict([
            ("gap", nn.AdaptiveAvgPool2d(1)), ("flatten", nn.Flatten()), ("linear", nn.Linear(n_filters, 1)),
        ]))

    def forward(self, y):
        """y (N, C, H/4, W/4) -> (conv4 output after ReLU, pooled (N, 64), s (N,))."""
        f = self.ins_cls_cnn(y)
        pooled = F.adaptive_avg_pool2d(f, 1).flatten(1)
        s = torch.sigmoid(self.ins_cls_out(f)).reshape(-1)
        return f, pooled, s


def tail(y, w, b):
    """The fused tail from the (already ReLU'd) conv4 output y (N, C, H, W): -> (pooled (N, C), s (N,))."""
    pooled = nn.AdaptiveAvgPool2d(1)(y).flatten(1)
    s = torch.sigmoid(F.linear(pooled, w.reshape(1, -1), b.reshape(1))).reshape(-1)
    return pooled, s


def count_loss(s, n_objects, K):
    return nn.MSELoss()(s, torch.as_tensor(n_objects, dtype=s.dtype) / K)


def n_pred(s, K):
    return torch.round(s * K).clamp(1, K).to(torch.int32)


def tail_grad(y, pooled, s, w, n_objects, K, grad_loss=1.0):
    """Hand-written gradient of count_loss(tail(relu(x + conv_bias))) -> (gx, dconv_bias, dw, db), with gx the gradient
    of the PRE-ReLU conv4 output x (y = relu(x + conv_bias) given); every argument a float64 tensor."""
    n, C, H, W = y.shape
    t = torch.as_tensor(n_objects, dtype=s.dtype) / K
    dz = grad_loss * 2.0 * (s - t) / n * s * (1.0 - s)                     # (N,)
    gx = (y > 0).to(y.dtype) * (dz.view(n, 1, 1, 1) * w.reshape(1, C, 1, 1) / (H * W))
    return gx, gx.sum((0, 2, 3)), (dz.view(n, 1) * pooled).sum(0), dz.sum().reshape(1)
