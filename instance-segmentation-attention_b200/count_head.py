"""The tail of the instance-count branch of `archs.ReSeg(count_head=True)` (csrc/count_head.cu through the C-ABI):

    y = relu(conv4(x) + conv4.bias)   pooled = mean over H, W   s = sigmoid(linear(pooled))
    n_pred = clamp(round(s * K), 1, K)        loss = mean_b (s_b - n_objects_b / K)^2

conv4 itself runs bias-free on cuDNN; everything after it is one fused forward and one streaming backward.  Only `loss` is
differentiable; `y`, `pooled`, `s` and `n_pred` are returned for inspection and prediction.
"""
import collections

import torch
import torch.nn.functional as F

from . import _lib

CountOutput = collections.namedtuple("CountOutput", ["loss", "s", "n_pred", "pooled", "y"])


def _tail_fwd(z, conv_bias, w, b, n_objects, K, want_loss):
    """Runs isa_count_head_fwd over the bias-free conv4 output z (NHWC-dense, finished in place) -> (loss or None, s,
    n_pred, pooled, workspace)."""
    lib = _lib.load()
    n, C, H, W = z.shape
    P = H * W
    dev = z.device
    pooled = torch.empty(n, C, device=dev, dtype=torch.float32)
    s = torch.empty(n, device=dev, dtype=torch.float32)
    n_pred = torch.empty(n, device=dev, dtype=torch.int32)
    loss = torch.empty((), device=dev, dtype=torch.float32) if want_loss else None
    wsb = lib.isa_count_head_workspace_bytes(n, P, C)
    ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
    rc = lib.isa_count_head_fwd(z.data_ptr(), _lib.ptr(conv_bias), _lib.ptr(w), _lib.ptr(b), _lib.ptr(n_objects), n, P, C, K,
                                pooled.data_ptr(), s.data_ptr(), n_pred.data_ptr(), _lib.ptr(loss), ws.data_ptr(), wsb,
                                _lib.stream_ptr(dev))
    _lib.check(rc, "isa_count_head_fwd")
    return loss, s, n_pred, pooled, ws


class _CountTailFn(torch.autograd.Function):
    """loss of the count branch from conv3's output x: the bias-free cuDNN conv4, then isa_count_head_fwd; backward
    isa_count_head_bwd, then the library's convolution backward."""

    @staticmethod
    def forward(ctx, x, w4, b4, w, b, n_objects, K, padding):
        z = F.conv2d(x, w4, None, 1, padding).contiguous(memory_format=torch.channels_last)
        loss, s, n_pred, pooled, ws = _tail_fwd(z, b4, w, b, n_objects, K, True)
        ctx.save_for_backward(x, w4, w, n_objects, z, pooled, s, ws)
        ctx.K, ctx.padding = K, padding
        ctx.mark_non_differentiable(s, n_pred, pooled, z)
        return loss, s, n_pred, pooled, z

    @staticmethod
    def backward(ctx, g_loss, _gs, _gn, _gp, _gz):
        lib = _lib.load()
        x, w4, w, n_objects, y, pooled, s, ws = ctx.saved_tensors
        n, C, H, W = y.shape
        gl = g_loss.reshape(1).contiguous()
        gx = torch.empty_like(y)
        dconv_bias = torch.empty(C, device=y.device, dtype=torch.float32)
        dw = torch.empty(C, device=y.device, dtype=torch.float32)
        db = torch.empty(1, device=y.device, dtype=torch.float32)
        rc = lib.isa_count_head_bwd(y.data_ptr(), pooled.data_ptr(), s.data_ptr(), w.data_ptr(), n_objects.data_ptr(),
                                    gl.data_ptr(), n, H * W, C, ctx.K, gx.data_ptr(), dconv_bias.data_ptr(), dw.data_ptr(),
                                    db.data_ptr(), ws.data_ptr(), ws.numel(), _lib.stream_ptr(y.device))
        _lib.check(rc, "isa_count_head_bwd")
        p = list(ctx.padding)
        g_in, g_w4, _ = torch.ops.aten.convolution_backward(gx, x, w4, None, [1, 1], p, [1, 1], False, [0, 0], 1,
                                                            [ctx.needs_input_grad[0], ctx.needs_input_grad[1], False])
        return g_in, g_w4, dconv_bias, dw, db, None, None, None


def count_tail(x, conv4, linear, K, n_objects=None):
    """CountOutput of the branch tail from conv3's output x (N, C, h, w) NHWC-dense: conv4 (nn.Conv2d C -> C', stride 1),
    global average pool, linear (nn.Linear C' -> 1), sigmoid.  n_objects (N,) integer targets or None: with targets the
    loss is computed (and differentiable), without it `loss` is None."""
    _lib.require_cuda(x, "activation")
    K = int(K)
    w = linear.weight.reshape(-1).contiguous()
    if n_objects is None:
        with torch.no_grad():
            z = F.conv2d(x, conv4.weight, None, 1, conv4.padding).contiguous(memory_format=torch.channels_last)
            _, s, n_pred, pooled, _ = _tail_fwd(z, conv4.bias.contiguous(), w, linear.bias.contiguous(), None, K, False)
        return CountOutput(None, s, n_pred, pooled, z)
    nobj = n_objects.to(device=x.device, dtype=torch.int32).reshape(-1).contiguous()
    loss, s, n_pred, pooled, y = _CountTailFn.apply(x, conv4.weight, conv4.bias, w, linear.bias, nobj, K,
                                                    tuple(conv4.padding))
    return CountOutput(loss, s, n_pred, pooled, y)
