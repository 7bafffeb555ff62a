"""Channels-last epilogues of the embedding network and the residual + LayerNorm of the attention block
(csrc/pointwise.cu through the C-ABI).

  ConvBiasAct / ConvTransposeBiasAct   nn.Conv2d / nn.ConvTranspose2d (same parameter names, so state_dicts
        interchange with stock layers) whose bias add and optional ReLU run as ONE in-place pass over the bias-free
        cuDNN output, and whose backward produces the masked gradient and the bias gradient in ONE pass
        (/root/reference/code/lib/archs/modules/vgg16.py:82-140 conv+ReLU stacks; reseg.py:117-121).
  add_layer_norm                      MultiHeadAttention's layer_norm(output + residual)
        (/root/reference/code/lib/archs/modules/utils.py:218-219).
  pixel_heads                         the semantic + embedding 1x1 heads over [features | skip] as ONE pass from NHWC
        sources to NCHW planes, no concatenation (reseg.py:122-126).
  thin_linear                         nn.Linear arithmetic for the attention projections (utils.py:177-179, 189) whose
        weight gradient (out x in = 24 x 24 from 65 536 rows) is a split-K batched GEMM instead of the single-CTA
        SIMT sgemm the library picks for that shape.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib


def _rows_c(t):
    """(rows, C) of an NHWC-dense 4-d tensor or a contiguous (..., C) matrix, or None if the layout is not token-major."""
    if t.dim() == 4:
        if t.is_contiguous(memory_format=torch.channels_last):
            return t.numel() // t.shape[1], t.shape[1]
        return None
    if t.is_contiguous():
        return t.numel() // t.shape[-1], t.shape[-1]
    return None


class _BiasActFn(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x, bias, relu):
        lib = _lib.load()
        rows, C = _rows_c(x)
        rc = lib.isa_bias_act_fwd(x.data_ptr(), _lib.ptr(bias.contiguous()), rows, C, int(relu), _lib.stream_ptr(x.device))
        _lib.check(rc, "isa_bias_act_fwd")
        ctx.mark_dirty(x)
        ctx.relu = bool(relu)
        ctx.geom = (rows, C)
        if relu:
            ctx.save_for_backward(x)
        return x

    @staticmethod
    def backward(ctx, gy):
        lib = _lib.load()
        rows, C = ctx.geom
        y = ctx.saved_tensors[0] if ctx.relu else None
        gy = gy.contiguous(memory_format=torch.channels_last) if gy.dim() == 4 else gy.contiguous()
        db = torch.empty(C, device=gy.device, dtype=torch.float32)
        wsb = lib.isa_bias_act_workspace_bytes(C)
        ws = torch.empty(wsb, device=gy.device, dtype=torch.uint8)
        gx = torch.empty_like(gy) if ctx.relu else gy
        rc = lib.isa_bias_act_bwd(gy.data_ptr(), y.data_ptr() if y is not None else None, gx.data_ptr() if ctx.relu else None,
                                  db.data_ptr(), rows, C, int(ctx.relu), ws.data_ptr(), wsb, _lib.stream_ptr(gy.device))
        _lib.check(rc, "isa_bias_act_bwd")
        return gx, db, None


class _ConvBiasReluFn(torch.autograd.Function):
    """relu(conv2d(x, w) + b) with the bias + ReLU inside cuDNN's convolution epilogue (forward: no pass over the output
    at all, bit-identical to the convolution followed by the in-place epilogue kernel, measured on B200: 3x3 convolutions
    of the backbone 129-145 us fused against 218-220 us unfused at 16 x 64 x 256^2); backward: the single-pass
    masked-gradient + bias-gradient kernel (isa_bias_act_bwd) in front of the library's convolution backward."""

    @staticmethod
    def forward(ctx, x, w, b, stride, padding, dilation, groups):
        y = torch.cudnn_convolution_relu(x, w, b, stride, padding, dilation, groups)
        ctx.conf = (stride, padding, dilation, groups)
        ctx.save_for_backward(x, w, y)
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _lib.load()
        x, w, y = ctx.saved_tensors
        stride, padding, dilation, groups = ctx.conf
        if not y.is_contiguous(memory_format=torch.channels_last):
            gm = gy * (y > 0)
            db = gm.sum((0, 2, 3))
        else:
            rows, C = _rows_c(y)
            gy = gy.contiguous(memory_format=torch.channels_last)
            db = torch.empty(C, device=gy.device, dtype=torch.float32)
            wsb = lib.isa_bias_act_workspace_bytes(C)
            ws = torch.empty(wsb, device=gy.device, dtype=torch.uint8)
            gm = torch.empty_like(gy)
            rc = lib.isa_bias_act_bwd(gy.data_ptr(), y.data_ptr(), gm.data_ptr(), db.data_ptr(), rows, C, 1, ws.data_ptr(), wsb,
                                      _lib.stream_ptr(gy.device))
            _lib.check(rc, "isa_bias_act_bwd")
        gx, gw, _ = torch.ops.aten.convolution_backward(gm, x, w, None, list(stride), list(padding), list(dilation), False, [0, 0], groups,
                                                        [ctx.needs_input_grad[0], ctx.needs_input_grad[1], False])
        return gx, gw, db, None, None, None, None


def bias_act_(y, bias, relu):
    """y <- act(y + bias[channel]) in place (y: fresh convolution output, NHWC-dense or (..., C) contiguous)."""
    _lib.require_cuda(y, "activation")
    if y.dtype != torch.float32 or _rows_c(y) is None or _rows_c(y)[1] > 256:
        # layouts the token-major kernel does not cover (NCHW-dense outputs): library ops, still on the GPU
        shape = (1, -1, 1, 1) if y.dim() == 4 else (-1,)
        y = y + bias.view(shape)
        return F.relu(y) if relu else y
    return _BiasActFn.apply(y, bias, relu)


class ConvBiasAct(nn.Conv2d):
    """nn.Conv2d (+ ReLU when relu=True) with the fused epilogue; parameters named like nn.Conv2d's."""

    def __init__(self, *args, relu=False, **kwargs):
        super(ConvBiasAct, self).__init__(*args, **kwargs)
        self.relu = relu

    def forward(self, x):
        if (self.relu and self.bias is not None and x.is_cuda and x.dtype == torch.float32 and self.padding_mode == 'zeros'
                and not isinstance(self.padding, str) and self.weight.shape[0] <= 256
                and x.is_contiguous(memory_format=torch.channels_last)):
            return _ConvBiasReluFn.apply(x, self.weight, self.bias, tuple(self.stride), tuple(self.padding), tuple(self.dilation), self.groups)
        y = self._conv_forward(x, self.weight, None)
        if self.bias is None:
            return F.relu(y) if self.relu else y
        return bias_act_(y, self.bias, self.relu)


class ConvTransposeBiasAct(nn.ConvTranspose2d):
    """nn.ConvTranspose2d (+ ReLU) with the fused epilogue."""

    def __init__(self, *args, relu=False, **kwargs):
        super(ConvTransposeBiasAct, self).__init__(*args, **kwargs)
        self.relu = relu

    def forward(self, x, output_size=None):
        num_spatial_dims = 2
        output_padding = self._output_padding(x, output_size, self.stride, self.padding, self.kernel_size,
                                              num_spatial_dims, self.dilation)
        y = F.conv_transpose2d(x, self.weight, None, self.stride, self.padding, output_padding, self.groups, self.dilation)
        if self.bias is None:
            return F.relu(y) if self.relu else y
        return bias_act_(y, self.bias, self.relu)


class _AddLayerNormFn(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x, res, gamma, beta, eps):
        lib = _lib.load()
        x = x.contiguous()
        res = res.contiguous()
        C = x.shape[-1]
        rows = x.numel() // C
        y = torch.empty_like(x)
        stats = torch.empty(rows, 2, device=x.device, dtype=torch.float32)
        rc = lib.isa_add_layernorm_fwd(x.data_ptr(), res.data_ptr(), _lib.ptr(gamma.contiguous()), _lib.ptr(beta.contiguous()),
                                       rows, C, float(eps), y.data_ptr(), stats.data_ptr(), _lib.stream_ptr(x.device))
        _lib.check(rc, "isa_add_layernorm_fwd")
        ctx.save_for_backward(x, res, gamma, stats)
        return y

    @staticmethod
    def backward(ctx, gy):
        lib = _lib.load()
        x, res, gamma, stats = ctx.saved_tensors
        gy = gy.contiguous()
        C = x.shape[-1]
        rows = x.numel() // C
        gv = torch.empty_like(x)
        dgamma = torch.empty(C, device=x.device, dtype=torch.float32)
        dbeta = torch.empty(C, device=x.device, dtype=torch.float32)
        wsb = lib.isa_add_layernorm_workspace_bytes(rows, C)
        ws = torch.empty(wsb, device=x.device, dtype=torch.uint8)
        rc = lib.isa_add_layernorm_bwd(gy.data_ptr(), x.data_ptr(), res.data_ptr(), _lib.ptr(gamma.contiguous()), stats.data_ptr(),
                                       rows, C, gv.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), ws.data_ptr(), wsb,
                                       _lib.stream_ptr(x.device))
        _lib.check(rc, "isa_add_layernorm_bwd")
        return gv, gv, dgamma, dbeta, None


_LN_WIDTHS = (8, 16, 24, 32, 40, 48, 64)


def add_layer_norm(x, res, ln):
    """ln(x + res) for an nn.LayerNorm `ln` over the last dimension (fused kernel for the widths it is built for)."""
    _lib.require_cuda(x, "activation")          # no CPU fallback: other widths / dtypes use the library op ON THE GPU
    C = x.shape[-1]
    if (x.dtype == torch.float32 and C in _LN_WIDTHS and ln.elementwise_affine and ln.bias is not None
            and tuple(ln.normalized_shape) == (C,) and x.shape == res.shape):
        return _AddLayerNormFn.apply(x, res, ln.weight, ln.bias, ln.eps)
    return ln(x + res)


class _ThinLinearFn(torch.autograd.Function):
    """y = x W^T + b for a tall x (rows >> in, out): the weight gradient is a split-K batched GEMM."""
    CHUNK = 512

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        if bias is not None:
            return torch.addmm(bias, x, weight.t())
        return torch.mm(x, weight.t())

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        gy = gy.contiguous()
        gx = torch.mm(gy, weight) if ctx.needs_input_grad[0] else None
        rows = x.shape[0]
        ch = _ThinLinearFn.CHUNK
        if rows % ch == 0 and rows >= 4 * ch:
            s = rows // ch
            gw = torch.bmm(gy.view(s, ch, -1).transpose(1, 2), x.view(s, ch, -1)).sum(0)
        else:
            gw = torch.mm(gy.t(), x)
        gb = gy.sum(0) if ctx.has_bias else None
        return gx, gw, gb


def thin_linear(x, lin):
    """nn.Linear `lin` applied to (..., in) with the split-K weight gradient."""
    shp = x.shape
    x2 = x.reshape(-1, shp[-1])
    if not x2.is_contiguous():
        x2 = x2.contiguous()
    y = _ThinLinearFn.apply(x2, lin.weight, lin.bias)
    return y.view(*shp[:-1], -1)


def _nhwc(t):
    return t if t.is_contiguous(memory_format=torch.channels_last) else t.contiguous(memory_format=torch.channels_last)


class _PixelHeadsFn(torch.autograd.Function):
    """(out0 (n,Co0,H,W), out1 (n,Co1,H,W)) NCHW = 1x1 convolutions of cat(xa, xb) (both NHWC-dense)."""

    @staticmethod
    def forward(ctx, xa, xb, w0, b0, w1, b1):
        lib = _lib.load()
        n, Ca, H, W = xa.shape
        Cb = xb.shape[1]
        HW = H * W
        Co0, Co1 = w0.shape[0], (w1.shape[0] if w1 is not None else 0)
        w = w0.reshape(Co0, Ca + Cb) if w1 is None else torch.cat([w0.reshape(Co0, Ca + Cb), w1.reshape(Co1, Ca + Cb)], 0)
        b = b0 if w1 is None else torch.cat([b0, b1], 0)
        w, b = w.contiguous(), b.contiguous()
        out0 = torch.empty(n, Co0, H, W, device=xa.device, dtype=torch.float32)
        out1 = torch.empty(n, Co1, H, W, device=xa.device, dtype=torch.float32) if Co1 else None
        rc = lib.isa_pixel_heads_fwd(xa.data_ptr(), Ca, xb.data_ptr(), Cb, w.data_ptr(), b.data_ptr(), out0.data_ptr(), Co0,
                                     _lib.ptr(out1), Co1, n * HW, HW, _lib.stream_ptr(xa.device))
        _lib.check(rc, "isa_pixel_heads_fwd")
        ctx.save_for_backward(xa, xb, w)
        ctx.geom = (n, Ca, Cb, H, W, Co0, Co1)
        if Co1:
            return out0, out1
        return out0, out0.new_zeros(())

    @staticmethod
    def backward(ctx, g0, g1):
        lib = _lib.load()
        xa, xb, w = ctx.saved_tensors
        n, Ca, Cb, H, W, Co0, Co1 = ctx.geom
        HW = H * W
        g0 = g0.contiguous() if g0 is not None else None
        g1 = g1.contiguous() if (g1 is not None and Co1) else None
        ga = torch.empty_like(xa) if ctx.needs_input_grad[0] else None      # keeps the NHWC-dense strides
        gb = torch.empty_like(xb) if ctx.needs_input_grad[1] else None
        if ga is not None or gb is not None:
            rc = lib.isa_pixel_heads_bwd(_lib.ptr(g0), Co0, _lib.ptr(g1), Co1, w.data_ptr(), ga.data_ptr() if ga is not None else None, Ca,
                                         gb.data_ptr() if gb is not None else None, Cb, n * HW, HW, _lib.stream_ptr(xa.device))
            _lib.check(rc, "isa_pixel_heads_bwd")
        Co, K = Co0 + Co1, Ca + Cb
        dw_db = torch.empty(Co * K + Co, device=xa.device, dtype=torch.float32)
        wsb = lib.isa_pixel_heads_wgrad_workspace_bytes(Ca, Cb, Co0, Co1)
        ws = torch.empty(wsb, device=xa.device, dtype=torch.uint8)
        rc = lib.isa_pixel_heads_wgrad(_lib.ptr(g0), Co0, _lib.ptr(g1), Co1, xa.data_ptr(), Ca, xb.data_ptr(), Cb, n * HW, HW,
                                       dw_db.data_ptr(), ws.data_ptr(), wsb, _lib.stream_ptr(xa.device))
        _lib.check(rc, "isa_pixel_heads_wgrad")
        dw, db = dw_db[:Co * K].view(Co, K, 1, 1), dw_db[Co * K:]
        gw0, gb0 = dw[:Co0], db[:Co0]
        gw1, gb1 = (dw[Co0:], db[Co0:]) if Co1 else (None, None)
        return ga, gb, gw0, gb0, gw1, gb1


def pixel_heads(xa, xb, head0, head1=None):
    """head0(cat(xa, xb)), head1(cat(xa, xb)) for 1x1 nn.Conv2d heads, as contiguous NCHW tensors (head1 may be None)."""
    _lib.require_cuda(xa, "features")
    Ca, Cb = xa.shape[1], xb.shape[1]
    Co = head0.out_channels + (head1.out_channels if head1 is not None else 0)
    fused = (xa.dtype == torch.float32 and Ca % 2 == 0 and Cb % 2 == 0 and Co <= 32 and head0.kernel_size == (1, 1)
             and xa.shape[2] * xa.shape[3] >= 128
             and head0.bias is not None and (head1 is None or (head1.kernel_size == (1, 1) and head1.bias is not None)))
    if not fused:
        y = torch.cat((xa, xb), dim=1)
        return head0(y).contiguous(), (head1(y).contiguous() if head1 is not None else None)
    out0, out1 = _PixelHeadsFn.apply(_nhwc(xa), _nhwc(xb), head0.weight, head0.bias,
                                     head1.weight if head1 is not None else None, head1.bias if head1 is not None else None)
    return out0, (out1 if head1 is not None else None)


def _skip_grad_view(g, N, C, H, W):
    """(tensor to hand to the kernel, pixel stride in floats) of a gradient that is NHWC-dense or a channel slice of a
    wider NHWC-dense tensor (what torch.cat's backward returns); anything else is made NHWC-dense first."""
    if g.dtype == torch.float32 and g.dim() == 4 and g.stride(1) == 1 and g.stride(3) >= C and g.stride(3) % 4 == 0 \
            and g.stride(2) == W * g.stride(3) and g.stride(0) == H * W * g.stride(3) and g.data_ptr() % 16 == 0:
        return g, g.stride(3)
    g = g.contiguous(memory_format=torch.channels_last)
    return g, C


class _MaxPool2x2Fn(torch.autograd.Function):
    """y = maxpool2x2(x); with `with_skip` the function also returns x itself as a second output (the skip connection), so
    that BOTH gradients of x arrive in one backward call and are summed inside the scatter kernel."""

    @staticmethod
    def forward(ctx, x, with_skip):
        lib = _lib.load()
        N, C, H, W = x.shape
        y = torch.empty(N, C, H // 2, W // 2, device=x.device, dtype=torch.float32, memory_format=torch.channels_last)
        need = ctx.needs_input_grad[0]
        idx = torch.empty(N, H // 2, W // 2, C, device=x.device, dtype=torch.uint8) if need else None
        rc = lib.isa_maxpool2x2_fwd(x.data_ptr(), N, H, W, C, y.data_ptr(), _lib.ptr(idx), _lib.stream_ptr(x.device))
        _lib.check(rc, "isa_maxpool2x2_fwd")
        ctx.geom = (N, C, H, W)
        ctx.with_skip = bool(with_skip)
        if need:
            ctx.save_for_backward(idx)
        if with_skip:
            return y, x.view_as(x)
        return y

    @staticmethod
    def backward(ctx, gy, g_skip=None):
        lib = _lib.load()
        N, C, H, W = ctx.geom
        idx, = ctx.saved_tensors
        gx = torch.empty(N, C, H, W, device=idx.device, dtype=torch.float32, memory_format=torch.channels_last)
        if gy is None:                       # only the skip was used downstream
            gx.copy_(g_skip)
            return gx, None
        gy = gy.contiguous(memory_format=torch.channels_last)
        skip_ptr, skip_px = None, 0
        if g_skip is not None and not ((H | W) & 1):
            g_skip, skip_px = _skip_grad_view(g_skip, N, C, H, W)
            skip_ptr = g_skip.data_ptr()
        rc = lib.isa_maxpool2x2_bwd(gy.data_ptr(), idx.data_ptr(), N, H, W, C, skip_ptr, skip_px, gx.data_ptr(), _lib.stream_ptr(gy.device))
        _lib.check(rc, "isa_maxpool2x2_bwd")
        if g_skip is not None and skip_ptr is None:
            gx.add_(g_skip)
        return gx, None


class MaxPool2x2(nn.Module):
    """nn.MaxPool2d(2, 2) for NHWC-dense fp32 CUDA activations (index-byte forward, scatter backward); other inputs go to
    the library op."""

    def forward(self, x):
        _lib.require_cuda(x, "activation")      # no CPU fallback: other layouts use the library op ON THE GPU
        if (x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] % 4 == 0 and x.shape[2] >= 2 and x.shape[3] >= 2
                and x.is_contiguous(memory_format=torch.channels_last)):
            return _MaxPool2x2Fn.apply(x, False)
        return F.max_pool2d(x, 2, 2)

    def with_skip(self, x):
        """-> (pooled, skip): `skip` is x itself, routed through the pooling function so that the gradient coming back
        through the skip connection is added inside the pooling backward kernel (one pass) instead of being copied and
        accumulated by autograd (0.6 ms per step at batch 16)."""
        _lib.require_cuda(x, "activation")
        if (x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] % 4 == 0 and x.shape[2] >= 2 and x.shape[3] >= 2
                and x.is_contiguous(memory_format=torch.channels_last) and torch.is_grad_enabled() and x.requires_grad):
            return _MaxPool2x2Fn.apply(x, True)
        return self.forward(x), x
