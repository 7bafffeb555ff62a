"""GPU: channels-last bias/activation epilogue, residual + LayerNorm and the split-K thin linear (csrc/pointwise.cu)
against plain PyTorch fp32 on the same inputs (forward, input gradient, parameter gradients)."""
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("N,C,H,W", [(2, 64, 32, 48), (1, 100, 17, 9), (3, 50, 8, 8), (2, 2, 33, 31), (1, 256, 16, 16), (16, 24, 64, 64)])
@pytest.mark.parametrize("relu", [True, False])
def test_bias_act_matches_torch(cuda, N, C, H, W, relu):
    from isa_b200.pointwise import bias_act_
    torch.manual_seed(N * C + H)
    x = torch.randn(N, C, H, W, device=cuda).contiguous(memory_format=torch.channels_last)
    b = torch.randn(C, device=cuda, requires_grad=True)
    x1 = x.clone().requires_grad_(True)
    x2 = x.clone().requires_grad_(True)
    y_ref = x1 + b.view(1, -1, 1, 1)
    y_ref = F.relu(y_ref) if relu else y_ref
    g = torch.randn_like(y_ref)
    gx_ref, gb_ref = torch.autograd.grad(y_ref, (x1, b), g)
    y = bias_act_(x2 * 1.0, b, relu)          # * 1.0: a fresh non-leaf tensor, like a convolution output
    gx, gb = torch.autograd.grad(y, (x2, b), g)
    assert torch.equal(y, y_ref)
    assert torch.equal(gx, gx_ref)
    torch.testing.assert_close(gb, gb_ref, rtol=2e-5, atol=2e-4)


def test_conv_modules_match_stock_layers(cuda):
    from isa_b200.pointwise import ConvBiasAct, ConvTransposeBiasAct
    torch.manual_seed(3)
    for ours, ref, shape in ((ConvBiasAct(8, 20, 3, padding=1, relu=True), nn.Conv2d(8, 20, 3, padding=1), (2, 8, 24, 20)),
                             (ConvBiasAct(12, 2, 1), nn.Conv2d(12, 2, 1), (2, 12, 16, 16)),
                             (ConvTransposeBiasAct(8, 12, kernel_size=(2, 2), stride=(2, 2), relu=True),
                              nn.ConvTranspose2d(8, 12, kernel_size=(2, 2), stride=(2, 2)), (2, 8, 10, 12))):
        ours, ref = ours.to(cuda), ref.to(cuda)
        ref.load_state_dict(ours.state_dict())          # same parameter names
        x = torch.randn(*shape, device=cuda).contiguous(memory_format=torch.channels_last)
        xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        ya = ours(xa)
        yb = ref(xb)
        if ours.relu:
            yb = F.relu(yb)
        torch.testing.assert_close(ya, yb, rtol=1e-4, atol=1e-4)
        g = torch.randn_like(yb)
        ya.backward(g)
        yb.backward(g)
        torch.testing.assert_close(xa.grad, xb.grad, rtol=1e-4, atol=1e-4)
        torch.testing.assert_close(ours.weight.grad, ref.weight.grad, rtol=1e-3, atol=1e-3)
        torch.testing.assert_close(ours.bias.grad, ref.bias.grad, rtol=1e-4, atol=1e-3)


def test_conv_epilogue_in_cudnn_equals_epilogue_kernel(cuda):
    """relu(conv + bias) with the epilogue inside cuDNN's convolution (ConvBiasAct) against the bias-free convolution
    followed by the in-place epilogue kernel: same output bit for bit, same gradients."""
    from isa_b200.pointwise import ConvBiasAct, bias_act_
    torch.manual_seed(5)
    m = ConvBiasAct(16, 32, 3, padding=1, relu=True).to(cuda)
    x = torch.randn(3, 16, 40, 28, device=cuda).contiguous(memory_format=torch.channels_last)
    g = torch.randn(3, 32, 40, 28, device=cuda).contiguous(memory_format=torch.channels_last)
    outs = []
    for fused in (True, False):
        xa = x.clone().requires_grad_(True)
        y = m(xa) if fused else bias_act_(F.conv2d(xa, m.weight, None, padding=1), m.bias, True)
        grads = torch.autograd.grad(y, (xa, m.weight, m.bias), g)
        outs.append((y.detach(),) + grads)
    assert torch.equal(outs[0][0], outs[1][0])
    for a, b in zip(outs[0][1:], outs[1][1:]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("rows,C", [(1000, 24), (65536, 24), (257, 8), (300, 64), (77, 40)])
def test_add_layernorm_matches_torch(cuda, rows, C):
    from isa_b200.pointwise import add_layer_norm
    torch.manual_seed(rows + C)
    ln = nn.LayerNorm(C).to(cuda)
    with torch.no_grad():
        ln.weight.normal_(1.0, 0.3)
        ln.bias.normal_(0.0, 0.3)
    x = (torch.randn(rows, C, device=cuda) * 2 + 0.5)
    r = torch.randn(rows, C, device=cuda)
    xa, ra = x.clone().requires_grad_(True), r.clone().requires_grad_(True)
    xb, rb = x.clone().requires_grad_(True), r.clone().requires_grad_(True)
    g = torch.randn(rows, C, device=cuda)
    ya = add_layer_norm(xa, ra, ln)
    gxa, gra, gwa, gba = torch.autograd.grad(ya, (xa, ra, ln.weight, ln.bias), g)
    yb = ln(xb + rb)
    gxb, grb, gwb, gbb = torch.autograd.grad(yb, (xb, rb, ln.weight, ln.bias), g)
    torch.testing.assert_close(ya, yb, rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(gxa, gxb, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(gra, grb, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(gwa, gwb, rtol=1e-4, atol=1e-3 * (rows ** 0.5) / 30)
    torch.testing.assert_close(gba, gbb, rtol=1e-4, atol=1e-3 * (rows ** 0.5) / 30)


@pytest.mark.parametrize("rows,cin,cout", [(65536, 24, 24), (4096, 200, 24), (1000, 24, 24)])
def test_thin_linear_matches_linear(cuda, rows, cin, cout):
    from isa_b200.pointwise import thin_linear
    torch.manual_seed(rows)
    lin = nn.Linear(cin, cout).to(cuda)
    x = torch.randn(2, rows // 2, cin, device=cuda)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    g = torch.randn(2, rows // 2, cout, device=cuda)
    ya = thin_linear(xa, lin)
    ga = torch.autograd.grad(ya, (xa, lin.weight, lin.bias), g)
    yb = F.linear(xb, lin.weight, lin.bias)
    gb = torch.autograd.grad(yb, (xb, lin.weight, lin.bias), g)
    torch.testing.assert_close(ya, yb, rtol=1e-5, atol=1e-5)
    for a, b in zip(ga, gb):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=2e-3)


# (2, 80, 64, ...): more than 128 source channels, so forward, input gradient and weight gradient run the FFMA kernels
@pytest.mark.parametrize("n,Ca,Cb,H,W,Co0,Co1", [(2, 50, 64, 32, 40, 2, 24), (1, 6, 2, 9, 7, 3, 5), (3, 50, 64, 16, 16, 2, 0), (1, 20, 12, 8, 8, 2, 30),
                                                 (2, 80, 64, 16, 16, 2, 24)])
def test_pixel_heads_match_conv_of_concatenation(cuda, n, Ca, Cb, H, W, Co0, Co1):
    from isa_b200.pointwise import pixel_heads
    torch.manual_seed(Ca + Cb + Co1)
    torch.backends.cudnn.allow_tf32 = False
    try:
        h0 = nn.Conv2d(Ca + Cb, Co0, 1).to(cuda)
        h1 = nn.Conv2d(Ca + Cb, Co1, 1).to(cuda) if Co1 else None
        xa = torch.randn(n, Ca, H, W, device=cuda).contiguous(memory_format=torch.channels_last)
        xb = torch.randn(n, Cb, H, W, device=cuda).contiguous(memory_format=torch.channels_last)
        a1, b1 = xa.clone().requires_grad_(True), xb.clone().requires_grad_(True)
        a2, b2 = xa.clone().requires_grad_(True), xb.clone().requires_grad_(True)
        o0, o1 = pixel_heads(a1, b1, h0, h1)
        y = torch.cat((a2, b2), 1)
        r0, r1 = h0(y), (h1(y) if h1 is not None else None)
        assert o0.is_contiguous()
        torch.testing.assert_close(o0, r0, rtol=1e-4, atol=1e-4)     # bf16 hi/lo tensor-core products: ~2^-16 relative
        params = [h0.weight, h0.bias] + ([h1.weight, h1.bias] if h1 is not None else [])
        g0 = torch.randn_like(r0)
        if h1 is not None:
            torch.testing.assert_close(o1, r1, rtol=1e-4, atol=1e-4)
            g1 = torch.randn_like(r1)
            got = torch.autograd.grad([o0, o1], [a1, b1] + params, [g0, g1])
            ref = torch.autograd.grad([r0, r1], [a2, b2] + params, [g0, g1])
        else:
            got = torch.autograd.grad([o0], [a1, b1] + params, [g0])
            ref = torch.autograd.grad([r0], [a2, b2] + params, [g0])
        for a, b in zip(got, ref):
            torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-3)
    finally:
        torch.backends.cudnn.allow_tf32 = True


@pytest.mark.parametrize("N,C,H,W", [(2, 64, 32, 48), (1, 128, 17, 9), (3, 8, 7, 7), (16, 64, 64, 64)])
def test_maxpool2x2_matches_torch(cuda, N, C, H, W):
    from isa_b200.pointwise import MaxPool2x2
    torch.manual_seed(N + C + H)
    x = torch.randn(N, C, H, W, device=cuda)
    x = torch.relu(x)                                   # post-ReLU inputs: many exact ties at zero
    x[0, 0, 0, 0] = float("nan")
    x = x.contiguous(memory_format=torch.channels_last)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    ya = MaxPool2x2()(xa)
    yb = F.max_pool2d(xb, 2, 2)
    assert torch.equal(torch.nan_to_num(ya, nan=-7.0), torch.nan_to_num(yb, nan=-7.0))
    g = torch.randn_like(yb)
    ga, = torch.autograd.grad(ya, xa, g)
    gb, = torch.autograd.grad(yb, xb, g)
    assert torch.equal(ga, gb)
    with torch.no_grad():
        assert torch.equal(torch.nan_to_num(MaxPool2x2()(x), nan=-7.0), torch.nan_to_num(yb, nan=-7.0))


@pytest.mark.parametrize("N,C,H,W,wide", [(2, 64, 32, 48, 0), (2, 128, 16, 24, 100), (1, 8, 6, 10, 4), (1, 16, 7, 9, 0)])
def test_maxpool2x2_with_skip_sums_both_gradients(cuda, N, C, H, W, wide):
    """pool.with_skip: the pooled path and the skip path (directly, or through a channel slice of a wider concatenation like
    torch.cat((y, skip), 1) in the decoder) both send a gradient to the same activation; the fused backward must equal
    autograd's scatter + add."""
    from isa_b200.pointwise import MaxPool2x2
    torch.manual_seed(N * C + W)
    x = torch.randn(N, C, H, W, device=cuda).contiguous(memory_format=torch.channels_last)
    xa, xb = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    other = torch.randn(N, max(wide, 4), H, W, device=cuda).contiguous(memory_format=torch.channels_last)

    def loss(pooled, skip, wa, wb):
        z = torch.cat((other, skip), dim=1) if wide else skip
        return (pooled * wa).sum() + (z * wb).sum()

    ya, sa = MaxPool2x2().with_skip(xa)
    yb, sb = F.max_pool2d(xb, 2, 2), xb
    wa = torch.randn_like(yb)
    wb = torch.randn(N, C + (max(wide, 4) if wide else 0), H, W, device=cuda).contiguous(memory_format=torch.channels_last)
    loss(ya, sa, wa, wb).backward()
    loss(yb, sb, wa, wb).backward()
    assert torch.equal(ya, yb)
    torch.testing.assert_close(xa.grad, xb.grad, rtol=0, atol=0)
    # only one of the two outputs used
    xc = x.clone().requires_grad_(True)
    yc, sc = MaxPool2x2().with_skip(xc)
    (sc * 2.0).sum().backward()
    assert torch.equal(xc.grad, torch.full_like(xc, 2.0))


def test_fused_adadelta_matches_torch(cuda):
    """clip_grad_norm_ + torch.optim.Adadelta vs the flat fused optimizer on the same parameters / gradients."""
    from isa_b200.optim import FusedAdadelta
    torch.manual_seed(5)
    shapes = [(7, 3, 3, 3), (7,), (33, 17), (5,), (1,), (64, 64, 3, 3)]
    pa = [nn.Parameter(torch.randn(*s, device=cuda)) for s in shapes]
    pb = [nn.Parameter(p.detach().clone()) for p in pa]
    oa = FusedAdadelta(pa, lr=1.0, weight_decay=1e-3)
    ob = torch.optim.Adadelta(pb, lr=1.0, weight_decay=1e-3)
    for step in range(6):
        clip = 10.0 if step % 2 == 0 else 0.5
        oa.zero_grad()
        ob.zero_grad()
        for a, b in zip(pa, pb):
            g = torch.randn_like(a) * (3.0 if step < 3 else 0.01)
            a.grad.add_(g)                      # autograd accumulates in place into the flat views
            b.grad = g.clone()
        ref_norm = torch.nn.utils.clip_grad_norm_(pb, clip)
        ob.step()
        oa.step(clip_grad_norm=clip)
        torch.testing.assert_close(oa.grad_norm[0], ref_norm, rtol=1e-5, atol=1e-6)
        for a, b in zip(pa, pb):
            torch.testing.assert_close(a.data, b.data, rtol=2e-5, atol=2e-6)
    sd = oa.state_dict()
    oa.load_state_dict(sd)
    assert oa.param_groups[0]['lr'] == 1.0
