"""GPU: ReNet (persistent GRU scan kernels through the C-ABI) against the nn.GRU oracle
(oracle/renet_ref.py) on identical weights: forward, input gradient and every parameter gradient.
Tolerance: 1e-3 relative (north_star) -- asserted at 2e-4."""
import numpy as np
import pytest
import torch

from oracle.renet_ref import ReNetRef

pytestmark = pytest.mark.gpu

RTOL = 2e-4


def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


@pytest.mark.parametrize("B,C,H,W,n,patch", [(2, 16, 8, 12, 8, (1, 1)), (1, 3, 16, 16, 16, (2, 2)), (3, 32, 20, 9, 100, (1, 1)),
                                             (2, 7, 5, 33, 12, (1, 1)), (16, 64, 16, 16, 32, (1, 1)), (1, 5, 7, 9, 4, (2, 3))])
def test_renet_forward_backward(cuda, B, C, H, W, n, patch):
    from isa_b200.renet import ReNet
    torch.manual_seed(B * 100 + n)
    ref = ReNetRef(C, n, patch).double()
    mod = ReNet(C, n, patch).to(cuda)
    mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    x = torch.randn(B, C, H, W, dtype=torch.float64)
    xr = x.clone().requires_grad_(True)
    yr = ref(xr)
    gy = torch.randn_like(yr)
    yr.backward(gy)
    xg = x.float().to(cuda).requires_grad_(True)
    yg = mod(xg)
    assert yg.shape == yr.shape
    assert _rel(yg, yr) < RTOL
    yg.backward(gy.float().to(cuda))
    assert _rel(xg.grad, xr.grad) < RTOL
    for (name, p), (_, q) in zip(mod.named_parameters(), ref.named_parameters()):
        assert _rel(p.grad, q.grad) < RTOL, name


def test_renet_inference_no_stash(cuda):
    from isa_b200.renet import ReNet
    torch.manual_seed(0)
    ref = ReNetRef(24, 20)
    mod = ReNet(24, 20).to(cuda)
    mod.load_state_dict(ref.state_dict())
    x = torch.randn(2, 24, 10, 14)
    with torch.no_grad():
        assert _rel(mod(x.to(cuda)), ref(x)) < RTOL


def test_state_dict_names_match_nn_gru():
    from isa_b200.renet import ReNet
    names = set(ReNet(8, 4).state_dict().keys())
    assert {"rnn_hor.weight_ih_l0", "rnn_hor.weight_hh_l0_reverse", "rnn_ver.bias_hh_l0", "rnn_ver.weight_ih_l0_reverse"} <= names


@pytest.mark.parametrize("B", [16, 12, 8])
def test_renet_headline_shape_forward_backward(cuda, B):
    """The training step's shape (BASELINE.json configs[1]): (B,256,64,64) map, 100 units -- forward, input gradient and
    every parameter gradient against nn.GRU run in float64 ON THE GPU (the CPU oracle needs minutes at this size).
    On 148 SMs the tensor-core scans run 14 sequences per CTA at B = 16, 12 at B = 12, and 8 at B = 8, the per-rank
    batch of the two-GPU data-parallel run."""
    from isa_b200.renet import ReNet
    torch.manual_seed(7)
    C, H, W, n = 256, 64, 64, 100
    ref = ReNetRef(C, n, (1, 1)).double().to(cuda)
    mod = ReNet(C, n, (1, 1)).to(cuda)
    mod.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    x = torch.randn(B, C, H, W, dtype=torch.float64, device=cuda)
    xr = x.clone().requires_grad_(True)
    yr = ref(xr)
    gy = torch.randn_like(yr)
    yr.backward(gy)
    xg = x.float().requires_grad_(True)
    yg = mod(xg)
    assert _rel(yg, yr) < RTOL
    yg.backward(gy.float())
    assert _rel(xg.grad, xr.grad) < RTOL
    for (name, p), (_, q) in zip(mod.named_parameters(), ref.named_parameters()):
        assert _rel(p.grad, q.grad) < RTOL, name


@pytest.mark.parametrize("tokens,cin,n", [(128, 32, 8), (1000, 36, 12), (4096, 256, 100), (777, 200, 100), (65536, 200, 100)])
def test_projection_gemms_against_float64(cuda, tokens, cin, n):
    """csrc/proj_gemm.cu through the C-ABI: x W^T, dG W and [dgx | dghn]^T [x | h_prev | 1] against float64 matmuls;
    ragged token counts, widths that are not multiples of 8 / 16 / 32, both sweep geometries."""
    from isa_b200 import _lib
    lib = _lib.load()
    g = torch.Generator(device="cpu").manual_seed(tokens + cin)
    x = torch.randn(tokens, cin, generator=g).to(cuda)
    w = torch.randn(6 * n, cin, generator=g).to(cuda)
    st = _lib.stream_ptr(cuda)
    gx = torch.empty(tokens, 6 * n, device=cuda)
    wpb = lib.isa_renet_proj_workspace_bytes(cin, 6 * n)
    wpk = torch.empty(wpb, device=cuda, dtype=torch.uint8)
    _lib.check(lib.isa_renet_proj_fwd(_lib.ptr(x), _lib.ptr(w), tokens, cin, 6 * n, _lib.ptr(gx), _lib.ptr(wpk), wpb, st), "fwd")
    ref = x.double() @ w.double().t()
    assert _rel(gx, ref) < 2e-5
    dg = torch.randn(tokens, 2, 3 * n, generator=g).to(cuda)
    dx = torch.empty(tokens, cin, device=cuda)
    _lib.check(lib.isa_renet_proj_dx(_lib.ptr(dg), _lib.ptr(w), tokens, 6 * n, cin, _lib.ptr(dx), _lib.ptr(wpk), wpb, st), "dx")
    assert _rel(dx, dg.view(tokens, -1).double() @ w.double()) < 2e-5
    dghn = torch.randn(tokens, 2, n, generator=g).to(cuda)
    out = torch.randn(tokens, 2, n, generator=g).to(cuda)
    for step, pos_div, pos_mod in ((1, 1, 16 if tokens % 16 == 0 else 37 if tokens % 37 == 0 else 1),
                                   (8 if tokens % 64 == 0 else 1, 8 if tokens % 64 == 0 else 1, 8 if tokens % 64 == 0 else 1)):
        if tokens % (pos_div * pos_mod) != 0:
            continue
        dw_ih, dw_hh = torch.empty(2, 3 * n, cin, device=cuda), torch.empty(2, 3 * n, n, device=cuda)
        db_ih, db_hh = torch.empty(2, 3 * n, device=cuda), torch.empty(2, 3 * n, device=cuda)
        wsb = lib.isa_renet_proj_wgrad_workspace_bytes(tokens, cin, n)
        ws = torch.empty(wsb, device=cuda, dtype=torch.uint8)
        _lib.check(lib.isa_renet_proj_wgrad(_lib.ptr(dg), _lib.ptr(dghn), _lib.ptr(x), _lib.ptr(out), tokens, cin, n, step, pos_div, pos_mod,
                                            _lib.ptr(dw_ih), _lib.ptr(dw_hh), _lib.ptr(db_ih), _lib.ptr(db_hh), _lib.ptr(ws), wsb, st), "wgrad")
        t = torch.arange(tokens, device=cuda)
        pos = (t // pos_div) % pos_mod
        o = out.double()
        hp = torch.zeros_like(o)
        ok0, ok1 = pos >= 1, pos <= pos_mod - 2
        hp[ok0, 0] = o[t[ok0] - step, 0]
        hp[ok1, 1] = o[t[ok1] + step, 1]
        dgd, dnd = dg.double(), dghn.double()
        assert _rel(dw_ih, torch.einsum("tdg,tc->dgc", dgd, x.double())) < 2e-5
        assert _rel(db_ih, dgd.sum(0)) < 2e-5
        ref_hh = torch.cat([torch.einsum("tdg,tdu->dgu", dgd[:, :, :2 * n], hp), torch.einsum("tdg,tdu->dgu", dnd, hp)], dim=1)
        assert _rel(dw_hh, ref_hh) < 2e-5
        assert _rel(db_hh, torch.cat([dgd[:, :, :2 * n].sum(0), dnd.sum(0)], dim=1)) < 2e-5
