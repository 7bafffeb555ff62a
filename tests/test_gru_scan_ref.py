"""CPU: oracle/gru_scan_ref.py against nn.GRU(bidirectional=True, batch_first=True) in float64, on the row and the
column token maps of renet._geometry.  This fixes what the scan's outputs mean -- in particular that dghn is the
gradient of W_hn h + b_hn, so that [dgx_rz | dghn]^T h_prev is nn.GRU's weight_hh gradient -- independently of any
kernel."""
import pytest
import torch

from isa_b200.renet import _geometry
from oracle.gru_scan_ref import gru_scan_bwd, gru_scan_fwd, token_index

TOL = 1e-10


def _maxdiff(a, b):
    return float((a - b).abs().max())


@pytest.mark.parametrize("mode", ["hor", "ver"])
def test_reference_matches_nn_gru(mode):
    torch.manual_seed(3 if mode == "hor" else 4)
    B, H, W, C, n = 3, 5, 7, 6, 8
    gru = torch.nn.GRU(C, n, batch_first=True, bidirectional=True).double()
    x = torch.randn(B, H, W, C, dtype=torch.float64)
    if mode == "hor":
        seqs = x.reshape(B * H, W, C)
    else:
        seqs = x.permute(0, 2, 1, 3).reshape(B * W, H, C)
    y, _ = gru(seqs)
    dy = torch.randn_like(y)
    y.backward(dy)

    geom = _geometry(B, H, W, mode)
    n_seq, T = geom[0], geom[1]
    idx = token_index(*geom)
    tokens = B * H * W
    xt = torch.empty(tokens, C, dtype=torch.float64)
    xt[idx.reshape(-1)] = seqs.reshape(-1, C)
    out_ref = torch.empty(tokens, 2 * n, dtype=torch.float64)
    out_ref[idx.reshape(-1)] = y.detach().reshape(-1, 2 * n)
    dout = torch.empty_like(out_ref)
    dout[idx.reshape(-1)] = dy.reshape(-1, 2 * n)

    w_ih = torch.stack([gru.weight_ih_l0, gru.weight_ih_l0_reverse]).detach()
    w_hh = torch.stack([gru.weight_hh_l0, gru.weight_hh_l0_reverse]).detach()
    b_ih = torch.stack([gru.bias_ih_l0, gru.bias_ih_l0_reverse]).detach()
    b_hh = torch.stack([gru.bias_hh_l0, gru.bias_hh_l0_reverse]).detach()
    gx = torch.einsum("tc,dgc->tdg", xt, w_ih)

    out, stash = gru_scan_fwd(gx, w_hh, b_hh, b_ih, *geom)
    assert _maxdiff(out, out_ref) < TOL
    out_folded, stash_folded = gru_scan_fwd(gx + b_ih, w_hh, b_hh, None, *geom)
    assert _maxdiff(out_folded, out_ref) < TOL
    assert _maxdiff(stash_folded, stash) < TOL

    # h_{t-1} of every token: the output one step earlier in the direction's own order, 0 at the first step;
    # the stash's z and n quarters give back h_t = (1 - z) n + z h_{t-1}
    o = out.view(tokens, 2, n)
    h_prev = torch.zeros_like(o)
    h_prev[idx[:, 1:].reshape(-1), 0] = o[idx[:, :-1].reshape(-1), 0]
    h_prev[idx[:, :-1].reshape(-1), 1] = o[idx[:, 1:].reshape(-1), 1]
    z = stash[:, :, n:2 * n]
    assert _maxdiff((1 - z) * stash[:, :, 2 * n:3 * n] + z * h_prev, o) < TOL

    for b, bias in (("b_ih", b_ih), ("folded", None)):
        g_in = gx if bias is not None else gx + b_ih
        dgx, dghn = gru_scan_bwd(dout, g_in, w_hh, b_hh, bias, *geom)
        assert dgx.shape == (tokens, 2, 3 * n) and dghn.shape == (tokens, 2, n)
        dw_ih = torch.einsum("tdg,tc->dgc", dgx, xt)
        dw_hh = torch.cat([torch.einsum("tdg,tdu->dgu", dgx[:, :, :2 * n], h_prev),
                           torch.einsum("tdg,tdu->dgu", dghn, h_prev)], dim=1)
        db_hh = torch.cat([dgx[:, :, :2 * n].sum(0), dghn.sum(0)], dim=1)
        for d, sfx in enumerate(("", "_reverse")):
            assert _maxdiff(dw_ih[d], getattr(gru, "weight_ih_l0" + sfx).grad) < TOL, (b, d)
            assert _maxdiff(dw_hh[d], getattr(gru, "weight_hh_l0" + sfx).grad) < TOL, (b, d)
            assert _maxdiff(dgx[:, d].sum(0), getattr(gru, "bias_ih_l0" + sfx).grad) < TOL, (b, d)
            assert _maxdiff(db_hh[d], getattr(gru, "bias_hh_l0" + sfx).grad) < TOL, (b, d)
