"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the two GRU scan entry points of include/isa_b200.h,
isa_gru_scan_fwd and isa_gru_scan_bwd, on the ABI's own arrays:
    gx    [tokens][2][3n]   input projection of both directions (with or without b_ih)
    w_hh  [2][3n][n], b_hh [2][3n], b_ih [2][3n] or None
    out   [tokens][2n]      h_t of direction 0 in [0, n), of direction 1 in [n, 2n)
    stash [tokens][2][4n]   r, z, n, W_hn h + b_hn
    dgx   [tokens][2][3n]   dL/dgx
    dghn  [tokens][2][n]    dL/d(W_hn h + b_hn)
Sequence q at step t is token (q // inner) * outer + (q % inner) * inner_s + t * t_s; direction 0 runs t = 0 .. T-1,
direction 1 runs t = T-1 .. 0, and h_0 = 0 for both.  The gate arithmetic is nn.GRU's (gate order r, z, n):
    r = sigmoid(gx_r + b_ir + W_hr h + b_hr)   z = sigmoid(gx_z + b_iz + W_hz h + b_hz)
    n = tanh(gx_n + b_in + r * (W_hn h + b_hn))   h' = (1 - z) n + z h
tests/test_gru_scan_ref.py pins this file to nn.GRU; the backward is autograd through the forward.
Tokens that no sequence visits are 0 in every returned array.
"""
import torch


def token_index(n_seq, T, inner, outer, inner_s, t_s, device=None):
    """[n_seq][T] token of sequence q at step t."""
    q = torch.arange(n_seq, dtype=torch.int64, device=device)
    base = (q // inner) * outer + (q % inner) * inner_s
    return base[:, None] + torch.arange(T, dtype=torch.int64, device=device)[None, :] * t_s


def _scan(gx, w_hh, b_hh, b_ih, idx):
    """-> out [tokens][2][n], stash [tokens][2][4n], hn[d][t] = W_hn h + b_hn [n_seq][n] (the graph's own nodes)."""
    n_seq, T = idx.shape
    n = w_hh.shape[2]
    assert idx.numel() == idx.unique().numel(), "the token map visits a token twice"
    g = gx[idx]                                                 # [n_seq][T][2][3n]
    hs, sts, hn_nodes = [], [], []
    for d in range(2):
        h = gx.new_zeros(n_seq, n)
        h_t, st_t, hn_t = [None] * T, [None] * T, [None] * T
        for step in range(T):
            t = step if d == 0 else T - 1 - step
            gh = h @ w_hh[d].t() + b_hh[d]
            xi = g[:, t, d] if b_ih is None else g[:, t, d] + b_ih[d]
            r = torch.sigmoid(xi[:, :n] + gh[:, :n])
            z = torch.sigmoid(xi[:, n:2 * n] + gh[:, n:2 * n])
            hn = gh[:, 2 * n:]
            nn_ = torch.tanh(xi[:, 2 * n:] + r * hn)
            h = (1 - z) * nn_ + z * h
            h_t[t], hn_t[t] = h, hn
            st_t[t] = torch.cat([r, z, nn_, hn], dim=1)
        hs.append(torch.stack(h_t, 1))
        sts.append(torch.stack(st_t, 1))
        hn_nodes.append(hn_t)
    tokens = gx.shape[0]
    flat = idx.reshape(-1)
    out = gx.new_zeros(tokens, 2, n).index_put((flat,), torch.stack(hs, 2).reshape(-1, 2, n))
    stash = gx.new_zeros(tokens, 2, 4 * n).index_put((flat,), torch.stack(sts, 2).reshape(-1, 2, 4 * n))
    return out, stash, hn_nodes


def _abi(gx, w_hh, b_hh, b_ih):
    """float64 copies in the ABI's shapes."""
    w_hh = w_hh.detach().double()
    n = w_hh.shape[-1]
    f = lambda t: None if t is None else t.detach().double().reshape(2, 3 * n)
    return gx.detach().double().reshape(gx.shape[0], 2, 3 * n), w_hh.reshape(2, 3 * n, n), f(b_hh), f(b_ih)


def gru_scan_fwd(gx, w_hh, b_hh, b_ih, n_seq, T, inner, outer, inner_s, t_s):
    """isa_gru_scan_fwd in float64 -> (out [tokens][2n], stash [tokens][2][4n])."""
    gx, w_hh, b_hh, b_ih = _abi(gx, w_hh, b_hh, b_ih)
    idx = token_index(n_seq, T, inner, outer, inner_s, t_s, gx.device)
    with torch.no_grad():
        out, stash, _ = _scan(gx, w_hh, b_hh, b_ih, idx)
    return out.reshape(gx.shape[0], -1), stash


def gru_scan_bwd(dout, gx, w_hh, b_hh, b_ih, n_seq, T, inner, outer, inner_s, t_s):
    """isa_gru_scan_bwd in float64 for L = sum(out * dout), out the forward of these inputs
    -> (dgx = dL/dgx [tokens][2][3n], dghn = dL/d(W_hn h + b_hn) [tokens][2][n])."""
    gx, w_hh, b_hh, b_ih = _abi(gx, w_hh, b_hh, b_ih)
    gx.requires_grad_(True)
    b_hh.requires_grad_(True)       # so that the first step's W_hn h + b_hn = b_hn is a node of the graph as well
    idx = token_index(n_seq, T, inner, outer, inner_s, t_s, gx.device)
    with torch.enable_grad():
        out, _, hn = _scan(gx, w_hh, b_hh, b_ih, idx)
        for node in (x for per_dir in hn for x in per_dir):
            node.retain_grad()
        (out * dout.detach().double().reshape(out.shape)).sum().backward()
    g = torch.stack([torch.stack([x.grad for x in per_dir], 1) for per_dir in hn], 2)   # [n_seq][T][2][n]
    dghn = gx.new_zeros(gx.shape[0], 2, w_hh.shape[2]).index_put((idx.reshape(-1),), g.reshape(-1, 2, w_hh.shape[2]))
    return gx.grad.detach(), dghn
