"""TEST INFRASTRUCTURE ONLY -- the discriminative loss of isa_disc_loss_fwd / isa_disc_loss_bwd restated in float64 torch.

The same operation as oracle/disc_loss.py (pinned to it by tests/test_disc_loss_ref.py), written so that it runs on any
device and at full size, with the gradient taken by autograd instead of the analytic formulas.  Every image is reduced
over its list of (pixel, instance, weight) pairs with a non-zero weight, by gathers and index_add: O(pairs * C) memory,
one pair per foreground pixel of a hard label map (bs,H,W) uint8 (255 = background), one per non-zero entry of dense
masks (bs,K,H,W), soft or overlapping.  Working on the pairs alone also keeps a NaN mean out of the gradient of pixels
that do not belong to that image's instances, as in the kernels.
Semantics (the kernels' and the reference's): instances k < n_b = clamp(n_objects[b], 0, K) carry the means, variance,
distance and regulariser terms; every channel k < K counts as foreground for the q-regulariser.  An instance k < n_b
without pixels makes its mean 0/0 and the image's variance, distance and regulariser NaN; its gradient is NaN at the
pixels of the image's instances and finite elsewhere, as the kernels compute it.
"""
import math

import torch

SHIPPED_TERMS = (1.0, 0.0, 0.0, 0.005)


def _norm(v, norm):
    return v.norm(dim=-1) if norm == 2 else v.abs().sum(-1)


def discriminative_loss(emb, target, n_objects, K, delta_v, delta_d, norm=2, terms=SHIPPED_TERMS, normalize_means=True,
                        q_den=None, grad_loss=1.0, grad_means=None, want_grad=False):
    """emb (bs,C,H,W) tensor; target (bs,H,W) uint8 label map or (bs,K,H,W) masks; n_objects (bs,) ints.
    Returns dict(loss, terms (var, dist, reg, qreg), means (bs,K,C), grad (bs,C,H,W) if want_grad), float64 tensors on
    emb's device.  grad is the gradient of grad_loss * loss + sum(means[b, :n_b] * grad_means[b, :n_b])."""
    dev = emb.device
    bs, C, H, W = emb.shape
    P = H * W
    w_var, w_dist, w_reg, w_q = [float(t) for t in terms]
    x = emb.detach().to(torch.float64).reshape(bs, C, P).clone().requires_grad_(want_grad)
    target = torch.as_tensor(target, device=dev)
    dense = target.dim() == 4
    nobj = [min(max(int(n), 0), K) for n in torch.as_tensor(n_objects).reshape(-1).tolist()]
    f64 = dict(dtype=torch.float64, device=dev)
    nan = torch.tensor(float("nan"), **f64)
    zero = torch.zeros((), **f64)

    var_b, dist_b, reg_b, means, extra = [], [], [], [], zero
    q_sum, n_fg = zero, 0.0
    for b in range(bs):
        n = nobj[b]
        xb = x[b].t()                                                     # (P, C)
        # the (pixel, instance k < n, weight) pairs with a non-zero weight: one per foreground pixel of a label map
        if dense:
            M = target[b].reshape(K, P).to(torch.float64)
            p_idx, idx = M[:n].t().nonzero(as_tuple=True)
            w = M[idx, p_idx]
            fg = M.sum(0)
        else:
            lab = target[b].reshape(P).long()
            p_idx = (lab < n).nonzero(as_tuple=True)[0]
            idx = lab[p_idx]
            w = torch.ones(len(idx), **f64)
            fg = (lab < K).to(torch.float64)
        xs = xb[p_idx]
        sums = torch.zeros(n, C, **f64).index_add(0, idx, w[:, None] * xs)
        cnt = torch.zeros(n, **f64).index_add(0, idx, w)
        # an absent instance: NaN mean and NaN image terms, without sending NaN through the other instances' gradient
        present = cnt > 0
        poison = nan if bool((~present).any()) else zero
        mu = sums / torch.where(present, cnt, torch.ones_like(cnt))[:, None]
        r = mu.norm(dim=1)
        if normalize_means:
            mu = mu / torch.where(r > 0, r, torch.ones_like(r))[:, None]
        mu_out = torch.where(present[:, None], mu, nan)
        means.append(torch.cat([mu_out, torch.zeros(K - n, C, **f64)]))
        if grad_means is not None and n > 0:
            extra = extra + (mu * torch.as_tensor(grad_means, **f64)[b, :n]).sum()

        h = torch.clamp(_norm(xs - mu[idx], norm) - delta_v, min=0.0)
        hsum = (w * h * h).sum()
        var_b.append(hsum / (cnt.sum() + poison))
        if n > 1:
            e = _norm(mu[:, None, :] - mu[None, :, :], norm)
            off = ~torch.eye(n, dtype=torch.bool, device=dev)
            m = torch.clamp(2 * delta_d - e[off], min=0.0)
            dist_b.append((m * m).sum() / (n * (n - 1)) + poison)
        else:
            dist_b.append(zero)
        reg_b.append(_norm(mu, norm).mean() + poison if n > 0 else nan)

        # q-regulariser (|x_p * fg_p|_2 - 1)^2 over every pixel: a background pixel adds exactly 1
        on = fg != 0
        lq = (xb[on] * fg[on][:, None]).norm(dim=1)
        q_sum = q_sum + ((lq - 1) ** 2).sum() + float((~on).sum())
        n_fg += float(fg.sum())

    den = float(math.floor(n_fg)) if q_den is None else float(q_den)
    qreg = q_sum / den if den != 0 else torch.tensor(float("inf"), **f64)
    var_t = torch.stack(var_b).sum() / bs
    dist_t = torch.stack(dist_b).sum() / bs if w_dist != 0 else zero
    reg_t = torch.stack(reg_b).sum() / bs if w_reg != 0 else zero
    loss = zero
    for w, t in ((w_var, var_t), (w_dist, dist_t), (w_reg, reg_t), (w_q, qreg)):
        if w != 0:
            loss = loss + w * t
    out = dict(loss=loss.detach(), terms=torch.stack([var_t, dist_t, reg_t, qreg]).detach(),
               means=torch.stack(means).detach())
    if want_grad:
        total = float(grad_loss) * loss + extra
        (g,) = torch.autograd.grad(total, x, allow_unused=True)
        out["grad"] = (torch.zeros_like(x) if g is None else g).reshape(bs, C, H, W)
    return out
