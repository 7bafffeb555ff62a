"""TEST INFRASTRUCTURE ONLY -- the CPU oracle of the discriminative loss.

A numpy restatement (float64 by default) of the reference's loss, function by function:
  means            /root/reference/code/lib/losses/discriminative.py:7-62   (M='intri': L2-normalised)
  variance term    /root/reference/code/lib/losses/discriminative.py:65-95  (M='_intri' => else-branch :84-93,
                                                                             pooled over all fg pixels of the image)
  distance term    /root/reference/code/lib/losses/discriminative.py:98-132
  regulariser      /root/reference/code/lib/losses/discriminative.py:135-147
  q-regulariser    /root/reference/code/lib/losses/discriminative.py:149-160 (every pixel, denominator int(sum target))
  composite        /root/reference/code/lib/losses/discriminative.py:162-188 (1.0*var + 0.005*qreg)
plus the analytic gradient of SURVEY.md Appendix A (validated against autograd of the
reference in tests/test_oracle_disc_loss.py).

Pinned against the reference itself: tests/golden/disc_loss_*.npz hold loss / means /
input-gradient produced by importing the reference file (tests/golden/make_golden.py).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may import this.
"""
import numpy as np

SHIPPED_TERMS = (1.0, 0.0, 0.0, 0.005)


def _dense_masks(target, K, dtype):
    """-> (bs, P, K) weights from a (bs,H,W) uint8 label map (255=bg) or (bs,K,H,W) masks."""
    target = np.asarray(target)
    if target.ndim == 3:
        bs = target.shape[0]
        lab = target.reshape(bs, -1).astype(np.int64)
        m = np.zeros((bs, lab.shape[1], K), dtype=dtype)
        for b in range(bs):
            idx = np.nonzero(lab[b] < K)[0]
            m[b, idx, lab[b, idx]] = 1
        return m
    bs, K2, H, W = target.shape
    assert K2 == K
    return np.ascontiguousarray(target.reshape(bs, K, H * W).transpose(0, 2, 1)).astype(dtype)


def _norm(v, norm, axis):
    if norm == 2:
        return np.sqrt(np.sum(v * v, axis=axis))
    return np.sum(np.abs(v), axis=axis)


def discriminative_loss(emb, target, n_objects, max_n_objects, delta_v, delta_d, norm=2,
                        terms=SHIPPED_TERMS, normalize_means=True, dtype=np.float64, want_grad=False,
                        grad_means=None, q_den=None, grad_loss=1.0):
    """Returns dict(loss, means (bs,K,C), terms (var, dist, reg, qreg)[, grad (bs,C,H,W)]).

    q_den replaces the q-regulariser's denominator int(sum(target)) (the data-parallel run passes
    global foreground / world size).  grad is the gradient of grad_loss * loss + sum(means * grad_means):
    grad_loss scales the loss terms' part, not the grad_means part."""
    emb = np.asarray(emb)
    bs, C, H, W = emb.shape
    K = int(max_n_objects)
    P = H * W
    X = np.ascontiguousarray(emb.reshape(bs, C, P).transpose(0, 2, 1)).astype(dtype)  # bs,P,C
    M = _dense_masks(target, K, dtype)  # bs,P,K
    n_objects = [int(n) for n in np.asarray(n_objects).reshape(-1)]
    w_var, w_dist, w_reg, w_q = [dtype(t) for t in terms]

    means = np.zeros((bs, K, C), dtype=dtype)
    var_b = np.zeros(bs, dtype=dtype)
    dist_b = np.zeros(bs, dtype=dtype)
    reg_b = np.zeros(bs, dtype=dtype)
    cache = []
    with np.errstate(divide="ignore", invalid="ignore"):
        for b in range(bs):
            n = min(max(n_objects[b], 0), K)
            Mb = M[b][:, :n]
            cnt = Mb.sum(0)  # n
            s = Mb.T @ X[b]  # n,C
            mu_t = s / cnt[:, None]
            r = np.sqrt(np.sum(mu_t * mu_t, axis=1))
            mu = mu_t / r[:, None] if normalize_means else mu_t
            means[b, :n] = mu
            # variance: sum_{p,k<n} m_pk max(|x_p-mu_k|-dv,0)^2 / sum_{p,k<n} m_pk
            diff = X[b][:, None, :] - mu[None, :, :]  # P,n,C
            d = _norm(diff, norm, 2)  # P,n
            h = np.maximum(d - delta_v, 0)
            Nb = Mb.sum()
            var_b[b] = ((h * h) * Mb).sum() / Nb
            if n > 1:
                e = _norm(mu[:, None, :] - mu[None, :, :], norm, 2)
                margin = 2 * delta_d * (1.0 - np.eye(n))
                dist_b[b] = (np.maximum(margin - e, 0) ** 2).sum() / (n * (n - 1))
            reg_b[b] = _norm(mu, norm, 1).mean() if n > 0 else np.nan
            cache.append((n, Mb, cnt, mu, r, diff, d, h, Nb))
        fg = M.sum(2)  # bs,P   (all K channels)
        num = int(fg.sum()) if q_den is None else q_den
        l2 = np.sqrt(np.sum((X * fg[:, :, None]) ** 2, axis=2))
        qreg = ((l2 - 1) ** 2).sum() / dtype(num) if num != 0 else np.inf
        var_t = var_b.sum() / bs
        dist_t = dist_b.sum() / bs if w_dist != 0 else dtype(0)
        reg_t = reg_b.sum() / bs if w_reg != 0 else dtype(0)
        loss = dtype(0)
        if w_var != 0:
            loss = loss + w_var * var_t
        if w_dist != 0:
            loss = loss + w_dist * dist_t
        if w_reg != 0:
            loss = loss + w_reg * reg_t
        if w_q != 0:
            loss = loss + w_q * qreg
    out = dict(loss=loss, means=means, terms=np.array([var_t, dist_t, reg_t, qreg], dtype=dtype))
    if not want_grad:
        return out

    # ---- analytic gradient wrt emb (SURVEY.md Appendix A) ----
    G = np.zeros((bs, P, C), dtype=dtype)
    gl = dtype(grad_loss)
    with np.errstate(divide="ignore", invalid="ignore"):
        for b in range(bs):
            n, Mb, cnt, mu, r, diff, d, h, Nb = cache[b]
            if n == 0:
                continue
            if norm == 2:
                dirv = np.where(d[:, :, None] > 0, diff / np.where(d > 0, d, 1)[:, :, None], 0)
            else:
                dirv = np.sign(diff)
            gs = (2 * h * Mb)[:, :, None] * dirv  # P,n,C : d(m h^2)/dx
            cdir = gl * w_var / (bs * Nb)
            G[b] += cdir * gs.sum(1)
            Gam = -cdir * gs.sum(0)  # n,C  dL/dmu_k
            if grad_means is not None:
                Gam = Gam + np.asarray(grad_means, dtype=dtype)[b, :n]
            if w_reg != 0:
                if norm == 2:
                    nr = np.sqrt(np.sum(mu * mu, 1))
                    Gam = Gam + (gl * w_reg / bs / n) * np.where(nr[:, None] > 0, mu / np.where(nr > 0, nr, 1)[:, None], 0)
                else:
                    Gam = Gam + (gl * w_reg / bs / n) * np.sign(mu)
            if w_dist != 0 and n > 1:
                dm = mu[:, None, :] - mu[None, :, :]
                e = _norm(dm, norm, 2)
                mg = np.maximum(2 * delta_d - e, 0) * (1.0 - np.eye(n))
                if norm == 2:
                    dire = np.where(e[:, :, None] > 0, dm / np.where(e > 0, e, 1)[:, :, None], 0)
                else:
                    dire = np.sign(dm)
                Gam = Gam + (gl * w_dist / bs / (n * (n - 1))) * (-4 * mg[:, :, None] * dire).sum(1)
            if normalize_means:
                Gam = (Gam - mu * np.sum(mu * Gam, axis=1, keepdims=True)) / r[:, None]
            T = Gam / cnt[:, None]
            G[b] += Mb @ T
        if w_q != 0:
            cq = gl * w_q / dtype(num)
            sc = np.where(l2 > 0, 2 * (l2 - 1) * fg * fg / np.where(l2 > 0, l2, 1), 0)
            G += cq * sc[:, :, None] * X
    out["grad"] = np.ascontiguousarray(G.transpose(0, 2, 1)).reshape(bs, C, H, W)
    return out
