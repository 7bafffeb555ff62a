"""CPU: the float64 oracle of the instance-count branch (oracle/count_head_ref.py) -- its hand-written tail gradient
against autograd, its rounding rule, and the parameter names it shares with isa_b200.archs.ReSeg(count_head=True)."""
import numpy as np
import pytest
import torch

from oracle import count_head_ref as CH


def test_tail_gradient_matches_autograd():
    torch.manual_seed(0)
    for n, C, H, W, K in ((3, 64, 4, 4, 32), (1, 8, 1, 7, 1), (5, 4, 6, 3, 64)):
        x = (torch.randn(n, C, H, W, dtype=torch.float64) - 0.3).requires_grad_(True)
        cb = (0.1 * torch.randn(C, dtype=torch.float64)).requires_grad_(True)
        w = torch.randn(C, dtype=torch.float64).requires_grad_(True)
        b = torch.randn(1, dtype=torch.float64).requires_grad_(True)
        x.data[:, 0] = -5.0                       # a channel ReLU kills everywhere
        nobj = torch.randint(0, K + 1, (n,))
        y = torch.relu(x + cb.view(1, C, 1, 1))
        pooled, s = CH.tail(y, w, b)
        loss = CH.count_loss(s, nobj, K)
        loss.backward(torch.tensor(0.7, dtype=torch.float64))
        gx, dcb, dw, db = CH.tail_grad(y.detach(), pooled.detach(), s.detach(), w.detach(), nobj, K, grad_loss=0.7)
        for got, want in ((gx, x.grad), (dcb, cb.grad), (dw, w.grad), (db, b.grad)):
            assert float((got - want).abs().max()) < 1e-10
        assert float(x.grad[:, 0].abs().max()) == 0.0


def test_count_rounding_rule_with_exact_ties():
    K = 4
    # s * K exactly representable halves: 0.5 -> 0 -> clamp 1, 1.5 -> 2, 2.5 -> 2, 3.5 -> 4 (half to even)
    s = torch.tensor([0.125, 0.375, 0.625, 0.875, 0.0, 1.0, 0.3, 0.99], dtype=torch.float64)
    got = CH.n_pred(s, K).tolist()
    assert got == [1, 2, 2, 4, 1, 4, 1, 4]
    for K in (1, 7, 32, 64, 254):
        s = torch.cat([(torch.arange(0, 2 * K + 1, dtype=torch.float64) / (2 * K)), torch.rand(100, dtype=torch.float64)])
        want = [min(max(round(float(v) * K), 1), K) for v in s]     # Python's round() is half to even
        assert CH.n_pred(s, K).tolist() == want


def test_branch_parameter_names_match_reseg():
    from isa_b200.archs import ReSeg
    net = ReSeg(2, n_units=20, count_head=True, max_n_objects=32)
    ref = CH.CountBranchRef(2 * 20 + 24)
    mine = {k: tuple(v.shape) for k, v in net.state_dict().items() if k.startswith(("ins_cls_cnn.", "ins_cls_out."))}
    theirs = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    assert mine == theirs
    assert sorted(mine) == sorted(["ins_cls_cnn.conv%d.%s" % (i, p) for i in range(1, 5) for p in ("weight", "bias")]
                                  + ["ins_cls_out.linear.weight", "ins_cls_out.linear.bias"])
    # a head-less network's state_dict is unchanged
    assert not any(k.startswith("ins_cls") for k in ReSeg(2, n_units=20).state_dict())


def test_count_head_arguments_are_checked():
    from isa_b200.archs import ReSeg
    with pytest.raises(ValueError):
        ReSeg(2, n_units=20, count_head=True)
    with pytest.raises(ValueError):
        ReSeg(2, n_units=20, count_head=True, max_n_objects=255)
    net = ReSeg(2, n_units=20, count_head=True, max_n_objects=8)
    for h, w in ((12, 64), (64, 15)):
        with pytest.raises(ValueError):
            net(False, torch.zeros(1, 3, h, w))


def test_oracle_branch_runs_end_to_end():
    torch.manual_seed(1)
    ref = CH.CountBranchRef(16).double()
    y = torch.randn(2, 16, 16, 12, dtype=torch.float64)
    f, pooled, s = ref(y)
    assert f.shape == (2, 64, 4, 3) and pooled.shape == (2, 64) and s.shape == (2,)
    p2, s2 = CH.tail(f, ref.ins_cls_out.linear.weight, ref.ins_cls_out.linear.bias)
    assert torch.equal(p2, pooled) and torch.allclose(s2, s, rtol=0, atol=1e-15)
    assert np.all((CH.n_pred(s, 16).numpy() >= 1) & (CH.n_pred(s, 16).numpy() <= 16))
