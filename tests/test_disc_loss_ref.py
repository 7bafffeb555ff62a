"""CPU: oracle/disc_loss_torch.py (float64 torch, autograd) against the numpy oracle oracle/disc_loss.py (analytic
gradient) within 1e-10, for label maps, soft and overlapping masks, every term and flag, q_den and grad_loss."""
import numpy as np
import pytest
import torch

from isa_b200 import synth
from oracle import disc_loss as O
from oracle import disc_loss_torch as T

TOL = 1e-10
ALL_TERMS = (1.0, 1.0, 0.001, 0.005)


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _targets(kind, seed, bs, C, H, W, K, n_min, n_max):
    d = synth.batch(seed, bs, C, H, W, K, n_min=n_min, n_max=n_max, pull=0.3)
    rs = np.random.RandomState(seed + 1)
    if kind == "label":
        tgt = d["labels"]
    elif kind == "soft":
        tgt = (rs.uniform(size=(bs, K, H, W)) * (rs.uniform(size=(bs, K, H, W)) > 0.5)).astype(np.float32)
    else:   # overlapping integer masks with some weights of 2
        tgt = synth.onehot(d["labels"], K, np.int64)
        tgt = tgt + (rs.uniform(size=tgt.shape) > 0.8) * rs.randint(1, 3, size=tgt.shape)
    return d["emb"], tgt, d["n_objects"]


def _both(emb, tgt, nobj, K, norm, **kw):
    o = O.discriminative_loss(emb, tgt, nobj, K, 0.5, 1.5, norm, want_grad=True, **kw)
    t = T.discriminative_loss(torch.tensor(emb), torch.tensor(tgt), torch.tensor(nobj), K, 0.5, 1.5, norm, want_grad=True, **kw)
    return o, {k: v.numpy() for k, v in t.items()}


def _assert_same(o, t):
    assert _rel(t["loss"], o["loss"]) < TOL
    assert _rel(t["terms"], o["terms"]) < TOL
    assert _rel(t["means"], o["means"]) < TOL
    assert _rel(t["grad"], o["grad"]) < TOL


@pytest.mark.parametrize("kind", ["label", "soft", "overlap"])
@pytest.mark.parametrize("norm", [1, 2])
@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("terms", [O.SHIPPED_TERMS, ALL_TERMS], ids=["shipped", "all_terms"])
def test_matches_numpy_oracle(kind, norm, normalize, terms):
    emb, tgt, nobj = _targets(kind, 3 + norm, 3, 6, 9, 11, 5, 1, 5)
    gm = np.random.RandomState(9).standard_normal((3, 5, 6)) * 0.01
    o, t = _both(emb, tgt, nobj, 5, norm, terms=terms, normalize_means=normalize, grad_means=gm)
    _assert_same(o, t)


@pytest.mark.parametrize("kind", ["label", "soft", "overlap"])
@pytest.mark.parametrize("grad_loss", [1.0, 0.37, 0.0])
def test_q_den_and_grad_loss(kind, grad_loss):
    emb, tgt, nobj = _targets(kind, 21, 2, 5, 8, 13, 4, 2, 4)
    fg = int(O._dense_masks(tgt, 4, np.float64).sum())
    gm = np.random.RandomState(4).standard_normal((2, 4, 5)) * 0.02
    for q_den in (None, 1.7 * fg):
        o, t = _both(emb, tgt, nobj, 4, 2, terms=ALL_TERMS, q_den=q_den, grad_loss=grad_loss, grad_means=gm)
        _assert_same(o, t)
    if grad_loss == 0.0:    # only the grad_means part is left
        assert np.abs(t["grad"]).max() > 0


def test_q_den_scales_the_q_regulariser():
    emb, tgt, nobj = _targets("label", 5, 2, 4, 7, 9, 3, 1, 3)
    a, _ = _both(emb, tgt, nobj, 3, 2)
    fg = int((tgt < 3).sum())
    b, _ = _both(emb, tgt, nobj, 3, 2, q_den=2.5 * fg)
    assert abs(b["terms"][3] * 2.5 - a["terms"][3]) < 1e-12 * a["terms"][3]


def test_n_objects_above_K_and_labels_above_K():
    # n_objects is clamped to K; labels in [K, 255) are background for every term
    emb, tgt, _ = _targets("label", 8, 2, 6, 10, 10, 6, 6, 6)
    tgt = tgt.copy()
    tgt[0, :2] = 7
    tgt[1, -1] = 200
    K = 4
    tgt[tgt == 4] = 0
    tgt[tgt == 5] = 1
    o, t = _both(emb, tgt, np.array([9, 4], dtype=np.int32), K, 2, terms=ALL_TERMS)
    _assert_same(o, t)
    o2, _ = _both(emb, np.where(tgt >= K, 255, tgt).astype(np.uint8), np.array([4, 4], dtype=np.int32), K, 2, terms=ALL_TERMS)
    assert _rel(o["loss"], o2["loss"]) < TOL


@pytest.mark.parametrize("kind", ["label", "soft"])
def test_absent_instance_gives_nan_where_the_oracle_does(kind):
    emb, tgt, _ = _targets(kind, 13, 2, 5, 8, 8, 4, 2, 2)
    tgt = tgt.copy()
    if kind == "label":
        tgt[0][tgt[0] == 1] = 0
    else:
        tgt[0, 1] = 0
    nobj = np.array([3, 2], dtype=np.int32)
    o, t = _both(emb, tgt, nobj, 4, 2, terms=ALL_TERMS)
    assert np.isnan(o["loss"]) and np.isnan(t["loss"])
    for key in ("terms", "means"):
        assert np.array_equal(np.isnan(o[key]), np.isnan(t[key])), key
        fin = ~np.isnan(o[key])
        assert _rel(t[key][fin], o[key][fin]) < TOL
    # image 1 is untouched; in image 0 the torch form is NaN only where the kernels are (pixels of its instances)
    assert not np.isnan(t["grad"][1]).any()
    assert _rel(t["grad"][1], o["grad"][1]) < TOL
    nan0 = np.isnan(t["grad"][0]).any(0)
    inst0 = (O._dense_masks(tgt, 4, np.float64)[0, :, :3] != 0).any(1).reshape(8, 8)
    assert np.array_equal(nan0, inst0)
