"""GPU: the clustering kernels through the C-ABI.
  * bit-exact against the deterministic oracle (labels, k-means++ picks, n_iter, inertia, centres);
  * identical partitions (up to label permutation) to golden labels from the real scikit-learn;
  * fg compaction / label scatter / nearest up-sampling bit-exact against numpy + OpenCV."""
import os
import sys

import numpy as np
import pytest
import torch

from isa_b200 import synth
from oracle import kmeans as KM

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden_kmeans import KM_CASES, NET_CASES, case_inputs, net_inputs  # noqa: E402

pytestmark = pytest.mark.gpu


def _gpu_fit(dev, X, k, **kw):
    from isa_b200 import clustering
    labels, res = clustering.kmeans_fit_predict(torch.tensor(X, device=dev), k, **kw)
    torch.cuda.synchronize()
    return labels.cpu().numpy(), res


def _assert_same_as_oracle(labels, res, o):
    assert np.array_equal(res.seed_idx.cpu().numpy(), o["seed_idx"]), "k-means++ picks differ"
    assert np.array_equal(res.n_iter.cpu().numpy(), o["n_iter"]), (res.n_iter.cpu().numpy(), o["n_iter"])
    assert np.array_equal(res.inertia.cpu().numpy(), o["inertia"]), "inertia differs"
    assert res.best == o["best"]
    assert np.array_equal(labels, o["labels"]), "labels differ"
    assert np.array_equal(res.centers.cpu().numpy(), o["centers"]), "centres differ"


@pytest.mark.parametrize("case", KM_CASES, ids=[c[0] for c in KM_CASES])
def test_bit_exact_vs_oracle_and_sklearn_golden(cuda, golden_dir, case):
    name, seed, C, H, W, k, pull, n_init, km_seed = case
    g = np.load(os.path.join(golden_dir, "kmeans.npz"))
    sem, emb = case_inputs(case)
    _, X = KM.gather_foreground(sem, emb)
    o = KM.kmeans_oracle(X, k, seed=km_seed, n_init=n_init)
    labels, res = _gpu_fit(cuda, X, k, seed=km_seed, n_init=n_init)
    _assert_same_as_oracle(labels, res, o)
    assert KM.same_up_to_permutation(labels, g[name + "_sk_labels"])
    # Lloyd from scikit-learn's own seeds
    inits = g[name + "_inits"]
    for r in range(inits.shape[0]):
        lab_r, _ = _gpu_fit(cuda, X, k, n_init=1, init_centers=inits[r:r + 1])
        assert KM.same_up_to_permutation(lab_r, g[name + "_init_labels"][r])


@pytest.mark.parametrize("case", NET_CASES, ids=[c[0] for c in NET_CASES])
def test_network_embeddings_bit_exact_and_sklearn_golden(cuda, golden_dir, case):
    """Near-tied random-init network embeddings: scikit-learn's seeds, scikit-learn's partition."""
    name, k, n_init, km_seed = case
    g = np.load(os.path.join(golden_dir, "kmeans.npz"))
    X = net_inputs(name)
    o = KM.kmeans_oracle(X, k, seed=km_seed, n_init=n_init)
    labels, res = _gpu_fit(cuda, X, k, seed=km_seed, n_init=n_init)
    _assert_same_as_oracle(labels, res, o)
    assert np.array_equal(res.seed_idx.cpu().numpy()[0], g[name + "_sk_first_seeds"])
    assert KM.same_up_to_permutation(labels, g[name + "_sk_labels"])


def _planted_3001():
    rs = np.random.RandomState(1)
    cent = rs.standard_normal((20, 12)) * 2
    return (cent[rs.randint(0, 20, 3001)] + rs.standard_normal((3001, 12))).astype(np.float32)


@pytest.mark.parametrize("data,k,n_init,seed", [("net0", 16, 8, 0), ("net0", 40, 4, 0), ("planted", 40, 5, 4)],
                         ids=["net0_k16_packed_fp32", "net0_k40_tensor_core", "planted_k40_tensor_core"])
def test_lloyd_paths_bit_exact(cuda, data, k, n_init, seed):
    """The Lloyd E-step paths, each reached through its input, reproduce the oracle bit for bit: the packed-FP32 kernel
    with the Hamerly bounds on a near-tied network embedding (k = 16), the tensor-core filter on the same embedding
    (k = 40) and on a planted case with few points per centre (k = 40, C = 12)."""
    X = net_inputs("net0") if data == "net0" else _planted_3001()
    o = KM.kmeans_oracle(X, k, seed=seed, n_init=n_init)
    labels, res = _gpu_fit(cuda, X, k, seed=seed, n_init=n_init)
    _assert_same_as_oracle(labels, res, o)
    if k <= 32:
        assert int(res.n_iter.max()) > 32, "the bounded E-step (from Lloyd iteration 32 on) never ran"


def test_cumsum_search_edge_cases(cuda):
    """The parallel float32 running-sum search against the oracle's sequential loop on inputs that stress it: exact ties
    (dyadic coordinates), long runs of zero distances (duplicates of the first centre), a heavy tail, a point count that
    is not a multiple of anything, fewer CTAs than restarts."""
    rs = np.random.RandomState(3)
    cases = []
    cases.append(((rs.randint(0, 8, size=(9001, 4)) / 4.0).astype(np.float32), 6, 9))
    X = rs.standard_normal((20011, 6)).astype(np.float32)
    X[:5000] = X[0]
    cases.append((X, 5, 12))
    cases.append((np.exp(3 * rs.standard_normal((33333, 3))).astype(np.float32), 7, 8))
    cases.append((rs.standard_normal((300, 2)).astype(np.float32), 4, 35))
    for X, k, n_init in cases:
        o = KM.kmeans_oracle(X, k, seed=1, n_init=n_init, max_iter=5)
        labels, res = _gpu_fit(cuda, X, k, seed=1, n_init=n_init, max_iter=5)
        _assert_same_as_oracle(labels, res, o)


@pytest.mark.parametrize("n,C,k,n_init", [(1000, 3, 1, 2), (5000, 5, 7, 4), (40000, 24, 16, 6), (20000, 32, 64, 2),
                                          (3000, 40, 5, 3), (777, 16, 200, 2), (1025, 8, 3, 35)])
def test_bit_exact_vs_oracle_shapes(cuda, n, C, k, n_init):
    rs = np.random.RandomState(n + C)
    cent = rs.standard_normal((max(k // 2, 1), C)) * 2
    X = (cent[rs.randint(0, len(cent), n)] + rs.standard_normal((n, C))).astype(np.float32) + 3.0
    o = KM.kmeans_oracle(X, k, seed=11, n_init=n_init, max_iter=60)
    labels, res = _gpu_fit(cuda, X, k, seed=11, n_init=n_init, max_iter=60)
    _assert_same_as_oracle(labels, res, o)


def test_empty_cluster_relocation_and_duplicates(cuda):
    X = np.repeat(np.array([[0, 0], [1, 1], [5, 5], [5, 6]], dtype=np.float32), 64, axis=0)
    for k in (4, 6, 9):
        o = KM.kmeans_oracle(X, k, seed=2, n_init=5)
        labels, res = _gpu_fit(cuda, X, k, seed=2, n_init=5)
        _assert_same_as_oracle(labels, res, o)
    # array init that leaves clusters empty on the first E-step
    rs = np.random.RandomState(0)
    Xr = rs.standard_normal((4000, 6)).astype(np.float32)
    init = np.concatenate([Xr[:3], 100 + rs.standard_normal((3, 6)).astype(np.float32)])[None]
    o = KM.kmeans_oracle(Xr, 6, n_init=1, init_centers=init)
    labels, res = _gpu_fit(cuda, Xr, 6, n_init=1, init_centers=init)
    assert np.array_equal(res.n_iter.cpu().numpy(), o["n_iter"])
    assert np.array_equal(labels, o["labels"])
    assert np.array_equal(res.inertia.cpu().numpy(), o["inertia"])


def test_errors_like_sklearn(cuda):
    from isa_b200 import _lib, clustering
    with pytest.raises(ValueError):
        clustering.kmeans_fit_predict(torch.zeros(3, 2, device=cuda), 5)
    bad = torch.tensor([[float("nan"), 0], [1, 1], [2, 2]], device=cuda)
    with pytest.raises(ValueError):
        clustering.kmeans_fit_predict(bad, 2)
    with pytest.raises(_lib.IsaError):
        clustering.kmeans_fit_predict(torch.zeros(30, 2, device=cuda), 300)
    with pytest.raises(_lib.IsaError):
        clustering.kmeans_fit_predict(torch.zeros(30, 2), 3)


@pytest.mark.parametrize("h,w,oh,ow,ncls", [(64, 80, 133, 171, 2), (256, 256, 530, 500, 2), (33, 47, 33, 47, 3), (128, 96, 50, 40, 2)])
def test_compaction_scatter_upsample(cuda, h, w, oh, ow, ncls):
    from isa_b200 import clustering
    rs = np.random.RandomState(h * w)
    sem = rs.uniform(size=(ncls, h, w)).astype(np.float32)
    sem[:, :3, :] = 0.5  # ties -> class 0 like np.argmax
    emb = rs.standard_normal((5, h, w)).astype(np.float32)
    fg_ref, X_ref = KM.gather_foreground(sem, emb)
    cls_map, Xt, fg_index, n_dev = clustering.fg_compact(torch.tensor(sem, device=cuda), torch.tensor(emb, device=cuda))
    n = int(n_dev)
    assert n == len(X_ref)
    assert np.array_equal(cls_map.cpu().numpy(), fg_ref)
    assert np.array_equal(Xt[:, :n].t().cpu().numpy(), X_ref)
    ys, xs = np.where(fg_ref != 0)
    assert np.array_equal(fg_index[:n].cpu().numpy(), ys * w + xs)
    labels = rs.randint(0, 16, size=h * w).astype(np.int32)
    ins_small, ins_up, cls_up = clustering.scatter_labels_upsample(torch.tensor(labels, device=cuda), fg_index, n_dev, cls_map, oh, ow)
    ref_small = KM.scatter_labels(fg_ref, labels[:n])
    assert np.array_equal(ins_small.cpu().numpy(), ref_small)
    assert np.array_equal(ins_up.cpu().numpy(), KM.upsample_nearest(ref_small, oh, ow))
    assert np.array_equal(cls_up.cpu().numpy(), KM.upsample_nearest(fg_ref, oh, ow))


def test_cluster_pipeline_cvppp_shape(cuda):
    """CVPPP-shaped end to end (256x256 net size, k=16, n_init=35, raw 530x500): device pipeline ==
    oracle pipeline bit for bit, and idempotent."""
    from isa_b200 import clustering
    d = synth.batch(42, 1, 24, 256, 256, 32, n_min=16, n_max=16, pull=0.75)
    lab = d["labels"][0]
    sem = np.stack([(lab == 255).astype(np.float32), (lab != 255).astype(np.float32)])
    emb = d["emb"][0]
    out = clustering.cluster_embeddings(torch.tensor(sem, device=cuda), torch.tensor(emb, device=cuda), 16, 530, 500, seed=0)
    cls_map, ins_small, ins_up, cls_up, res = out
    res.check()
    fg, mask = KM.cluster_reference(sem, emb, 16, seed=0, impl="oracle")
    assert np.array_equal(ins_small.cpu().numpy(), mask)
    assert np.array_equal(ins_up.cpu().numpy(), KM.upsample_nearest(mask, 530, 500))
    out2 = clustering.cluster_embeddings(torch.tensor(sem, device=cuda), torch.tensor(emb, device=cuda), 16, 530, 500, seed=0)
    assert torch.equal(out2[2], ins_up)
