"""GPU: isa_augment against its numpy restatement (oracle/augment_ref.py) -- labels, class maps and counts bit for bit,
the normalised image within 3e-5 -- and the resident loader feeding Model.fit, the CUDA-graph step, data-parallel
shards and the train.py -> pred_list.py -> evaluate.py round trip."""
import ctypes
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from PIL import Image

from isa_b200 import _lib, parallel, settings, synth
from isa_b200 import augment as A
from oracle import augment_ref as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MEAN = [0.521697844321, 0.389775426267, 0.206216114391]
STD = [0.212398291819, 0.151755427041, 0.113022107204]


def _pair(seed, h, w, n):
    rs = np.random.RandomState(seed)
    rgb = rs.randint(0, 256, size=(h, w, 3)).astype(np.uint8)
    lab = synth.label_map(rs, h, w, n) if h * w >= n else np.zeros((h, w), np.uint8)
    return rgb, lab


def _store(pairs, dev):
    return A.ImageStore(["img%d" % i for i in range(len(pairs))], [p[0] for p in pairs], [p[1] for p in pairs],
                        MEAN, STD, dev)


def _check(store, pairs, table, H, W, dev):
    got = A.augment(store, torch.from_numpy(np.asarray(table, np.int64)).to(dev), H, W)
    torch.cuda.synchronize()
    want = R.augment([p[0] for p in pairs], [p[1] for p in pairs], table, H, W, MEAN, STD)
    img, sem, ins, n = got
    assert img.is_contiguous(memory_format=torch.channels_last) and img.shape == (len(table), 3, H, W)
    assert np.array_equal(ins.cpu().numpy(), want["ins"])
    assert np.array_equal(sem.cpu().numpy(), want["sem"])
    assert np.array_equal(n.cpu().numpy(), want["n_objects"])
    err = np.abs(img.permute(0, 2, 3, 1).cpu().double().numpy() - want["image"]).max()
    assert err <= 3e-5, err
    return got, want


def test_every_flag_combination(cuda):
    pairs = [_pair(1, 37, 29, 6), _pair(2, 30, 30, 5), _pair(3, 16, 40, 4)]
    store = _store(pairs, cuda)
    for i, bits in enumerate(itertools.product([False, True], repeat=6)):
        flags = dict(zip(A.IMPLEMENTED, bits))
        for epoch in range(2):
            _check(store, pairs, A.epoch_table(store.sizes, 24, 20, flags, 100 + i, epoch), 24, 20, cuda)


@pytest.mark.parametrize("theta", [0.0, 45.0, 90.0])
@pytest.mark.parametrize("center_cut", [False, True])
def test_exact_angles(cuda, theta, center_cut):
    pairs = [_pair(4, 33, 47, 7), _pair(5, 40, 40, 6)]
    store = _store(pairs, cuda)
    table = [[i] + list(A.quantise(A.inverse_map(h, w, 32, 36, theta=theta, center_cut=center_cut)))
             for i, (h, w) in enumerate(store.sizes)]
    _check(store, pairs, table, 32, 36, cuda)


def test_cvppp_shape_batch16(cuda):
    pairs = [(synth.leaf_image(i, 530, 500), synth.label_map(np.random.RandomState(i), 530, 500, 20)) for i in range(4)]
    store = _store(pairs, cuda)
    flags = A.flags_from_settings(settings.CVPPPTrainingSettings())
    table = np.concatenate([A.epoch_table(store.sizes, 256, 256, flags, 23, e) for e in range(4)])
    _check(store, pairs, table, 256, 256, cuda)


def test_cityscapes_shape_batch2(cuda):
    pairs = [_pair(6, 1024, 2048, 64), _pair(7, 1024, 2048, 40)]
    store = _store(pairs, cuda)
    table = [[i] + list(A.quantise(A.inverse_map(1024, 2048, 1024, 2048, hflip=i == 1, theta=7.5 + 20 * i,
                                                 center_cut=True))) for i in range(2)]
    got, _ = _check(store, pairs, table, 1024, 2048, cuda)
    assert int(got[3].max()) > 30


@pytest.mark.parametrize("src,out", [((1, 1), (1, 1)), ((1, 1), (5, 3)), ((1, 9), (1, 9)), ((1, 9), (3, 4)),
                                     ((8, 1), (8, 1)), ((8, 1), (2, 1)), ((5, 7), (1, 1)), ((13, 11), (61, 57))])
def test_small_and_upscaled_shapes(cuda, src, out):
    h, w = src
    lab = (np.arange(h * w) % 3).reshape(h, w).astype(np.uint8)
    pairs = [(np.random.RandomState(h * w).randint(0, 256, (h, w, 3)).astype(np.uint8), lab)]
    store = _store(pairs, cuda)
    flags = {k: True for k in A.IMPLEMENTED}
    table = np.concatenate([A.plain_table(store.sizes, *out), A.epoch_table(store.sizes, out[0], out[1], flags, 3, 0)])
    _check(store, pairs, table, out[0], out[1], cuda)


def test_64_ids_and_dropped_instances_are_renumbered(cuda):
    pairs = [_pair(8, 96, 96, 64), _pair(9, 200, 180, 64)]
    store = _store(pairs, cuda)
    # 8x8 samples of 64 cells in an ellipse over half the image: most cells are dropped, the survivors renumbered 0..n-1
    got, _ = _check(store, pairs, A.plain_table(store.sizes, 96, 96), 96, 96, cuda)
    assert int(got[3][0]) == 64
    got, _ = _check(store, pairs, A.plain_table(store.sizes, 8, 8), 8, 8, cuda)
    for i in range(2):
        n = int(got[3][i])
        assert n < 64 and set(np.unique(got[2][i].cpu().numpy())) == set(range(n)) | {255}


def test_sample_that_loses_every_instance_falls_back(cuda):
    rgb = np.random.RandomState(10).randint(0, 256, (20, 20, 3)).astype(np.uint8)
    lab = np.full((20, 20), 255, np.uint8)
    lab[15:, 15:] = 4            # one instance in a corner, id 4 in the store
    lab[0, 19] = 2
    pairs = [(rgb, lab)]
    store = _store(pairs, cuda)
    cut = A.quantise(A.inverse_map(20, 20, 10, 10) @ np.array([[0.5, 0, 0], [0, 0.5, 0], [0, 0, 1]]))   # top-left quarter
    table = [[0] + list(cut), [0] + list(A.plain_map(20, 20, 10, 10))]
    got, want = _check(store, pairs, table, 10, 10, cuda)
    for i in range(2):
        assert np.array_equal(got[2][i].cpu().numpy(), got[2][1].cpu().numpy())
        assert np.array_equal(got[0][i].cpu().numpy(), got[0][1].cpu().numpy())
    assert int(got[3][0]) == 1      # id 2 (one pixel) is not sampled at this scale; id 4 is renumbered 0


def test_invalid_source_index_or_map(cuda):
    pairs = [_pair(11, 16, 16, 3)]
    store = _store(pairs, cuda)
    table = torch.tensor([[5] + list(A.plain_map(16, 16, 8, 8)), [0] + [1 << 50, 0, 0, 0, 1 << 32, 0],
                          [0] + list(A.plain_map(16, 16, 8, 8))], dtype=torch.int64, device=cuda)
    img, sem, ins, n = A.augment(store, table, 8, 8)
    # a source index out of range: black and empty; a map out of range: no instance, so the plain view
    assert int(n[0]) == 0 and (ins[0] == 255).all() and (sem[0] == 0).all()
    assert int(n[1]) == int(n[2]) > 0 and torch.equal(ins[1], ins[2]) and torch.equal(img[1], img[2])


def test_two_calls_write_identical_bytes(cuda):
    pairs = [_pair(12, 530, 500, 25), _pair(13, 480, 510, 25)]
    store = _store(pairs, cuda)
    flags = A.flags_from_settings(settings.CVPPPTrainingSettings())
    table = torch.from_numpy(np.concatenate([A.epoch_table(store.sizes, 256, 256, flags, 1, e) for e in range(8)])).to(cuda)
    a = A.augment(store, table, 256, 256)
    b = A.augment(store, table, 256, 256)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_rejects_bad_arguments(cuda):
    lib = _lib.load()
    pairs = [_pair(14, 8, 8, 2)]
    store = _store(pairs, cuda)
    params = torch.from_numpy(A.plain_table(store.sizes, 4, 4)).to(cuda)
    img = torch.full((1, 4, 4, 3), 7.0, device=cuda)
    sem = torch.full((1, 4, 4), 7, device=cuda, dtype=torch.uint8)
    ins = sem.clone()
    n = torch.full((1,), 7, device=cuda, dtype=torch.int32)
    ws = torch.zeros(1024, device=cuda, dtype=torch.uint8)
    ms = store.mean_std
    bad_std = (ctypes.c_float * 6)(0.5, 0.5, 0.5, 0.2, 0.0, 0.2)
    ok = dict(rgb=store.rgb.data_ptr(), lab=store.labels.data_ptr(), table=store.table.data_ptr(), n_images=1,
              pixels=store.labels.numel(), params=params.data_ptr(), b=1, H=4, W=4, ms=ms, img=img.data_ptr(),
              sem=sem.data_ptr(), ins=ins.data_ptr(), n=n.data_ptr(), ws=ws.data_ptr(), wsb=1024)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.isa_augment(a["rgb"], a["lab"], a["table"], a["n_images"], a["pixels"], a["params"], a["b"], a["H"],
                               a["W"], a["ms"], a["img"], a["sem"], a["ins"], a["n"], a["ws"], a["wsb"], _lib.stream_ptr())

    for kw in [dict(rgb=None), dict(lab=None), dict(table=None), dict(params=None), dict(ms=None), dict(img=None),
               dict(sem=None), dict(ins=None), dict(n=None), dict(ws=None), dict(b=0), dict(b=-1), dict(H=0), dict(W=0),
               dict(H=40000), dict(W=32768), dict(n_images=0), dict(pixels=0), dict(ms=bad_std),
               dict(img=img.data_ptr() + 2)]:
        assert call(**kw) == -1, kw
    assert call(wsb=lib.isa_augment_workspace_bytes(1) - 1) == -3
    torch.cuda.synchronize()
    assert (img == 7).all() and (sem == 7).all() and (ins == 7).all() and (n == 7).all()
    assert call() == 0
    torch.cuda.synchronize()
    assert int(n[0]) > 0


# ---------------------------------------------------------------------------------------------------- loader
def _cvppp_dir(tmp_path, n, h=120, w=110, n_inst=4):
    out = str(tmp_path)
    gt = os.path.join(out, "gt")
    os.makedirs(gt, exist_ok=True)
    names = []
    for j in range(n):
        nm = "plant%03d_rgb" % j
        Image.fromarray(synth.leaf_image(j, h, w)).save(os.path.join(out, nm + ".png"))
        lab = synth.label_map(np.random.RandomState(j), h, w, n_inst + j % 3).astype(np.int64) + 1
        lab[lab == 256] = 0
        Image.fromarray(lab.astype(np.uint8)).save(os.path.join(gt, "plant%03d_label.png" % j))
        Image.fromarray((lab > 0).astype(np.uint8)).save(os.path.join(gt, "plant%03d_fg.png" % j))
        names.append(os.path.join(out, nm + ".png"))
    lst = os.path.join(out, "all.lst")
    with open(lst, "w") as f:
        f.write("\n".join(names) + "\n")
    return lst, gt


def _flags():
    return A.flags_from_settings(settings.CVPPPTrainingSettings())


def test_load_store_matches_the_files(cuda, tmp_path):
    lst, gt = _cvppp_dir(tmp_path, 3)
    store = A.load_store(lst, gt, 32, 64, 64, MEAN, STD, cuda)
    for i, p in enumerate(A.read_list(lst)):
        rgb, lab = A.read_pair(p, gt, 32)
        off, h, w = store.table[i].tolist()
        assert (h, w) == lab.shape
        assert np.array_equal(store.labels[off:off + h * w].cpu().numpy(), lab.reshape(-1))
        assert np.array_equal(store.rgb[3 * off:3 * (off + h * w)].cpu().numpy(), rgb.reshape(-1))


def test_load_refuses_an_image_without_instance_in_its_plain_view(cuda, tmp_path):
    lst, gt = _cvppp_dir(tmp_path, 2)
    lab = np.zeros((120, 110), np.uint8)
    # one pixel at (1, 1): the 64x64 plain view samples source columns 0, 2, 4, ... (x = 1.72 (i + 0.5)) and rows
    # 0, 2, 4, ... (y = 1.875 (j + 0.5)), so it is never read
    lab[1, 1] = 9
    Image.fromarray(lab).save(os.path.join(gt, "plant001_label.png"))
    with pytest.raises(ValueError, match="plant001_label.png: no instance left"):
        A.load_store(lst, gt, 32, 64, 64, MEAN, STD, cuda)


@pytest.mark.parametrize("world", [2, 4])
def test_ranks_yield_their_shard_of_the_global_batch(cuda, tmp_path, world):
    lst, gt = _cvppp_dir(tmp_path, 10)
    store = A.load_store(lst, gt, 32, 64, 64, MEAN, STD, cuda)
    for train in (True, False):
        full = list(A.AugmentLoader(store, 4, 64, 64, _flags(), 23, train).batches(3))
        shards = [list(A.AugmentLoader(store, 4, 64, 64, _flags(), 23, train, r, world).batches(3)) for r in range(world)]
        if train:           # 10 images, global batch 4: the partial third batch is dropped
            assert len(full) == 2
            for j, g in enumerate(full):
                for r in range(world):
                    lo, hi = parallel.shard_range(4, r, world)
                    for x, y in zip(shards[r][j], g):
                        assert torch.equal(x, y[lo:hi])
        else:               # every image scored once, in list order, on the same number of steps on every rank
            assert len(set(len(s) for s in shards)) == 1 and all(b[0].shape[0] > 0 for s in shards for b in s)
            for k in range(4):
                whole = torch.cat([g[k] for g in full])
                assert torch.equal(torch.cat([b[k] for j in range(len(shards[0])) for s in shards for b in [s[j]]]), whole)


def test_same_seed_and_epoch_same_batches(cuda, tmp_path):
    lst, gt = _cvppp_dir(tmp_path, 6)
    store = A.load_store(lst, gt, 32, 64, 64, MEAN, STD, cuda)
    ld = A.AugmentLoader(store, 2, 64, 64, _flags(), 23, True)
    e0, e1 = list(ld), list(ld)            # epochs 0 and 1
    again = list(A.AugmentLoader(store, 2, 64, 64, _flags(), 23, True).batches(0))
    for x, y in zip(e0, again):
        for s, t in zip(x, y):
            assert torch.equal(s, t)
    assert not all(torch.equal(x[2], y[2]) for x, y in zip(e0, e1))
    for x in e0 + e1:
        assert (x[3] > 0).all()


def _model(cuda, count_head):
    from isa_b200.model import Model
    torch.manual_seed(23)
    return Model('CVPPP', 'ReSeg', 2, 32, use_instance_segmentation=True, n_embedding=24, device=cuda, count_head=count_head)


@pytest.mark.parametrize("count_head", [False, True])
def test_fit_on_a_directory(cuda, tmp_path, count_head):
    lst, gt = _cvppp_dir(tmp_path, 6)
    ts = settings.CVPPPTrainingSettings()
    store = A.load_store(lst, gt, 32, 64, 64, ts.MEAN, ts.STD, cuda)
    m = _model(cuda, count_head)
    hist = m.fit(ts.CRITERION, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM, ts.LEARNING_RATE, ts.WEIGHT_DECAY, ts.CLIP_GRAD_NORM,
                 ts.LR_DROP_FACTOR, ts.LR_DROP_PATIENCE, ts.OPTIMIZE_BG, ts.OPTIMIZER, ts.TRAIN_CNN, 3, None,
                 A.AugmentLoader(store, 2, 64, 64, _flags(), ts.SEED, True),
                 A.AugmentLoader(store, 4, 64, 64, _flags(), ts.SEED, False), os.path.join(str(tmp_path), "models"))
    assert len(hist) == 3
    for _, tr, va in hist:
        assert np.isfinite(tr) and np.isfinite(va)


def test_cuda_graph_step_from_the_loader_equals_eager(cuda, tmp_path):
    lst, gt = _cvppp_dir(tmp_path, 4)
    store = A.load_store(lst, gt, 32, 64, 64, MEAN, STD, cuda)
    runs = []
    for graph in (False, True):
        m = _model(cuda, True)
        m.define_criterion(None, 0.5, 1.5, 2, False, 'Multi')
        m.define_optimizer(1.0, 0.001, 0.5, 25, 'Adadelta')
        if graph:
            m.enable_cuda_graph(warmup_steps=2)
        ld = A.AugmentLoader(store, 2, 64, 64, _flags(), 23, True)
        costs = []
        for _ in range(3):
            for b in ld:
                costs.append(float(m.train_step(*b, clip_grad_norm=10.0)['Cost']))
        if graph:
            assert len(m._graphs) == 1
        runs.append((costs, torch.cat([p.detach().reshape(-1) for p in m.model.parameters()]).clone()))
    (c0, p0), (c1, p1) = runs
    assert c1[0] == c0[0]
    np.testing.assert_allclose(c1, c0, rtol=2e-4)
    assert float((p1 - p0).abs().max()) <= 1e-3 * float(p0.abs().max())


def _run(args):
    r = subprocess.run([sys.executable] + args, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


def test_train_pred_evaluate_on_one_directory(cuda, tmp_path):
    lst, gt = _cvppp_dir(tmp_path, 4)
    out = str(tmp_path)
    with open(os.path.join(out, "counts.txt"), "w") as f:
        f.write("".join("plant%03d,%d\n" % (j, 4 + j % 3) for j in range(4)))
    txt = _run([os.path.join(ROOT, "code", "train.py"), "--nepochs", "2", "--batchsize", "2", "--train_list", lst,
                "--val_list", lst, "--gt_dir", gt, "--count_head", "--cuda_graph", "--output", os.path.join(out, "models")])
    assert "image store: 4 images" in txt
    ckpts = sorted(f for f in os.listdir(os.path.join(out, "models", "CVPPP")) if f.endswith(".pth"))
    assert ckpts
    _run([os.path.join(ROOT, "code", "pred_list.py"), "--lst", lst, "--count_head", "--model",
          os.path.join(out, "models", "CVPPP", ckpts[-1]), "--output", os.path.join(out, "pred")])
    txt = _run([os.path.join(ROOT, "code", "evaluate.py"), "--pred_dir", os.path.join(out, "pred"), "--dataset", "CVPPP",
                "--names", lst, "--counts", os.path.join(out, "counts.txt"), "--gt_dir", gt, "--empty_as_zero"])
    assert "MEAN SBD" in txt and "MEAN |DIC|" in txt
