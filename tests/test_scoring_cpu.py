"""CPU: the host side of validation scoring (isa_b200.scoring) -- the list-order means, the padded gather of the per-image
scores over a gloo world of 2, the loading of the ground truth, and the argument errors of Model.fit and train.py."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _values(n, seed=0):
    """(n, 4) per-image scores whose float64 sum depends on the order of the additions."""
    rs = np.random.RandomState(seed)
    v = np.empty((n, 4))
    v[:, 0] = rs.rand(n) * 10.0 ** rs.randint(-8, 1, n)
    v[:, 1] = rs.randint(0, 9, n)
    v[:, 2] = rs.rand(n) / 3.0
    v[:, 3] = rs.rand(n) < 0.2
    return v


def test_list_order_means_are_numpy_means_of_the_lists():
    from isa_b200.scoring import list_order_means
    for n in (1, 7, 8, 9, 37, 130, 300):
        v = _values(n, n)
        sbd, dic, fg, unc = list_order_means(v)
        # what evaluate.py does: np.mean of a Python list, per metric, in list order
        assert sbd == np.mean([float(x) for x in v[:, 0]])
        assert dic == np.mean([np.int64(x) for x in v[:, 1]])
        assert fg == np.mean(list(v[:, 2]))
        assert unc == int(v[:, 3].sum()) and isinstance(unc, int)


def test_scored_epochs_and_the_sbd_rule():
    from isa_b200.scoring import BestSBD, is_scored_epoch
    assert [e for e in range(3) if is_scored_epoch(e, 3, 2)] == [1, 2]
    assert [e for e in range(6) if is_scored_epoch(e, 6, 2)] == [1, 3, 5]
    assert [e for e in range(4) if is_scored_epoch(e, 4, 1)] == [0, 1, 2, 3]
    assert [e for e in range(4) if is_scored_epoch(e, 4, 9)] == [3]
    best = BestSBD()
    assert [best.keep(s) for s in (0.2, 0.1, 0.2, 0.5, 0.49)] == [True, False, True, True, False]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


N_EPOCHS = 5


def _gather_worker(rank, world, port, out_dir, n_images):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    from isa_b200 import parallel, scoring
    parallel.init_from_env(backend="gloo")
    lo, hi = parallel.shard_range(n_images, rank, world)
    best = scoring.BestSBD()
    means, kept = [], []
    for epoch in range(N_EPOCHS):
        local = _values(n_images, 100 + epoch)[lo:hi]
        got = scoring.epoch_scores(local, n_images, torch.device("cpu"))
        means.append(got)
        kept.append(best.keep(got[0]))
    torch.save({"means": means, "kept": kept}, os.path.join(out_dir, "r%d.pt" % rank))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("n_images", [1, 7, 25])
def test_gathered_scores_give_every_rank_the_same_means_and_decisions(tmp_path, n_images):
    """Shards of unequal length (7 = 4 + 3; 1 = 1 + 0) are padded for one all_gather: both ranks get the single-process
    means bit for bit, and so keep the same checkpoints."""
    from isa_b200.scoring import BestSBD, list_order_means
    world = 2
    mp.spawn(_gather_worker, args=(world, _free_port(), str(tmp_path), n_images), nprocs=world, join=True)
    a = torch.load(os.path.join(str(tmp_path), "r0.pt"))
    b = torch.load(os.path.join(str(tmp_path), "r1.pt"))
    assert a == b
    best = BestSBD()
    want = [list_order_means(_values(n_images, 100 + e)) for e in range(N_EPOCHS)]
    assert a["means"] == want
    assert a["kept"] == [best.keep(m[0]) for m in want]
    assert any(a["kept"]) and not all(a["kept"])


def _write_set(d, with_fg):
    gt = os.path.join(d, "gt")
    os.makedirs(gt, exist_ok=True)
    names = []
    for j, (h, w) in enumerate([(40, 30), (24, 50)]):
        rs = np.random.RandomState(j)
        rgb = rs.randint(0, 256, (h, w, 3)).astype(np.uint8)
        lab = np.zeros((h, w), np.uint8)
        lab[2:10, 3:12] = 7           # PNG ids 7, 20, 3: compacted to 2, 3, 1 in the order of their values
        lab[12:20, 5:9] = 20
        lab[20:23, 20:28] = 3
        names.append(os.path.join(d, "leaf%d_rgb.png" % j))
        Image.fromarray(rgb).save(names[-1])
        Image.fromarray(lab).save(os.path.join(gt, "leaf%d_label.png" % j))
        if with_fg:
            fg = (lab > 0).astype(np.uint8)
            fg[0, :] = 1
            fg[1, :] = 2              # evaluate.py counts only the value 1 as foreground
            Image.fromarray(fg).save(os.path.join(gt, "leaf%d_fg.png" % j))
    return names, gt


@pytest.mark.parametrize("with_fg", [True, False])
def test_ground_truth_in_evaluate_convention(tmp_path, with_fg):
    from isa_b200.metrics import calc_sbd
    from isa_b200.prediction import Prediction
    from isa_b200.scoring import InstanceScorer
    names, gt = _write_set(str(tmp_path), with_fg)
    mean, std = [0.52, 0.39, 0.21], [0.21, 0.15, 0.11]
    sc = InstanceScorer(names, gt, 16, 20, mean, std, 32, device="cpu")
    assert len(sc) == 2 and sc.n_gt == [3, 3] and sc.sizes == [(40, 30), (24, 50)]
    pred = Prediction(16, 20, mean, std, False, None, 1)
    for j, p in enumerate(names):
        lab = np.array(Image.open(os.path.join(gt, "leaf%d_label.png" % j)))
        labels, fg = sc.truth[j].numpy()
        assert np.array_equal(labels == 0, lab == 0)
        assert calc_sbd(labels, lab) == 1.0 and len(np.unique(labels)) == 4
        assert np.array_equal(np.unique(labels[lab == 7]), [2])
        want_fg = lab != 0
        if with_fg:
            want_fg = want_fg.copy()
            want_fg[0, :] = True
            want_fg[1, :] = False
        assert np.array_equal(fg, want_fg.astype(np.uint8))
        x, h, w = pred.image_to_tensor(np.array(Image.open(p).convert('RGB')))
        assert torch.equal(sc.input(j)[0], x) and (h, w) == sc.sizes[j]


def test_shards_decode_only_their_images(tmp_path):
    from isa_b200.scoring import InstanceScorer
    names, gt = _write_set(str(tmp_path), True)
    names = names + names[:1]
    parts = [InstanceScorer(names, gt, 16, 20, [0.5] * 3, [0.2] * 3, 32, device="cpu", rank=r, world=2) for r in (0, 1)]
    assert [len(s) for s in parts] == [2, 1] and all(s.n_images == 3 for s in parts)
    assert parts[1].sizes == [(40, 30)]


def test_loading_refuses_a_foreground_file_of_another_size(tmp_path):
    from isa_b200.scoring import InstanceScorer
    names, gt = _write_set(str(tmp_path), True)
    Image.fromarray(np.ones((5, 5), np.uint8)).save(os.path.join(gt, "leaf1_fg.png"))
    with pytest.raises(ValueError, match="leaf1_fg.png: foreground size"):
        InstanceScorer(names, gt, 16, 20, [0.5] * 3, [0.2] * 3, 32, device="cpu")
    os.remove(os.path.join(gt, "leaf1_label.png"))
    with pytest.raises(FileNotFoundError, match="leaf1_label.png"):
        InstanceScorer(names, gt, 16, 20, [0.5] * 3, [0.2] * 3, 32, device="cpu")


def _fit_args(tmp_path):
    return ('Multi', 0.5, 1.5, 2, 1.0, 0.001, 10.0, 0.5, 25, False, 'Adadelta', True, 1, None, [], [],
            os.path.join(str(tmp_path), "models"))


@pytest.mark.parametrize("kwargs, message", [
    (dict(select_by='sbd'), "needs a scorer"),
    (dict(score_every=0), "score_every=0"),
    (dict(score_every=-2, scorer=object()), "score_every=-2"),
    (dict(select_by='loss'), "select_by='loss'"),
])
def test_fit_rejects_bad_scoring_arguments(tmp_path, kwargs, message):
    from isa_b200.model import Model
    m = Model.__new__(Model)          # the arguments are checked before anything touches the network or the device
    with pytest.raises(ValueError, match=message):
        m.fit(*_fit_args(tmp_path), **kwargs)
    assert not os.path.exists(os.path.join(str(tmp_path), "models"))


@pytest.mark.parametrize("args, message", [
    (["--score_every", "1"], "--score_every needs --train_list"),
    (["--score_every", "-1"], "--score_every must be >= 0"),
    (["--select_by", "sbd"], "--select_by sbd needs --score_every"),
    (["--select_by", "loss"], "invalid choice"),
])
def test_train_py_rejects_bad_scoring_arguments(tmp_path, args, message):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "code", "train.py"), "--output", str(tmp_path)] + args,
                       cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 2, r.stdout + r.stderr
    assert message in r.stderr
