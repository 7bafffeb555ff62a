"""GPU: validation scoring on the device (isa_b200.scoring) equals what pred_list.py + evaluate.py --empty_as_zero compute
on the host, image for image and in the epoch means; Model.fit logs, keeps and selects by it; train.py's scores agree
with the files pred_list.py and evaluate.py produce for the kept checkpoint."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch
from PIL import Image

from isa_b200 import augment as A
from isa_b200 import settings, synth
from isa_b200.metrics import calc_dic, calc_dice, calc_sbd
from isa_b200.prediction import Prediction
from isa_b200.scoring import COLUMNS, InstanceScorer, list_order_means

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MS = settings.CVPPPModelSettings()
MEAN, STD = MS.MEAN, MS.STD
SIZES = [(120, 110), (97, 143), (120, 110), (97, 143), (133, 125)]

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def data(tmp_path_factory):
    """Five annotated images of three sizes in the CVPPP layout, with _fg.png files that differ from label != 0 (a
    border row marked 1, a few labelled pixels marked 0), and the counts.txt evaluate.py reads."""
    out = str(tmp_path_factory.mktemp("scoring"))
    gt = os.path.join(out, "gt")
    os.makedirs(gt)
    names, counts = [], []
    for j, (h, w) in enumerate(SIZES):
        nm = "plant%03d" % j
        Image.fromarray(synth.leaf_image(j, h, w)).save(os.path.join(out, nm + "_rgb.png"))
        n_inst = 3 + j % 4
        lab = synth.label_map(np.random.RandomState(j), h, w, n_inst).astype(np.int64) + 1
        lab[lab == 256] = 0
        lab[lab > 0] += 10 * j                    # PNG ids need not start at 1
        Image.fromarray(lab.astype(np.uint8)).save(os.path.join(gt, nm + "_label.png"))
        fg = (lab > 0).astype(np.uint8)
        fg[0, :] = 1
        fg[h // 2, ::3] = 0
        Image.fromarray(fg).save(os.path.join(gt, nm + "_fg.png"))
        names.append(os.path.join(out, nm + "_rgb.png"))
        counts.append("%s,%d" % (nm, len(np.unique(lab)) - 1))
    lst = os.path.join(out, "all.lst")
    with open(lst, "w") as f:
        f.write("\n".join(names) + "\n")
    with open(os.path.join(out, "counts.txt"), "w") as f:
        f.write("\n".join(counts) + "\n")
    return dict(dir=out, gt=gt, lst=lst, names=names, counts=os.path.join(out, "counts.txt"))


def _model(cuda, count_head, seed=23):
    from isa_b200.model import Model
    torch.manual_seed(seed)
    return Model('CVPPP', 'ReSeg', 2, 32, use_instance_segmentation=True, n_embedding=24, device=cuda, count_head=count_head)


def _set_counts(m, scorer, counts):
    """Linear layer of the count head solved so that image j predicts counts[j] (min-norm solution)."""
    feats = []
    with torch.no_grad():
        for j in range(len(scorer)):
            x = scorer.input(j).contiguous(memory_format=torch.channels_last)
            feats.append(m.model(False, x)[2].evaluate().pooled[0].double().cpu())
    a = torch.cat([torch.stack(feats), torch.ones(len(feats), 1, dtype=torch.float64)], 1)
    s = torch.tensor(counts, dtype=torch.float64) / m.max_n_objects
    sol = torch.linalg.lstsq(a, torch.log(s / (1 - s)).reshape(-1, 1), driver="gelsd").solution.reshape(-1)
    lin = m.model.ins_cls_out.linear
    with torch.no_grad():
        lin.weight.copy_(sol[:-1].float().reshape(1, -1))
        lin.bias.copy_(sol[-1:].float())


def _host_scores(pred, data):
    """evaluate.py --empty_as_zero on the masks Prediction(strict=False).predict_array returns and the PNGs on disk:
    one row [SBD, |DiC|, FG dice, unclustered] per image."""
    rows = []
    for p in data["names"]:
        base = os.path.basename(p)[:-len("_rgb.png")]
        sem, ins, n = pred.predict_array(np.array(Image.open(p).convert('RGB')))
        lab = np.array(Image.open(os.path.join(data["gt"], base + "_label.png")))
        fg = np.array(Image.open(os.path.join(data["gt"], base + "_fg.png"))) == 1
        fg_pred = (sem * 255).astype(np.uint8) == 255          # the -fg_mask.png test
        sbd = 0.0 if ins.max() == 0 else calc_sbd(lab, ins)
        rows.append([sbd, calc_dic(len(np.unique(lab)) - 1, n), calc_dice(fg, fg_pred), float(n == 0)])
    return rows


def _check_equal(values, rows):
    assert values.shape == (len(rows), 4) and values.dtype == np.float64
    for got, want in zip(values.tolist(), rows):
        assert got == [float(v) for v in want], (got, want)
    sbd, dic, fg, unc = list_order_means(values)
    assert sbd == np.mean([r[0] for r in rows])
    assert dic == np.mean([r[1] for r in rows])
    assert fg == np.mean([r[2] for r in rows])
    assert unc == sum(int(r[3]) for r in rows)


def test_device_input_is_bit_identical_to_image_to_tensor(cuda, data, tmp_path):
    p = os.path.join(str(tmp_path), "big_rgb.png")
    Image.fromarray(synth.leaf_image(9, 530, 500)).save(p)
    lab = synth.label_map(np.random.RandomState(9), 530, 500, 5).astype(np.int64) + 1
    lab[lab == 256] = 0
    Image.fromarray(lab.astype(np.uint8)).save(os.path.join(data["gt"], "big_label.png"))
    names = data["names"] + [p]
    for (H, W), ms in (((256, 256), MS), ((64, 96), settings.CityscapesModelSettings())):
        sc = InstanceScorer(names, data["gt"], H, W, ms.MEAN, ms.STD, 32, cuda)
        pred = Prediction(H, W, ms.MEAN, ms.STD, False, None, 1)
        for j, q in enumerate(names):
            want, h, w = pred.image_to_tensor(np.array(Image.open(q).convert('RGB')))
            got = sc.input(j)
            assert got.shape == (1, 3, H, W) and got.dtype == torch.float32 and got.device == cuda
            assert torch.equal(got[0].cpu().contiguous().view(torch.int32), want.view(torch.int32)), q
            assert (h, w) == sc.sizes[j]


@pytest.mark.parametrize("count_head", [False, True])
def test_scores_equal_evaluate_on_the_host(cuda, data, count_head):
    m = _model(cuda, count_head)
    sc = InstanceScorer(data["lst"], data["gt"], 64, 64, MEAN, STD, 32, cuda)
    if count_head:
        _set_counts(m, sc, [3, 5, 7, 9, 4])
    values = sc.score(m)
    rows = _host_scores(Prediction(64, 64, MEAN, STD, False, m, 1, strict=False), data)
    _check_equal(values, rows)
    assert (values[:, 0] > 0).sum() >= 3, values            # the images are clustered: the SBDs are not a formality
    if count_head:
        n_gt = [3 + j % 4 for j in range(5)]
        assert [abs(g - k) for g, k in zip(n_gt, [3, 5, 7, 9, 4])] == values[:, 1].tolist()
    else:
        assert values[:, 1].tolist() == [abs(3 + j % 4 - 16) for j in range(5)]
    assert values.tolist() == sc.score(m).tolist()          # the same scores on a second pass


def _evaluate(data, pred_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "code", "evaluate.py"), "--pred_dir", pred_dir, "--dataset",
                        "CVPPP", "--names", data["lst"], "--counts", data["counts"], "--gt_dir", data["gt"],
                        "--empty_as_zero"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    means = {}
    for key in ("SBD", "|DIC|", "FG DICE"):
        means[key] = float(re.search(r"MEAN %s\s*:\s*(\S+)" % re.escape(key), r.stdout).group(1))
    return means, r.stdout


def test_unclustered_image_scores_like_empty_as_zero(cuda, data, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "code"))
    try:
        import _common
    finally:
        sys.path.pop(0)
    m = _model(cuda, False)
    sc = InstanceScorer(data["lst"], data["gt"], 64, 64, MEAN, STD, 32, cuda)
    # move the background bias so that image 0 keeps about ten foreground pixels, then ask for more clusters than that
    with torch.no_grad():
        sem = m.predict_device(sc.input(0))[0][0]
        d = (sem[1].log() - sem[0].log()).flatten().sort(descending=True).values
        m.model.sem_seg_output.bias[0] += float(d[9] + d[10]) / 2
        sem = m.predict_device(sc.input(0))[0][0]
    fg0 = int((sem[1] > sem[0]).sum())
    m.n_objects_prediction = fg0 + 1
    values = sc.score(m)
    assert values[0].tolist() == [0.0, 3.0, values[0, 2], 1.0]       # SBD 0, k = 0: |DiC| = n_gt, counted
    pred = Prediction(64, 64, MEAN, STD, False, m, 1, strict=False)
    _check_equal(values, _host_scores(pred, data))
    # the files pred_list.py would write for these masks, scored by evaluate.py --empty_as_zero
    pred_dir = os.path.join(str(tmp_path), "pred")
    for p in data["names"]:
        raw = np.array(Image.open(p).convert('RGB'))
        name = os.path.splitext(os.path.basename(p))[0]
        sem_seg, ins_seg, n = pred.predict_array(raw)
        _common.write_prediction(os.path.join(pred_dir, name), name, raw, sem_seg, ins_seg, n)
    means, out = _evaluate(data, pred_dir)
    sbd, dic, fg, unc = list_order_means(values)
    assert "no instance in plant000_rgb" in out
    assert (means["SBD"], means["|DIC|"], means["FG DICE"]) == (sbd, dic, fg)
    assert unc >= 1


def test_rank_shards_concatenate_to_the_whole_list(cuda, data):
    m = _model(cuda, True)
    whole = InstanceScorer(data["lst"], data["gt"], 64, 64, MEAN, STD, 32, cuda).score(m)
    parts = [InstanceScorer(data["lst"], data["gt"], 64, 64, MEAN, STD, 32, cuda, rank=r, world=2) for r in (0, 1)]
    assert [len(p) for p in parts] == [3, 2]
    got = np.concatenate([p.score(m) for p in parts])
    assert got.tolist() == whole.tolist()


def _fit(cuda, data, out, n_epochs, **kwargs):
    ts = settings.CVPPPTrainingSettings()
    store = A.load_store(data["lst"], data["gt"], 32, 64, 64, ts.MEAN, ts.STD, cuda)
    flags = A.flags_from_settings(ts)
    m = _model(cuda, False)
    hist = m.fit(ts.CRITERION, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM, ts.LEARNING_RATE, ts.WEIGHT_DECAY, ts.CLIP_GRAD_NORM,
                 ts.LR_DROP_FACTOR, ts.LR_DROP_PATIENCE, ts.OPTIMIZE_BG, ts.OPTIMIZER, ts.TRAIN_CNN, n_epochs, None,
                 A.AugmentLoader(store, 2, 64, 64, flags, ts.SEED, True),
                 A.AugmentLoader(store, 4, 64, 64, flags, ts.SEED, False), out, **kwargs)
    return m, hist


def _read_log(path):
    with open(path) as f:
        lines = f.read().splitlines()
    assert lines[0] == "Epoch," + ",".join(COLUMNS) == "Epoch,SBD,|DiC|,FgDice,Unclustered"
    return [tuple(float(v) for v in line.split(",")) for line in lines[1:]]


def test_fit_scores_every_second_epoch_and_the_last(cuda, data, tmp_path):
    out = os.path.join(str(tmp_path), "models")
    sc = InstanceScorer(data["lst"], data["gt"], 64, 64, MEAN, STD, 32, cuda)
    m, hist = _fit(cuda, data, out, 3, scorer=sc, score_every=2)
    assert [e for e, _, _ in hist] == [0, 1, 2]
    assert [s[0] for s in m.score_history] == [1, 2]
    rows = _read_log(os.path.join(out, "validation_scores.log"))
    assert rows == [tuple(float(v) for v in s) for s in m.score_history]
    for _, sbd, dic, fg, unc in rows:
        assert 0.0 <= sbd <= 1.0 and 0.0 <= fg <= 1.0 and dic >= 0 and unc in range(6)
    with open(os.path.join(out, "validation.log")) as f:
        assert f.read().splitlines()[0] == "Epoch,Cost"


def test_fit_selects_checkpoints_by_sbd(cuda, data, tmp_path):
    out = os.path.join(str(tmp_path), "models")
    sc = InstanceScorer(data["lst"], data["gt"], 64, 64, MEAN, STD, 32, cuda)
    m, _ = _fit(cuda, data, out, 4, scorer=sc, score_every=1, select_by='sbd')
    sbds = [s[1] for s in m.score_history]
    assert len(sbds) == 4
    kept = [e for e, s in enumerate(sbds) if s >= max(sbds[:e + 1])]
    ckpts = sorted(f for f in os.listdir(out) if f.endswith(".pth"))
    assert len(ckpts) == len(kept)
    for f in ckpts:
        g = re.match(r"model_(\d+)_sbd(.+)_(.+)\.pth$", f)
        assert g, f
        assert int(g.group(1)) in kept and float(g.group(2)) == sbds[int(g.group(1))]
    assert sorted(int(re.match(r"model_(\d+)_", f).group(1)) for f in ckpts) == kept


def test_fit_without_a_scorer_writes_what_it_wrote_before(cuda, data, tmp_path):
    out = os.path.join(str(tmp_path), "models")
    m, hist = _fit(cuda, data, out, 3)
    costs = [val for _, _, val in hist]
    kept = [e for e, c in enumerate(costs) if c <= min(costs[:e + 1])]
    files = set(os.listdir(out))
    assert {f for f in files if not f.endswith(".pth")} == {"training.log", "validation.log"}
    assert m.score_history == []
    ckpts = [re.match(r"model_(\d+)_(.+)_(.+)\.pth$", f).groups() for f in files if f.endswith(".pth")]
    assert sorted(int(e) for e, _, _ in ckpts) == kept
    assert all(float(c) == costs[int(e)] for e, c, _ in ckpts)


def _run(args):
    r = subprocess.run([sys.executable] + args, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


def test_train_scores_match_pred_list_and_evaluate(cuda, data, tmp_path):
    out = str(tmp_path)
    models = os.path.join(out, "models")
    txt = _run([os.path.join(ROOT, "code", "train.py"), "--nepochs", "2", "--batchsize", "2", "--train_list", data["lst"],
                "--val_list", data["lst"], "--gt_dir", data["gt"], "--score_every", "1", "--select_by", "sbd",
                "--output", models])
    assert "Validation SBD" in txt
    logged = {int(r[0]): r[1:] for r in _read_log(os.path.join(models, "CVPPP", "validation_scores.log"))}
    assert sorted(logged) == [0, 1]
    ckpts = [f for f in os.listdir(os.path.join(models, "CVPPP")) if f.endswith(".pth")]
    assert ckpts and all("_sbd" in f for f in ckpts)
    epoch = max(int(re.match(r"model_(\d+)_", f).group(1)) for f in ckpts)
    ckpt = [f for f in ckpts if f.startswith("model_%d_" % epoch)][0]
    _run([os.path.join(ROOT, "code", "pred_list.py"), "--lst", data["lst"], "--model", os.path.join(models, "CVPPP", ckpt),
          "--output", os.path.join(out, "pred")])
    means, _ = _evaluate(data, os.path.join(out, "pred"))
    sbd, dic, fg, _unc = logged[epoch]
    print("\nround trip, epoch %d: logged SBD %r |DiC| %r FG dice %r; evaluate.py %r; differences SBD %.3g FG dice %.3g"
          % (epoch, sbd, dic, fg, means, abs(means["SBD"] - sbd), abs(means["FG DICE"] - fg)))
    assert means["|DIC|"] == dic
    assert abs(means["SBD"] - sbd) <= 1e-3
    assert abs(means["FG DICE"] - fg) <= 1e-3
