"""Validation scoring while training: the SBD, |DiC| and foreground dice that `pred_list.py` + `evaluate.py
--empty_as_zero` report, computed on the device for a list of annotated images.

    scorer = InstanceScorer('val.lst', gt_dir, ms.IMAGE_HEIGHT, ms.IMAGE_WIDTH, ms.MEAN, ms.STD, ms.MAX_N_OBJECTS, device)
    values = scorer.score(model)            # (n_local, 4) float64: SBD, |DiC|, FgDice, unclustered, this rank's shard
    sbd, dic, fg_dice, unclustered = epoch_scores(values, scorer.n_images, device)     # every rank: the same numbers

Each image goes through the device path of `Prediction.predict_array`: the network at batch 1 (pred_list.py runs at
batch 1, and cuDNN may pick other algorithms at another batch size), k from the count head or
`model.n_objects_prediction`, then `Prediction.cluster_device` up to the image's own size.  The scores are computed
from the device masks by `metrics.sbd_device`, so nothing per-pixel visits the host:

* SBD: `sbd_device(label, ins_up)`; 0 when the image could not be clustered or its upsampled mask holds no instance
  (evaluate.py --empty_as_zero).
* |DiC| = |n_gt - k|, with k = 0 for an image that could not be clustered (pred_list.py writes 0 to -n_objects.npy).
* FG dice: `calc_dice(fg_gt, fg_mask == 255)`.  pred_list.py writes `cls_up * 255` as uint8, which is 255 exactly where
  cls_up == 1, and the dice of two binary images is BD(gt, pred) of their contingency table, which `sbd_device`
  evaluates as the same float64 ratio 2|gt and pred| / (|gt| + |pred|).

Inputs are read once, at construction: the image resized to the network size with PIL bilinear exactly as
`Prediction.image_to_tensor` does, kept as uint8; the labels at their original size (0 = background, instances 1..n
in the order of their PNG values); the foreground truth `<base>_fg.png == 1`, or `label != 0` without that file.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch
import torch.distributed as dist
from PIL import Image

from . import augment, metrics, parallel
from .prediction import Prediction

COLUMNS = ("SBD", "|DiC|", "FgDice", "Unclustered")


def fg_path(image_path, gt_dir):
    return augment.label_path(image_path, gt_dir)[:-len('_label.png')] + '_fg.png'


def list_order_means(values):
    """(n, 4) per-image values in list order -> (mean SBD, mean |DiC|, mean FG dice, number unclustered).  Each mean is
    np.mean of one contiguous column, the float64 pairwise sum evaluate.py takes over its lists (np.mean(values,
    axis=0) sums the rows one after the other and can differ in the last bit)."""
    values = np.asarray(values, dtype=np.float64)
    means = [float(np.mean(np.ascontiguousarray(values[:, j]))) for j in range(3)]
    return means[0], means[1], means[2], int(values[:, 3].sum())


def gather_shards(local, n_images, device):
    """This rank's (n_local, 4) values of its shard_range -> the (n_images, 4) values of every image in list order, on
    every rank.  The shards differ in length by at most one, so each is padded to the longest for one all_gather
    (NCCL tensors live on the GPU, gloo ones on the CPU: `device`)."""
    local = np.asarray(local, dtype=np.float64).reshape(-1, 4)
    if not parallel.is_distributed():
        return local
    world, rank = dist.get_world_size(), dist.get_rank()
    spans = [parallel.shard_range(n_images, r, world) for r in range(world)]
    lo, hi = spans[rank]
    if local.shape[0] != hi - lo:
        raise ValueError("rank %d holds %d values for its %d images" % (rank, local.shape[0], hi - lo))
    longest = max(h - l for l, h in spans)
    padded = torch.zeros(longest, 4, dtype=torch.float64, device=device)
    padded[:hi - lo] = torch.from_numpy(local).to(device)
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded)
    return np.concatenate([p.cpu().numpy()[:h - l] for p, (l, h) in zip(parts, spans)])


def epoch_scores(local, n_images, device):
    """This rank's score() values -> (mean SBD, mean |DiC|, mean FG dice, number unclustered) over the whole list, the
    same numbers on every rank, so every rank takes the same checkpoint decision."""
    if parallel.is_distributed() and dist.get_backend() != 'nccl':
        device = torch.device('cpu')
    return list_order_means(gather_shards(local, n_images, device))


def is_scored_epoch(epoch, n_epochs, score_every):
    """Model.fit scores every score_every-th epoch (0-based epoch + 1 divisible by it) and always the last one."""
    return (epoch + 1) % score_every == 0 or epoch == n_epochs - 1


class BestSBD(object):
    """select_by='sbd': a scored epoch is kept when its mean SBD is >= the best so far."""

    def __init__(self):
        self.best = -np.inf

    def keep(self, sbd):
        if sbd >= self.best:
            self.best = sbd
            return True
        return False


class InstanceScorer(object):
    """SBD, |DiC|, FG dice and the unclustered count of a validation list, scored on the device (see the module doc).
    rank / world: this process scores its `parallel.shard_range` of the list, and decodes only that."""

    def __init__(self, list_path, gt_dir, height, width, mean, std, max_n_objects, device=None, seed=0, n_init=35,
                 max_iter=500, rank=0, world=1):
        self.height, self.width = int(height), int(width)
        self.mean, self.std = list(mean), list(std)
        self.seed, self.n_init, self.max_iter = int(seed), int(n_init), int(max_iter)
        self.names = augment.read_list(list_path) if isinstance(list_path, str) else list(list_path)
        if not self.names:
            raise ValueError("empty validation list")
        self.n_images = len(self.names)
        self.rank, self.world = int(rank), int(world)
        self.lo, self.hi = parallel.shard_range(self.n_images, self.rank, self.world)
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        with ThreadPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:     # PIL decodes and resizes with the GIL released
            loaded = list(ex.map(lambda p: self._load(p, gt_dir, max_n_objects), self.names[self.lo:self.hi]))
        dev = self.device
        rgb = np.stack([l[0] for l in loaded]) if loaded else np.zeros((0, self.height, self.width, 3), np.uint8)
        self.rgb = torch.from_numpy(rgb).to(dev)                                    # (n_local, H, W, 3) u8
        self.truth = [torch.from_numpy(l[1]).to(dev) for l in loaded]               # (2, h, w) u8: labels, fg
        self.n_gt = [l[2] for l in loaded]
        self.sizes = [tuple(l[1].shape[1:]) for l in loaded]
        # float32 device tensors, not Python scalars: torch divides by a CPU scalar as a multiplication by its
        # reciprocal, which is not the correctly rounded quotient image_to_tensor computes in numpy
        self._255 = torch.full((3, 1, 1), 255.0, dtype=torch.float32, device=dev)
        self._mean = torch.tensor(self.mean, dtype=torch.float32, device=dev).reshape(3, 1, 1)
        self._std = torch.tensor(self.std, dtype=torch.float32, device=dev).reshape(3, 1, 1)

    def _load(self, image_path, gt_dir, max_n_objects):
        rgb, lab = augment.read_pair(image_path, gt_dir, max_n_objects)
        small = np.asarray(Image.fromarray(rgb).resize((self.width, self.height), Image.BILINEAR))
        lab = lab + np.uint8(1)              # ids 0..n-1 -> 1..n, background 255 -> 0 (evaluate.py's convention)
        n_gt = int(lab.max())
        fp = fg_path(image_path, gt_dir)
        if os.path.isfile(fp):
            with Image.open(fp) as im:
                fg = np.array(im)
            if fg.shape != lab.shape:
                raise ValueError("%s: foreground size %dx%d differs from the label's %dx%d"
                                 % (fp, fg.shape[1] if fg.ndim > 1 else 0, fg.shape[0], lab.shape[1], lab.shape[0]))
            fg = fg == 1
        else:
            fg = lab != 0
        return small, np.stack([lab, fg.astype(np.uint8)]), n_gt

    def __len__(self):
        return self.hi - self.lo

    def input(self, j):
        """The network input of this shard's image j, (1, 3, H, W) float32 on the device: x / 255, then (x - mean) / std,
        one correctly rounded float32 operation each, as in Prediction.image_to_tensor."""
        x = self.rgb[j:j + 1].permute(0, 3, 1, 2).float()
        return (x / self._255 - self._mean) / self._std

    @torch.no_grad()
    def score(self, model):
        """Per-image float64 (n_local, 4) [SBD, |DiC|, FgDice, unclustered] of this rank's shard, in list order.  Without
        the count head nothing synchronises until the final copy; with it, each image's 4-byte count is read back before
        its clustering is enqueued, as in Prediction.predict_array."""
        pred = Prediction(self.height, self.width, self.mean, self.std, False, model, 1, seed=self.seed,
                          n_init=self.n_init, max_iter=self.max_iter, strict=False)
        out = torch.empty(len(self), 4, dtype=torch.float64, device=self.device)
        for j in range(len(self)):
            h, w = self.sizes[j]
            sem, emb, n_pred = model.predict_device_with_counts(self.input(j))
            n = model.n_objects_prediction if n_pred is None else int(n_pred[0])
            _, _, ins_up, cls_up, res = pred.cluster_device(sem[0], emb[0], n, h, w)
            s = metrics.sbd_device(self.truth[j], torch.stack([ins_up, (cls_up == 1).to(torch.uint8)]))
            ok = res.info[0] == 0
            sbd = torch.where(ok, torch.nan_to_num(s[0, 0], nan=0.0), 0.0)
            dic = (self.n_gt[j] - ok.double() * n).abs()
            # dice of the foreground images; BD is NaN when one of them is empty: calc_dice gives 0 unless both are
            fg = s[1, 1]
            fg = torch.where(torch.isnan(fg) & (s[1, 3] + s[1, 4] > 0), 0.0, fg)
            out[j] = torch.stack([sbd, dic, fg, (~ok).double()])
        return out.cpu().numpy()
