"""train.py -- training entry point with the reference's flags (/root/reference/code/train.py:18-37).
The reference reads LMDB databases (lmdb is not installed).  `--train_list L --val_list V --gt_dir D` trains on a
directory of annotated images instead (the CVPPP layout pred_list.py and evaluate.py read: `<base>_rgb.png` listed in
L and V, `<base>_label.png` under D), decoded once into device memory and augmented on the device with the flags and
seed of the settings class (isa_b200.augment).  `--score_every N` also scores the V images every N epochs by the SBD,
|DiC| and foreground dice that pred_list.py + evaluate.py --empty_as_zero report (validation_scores.log, on the device:
isa_b200.scoring), and `--select_by sbd` keeps the checkpoints of the best mean SBD instead of the best validation
cost.  Without `--train_list`, `--synthetic N` trains on N seeded CVPPP-shaped synthetic batches, which is also what
bench.py measures.  Launch one process per GPU with torchrun for single-node data parallelism:

    python code/train.py --output out_dir --train_list train.lst --val_list val.lst --gt_dir A1 --batchsize 16
    python code/train.py --output out_dir --synthetic 8 --nepochs 2 --batchsize 16
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 code/train.py ...
"""
import argparse
import os
import random

import numpy as np
import torch

import _common  # noqa: F401
from isa_b200 import parallel, settings, synth
from isa_b200.model import Model

parser = argparse.ArgumentParser()
parser.add_argument('--model', default='', help='Filepath of trained model (to continue training) [Default: ""]')
parser.add_argument('--usegpu', action='store_true', default=True)
parser.add_argument('--nepochs', type=int, default=600, help='Number of epochs to train for [Default: 600]')
parser.add_argument('--batchsize', type=int, default=2, help='Batch size per process [Default: 2]')
parser.add_argument('--debug', action='store_true')
parser.add_argument('--nworkers', type=int, default=2)
parser.add_argument('--dataset', type=str, default='CVPPP')
parser.add_argument('--output', default='models', help='Directory for checkpoints and logs')
parser.add_argument('--synthetic', type=int, default=8, help='Number of synthetic minibatches per epoch (without --train_list)')
parser.add_argument('--train_list', default='', help='Text file of training image paths (<base>_rgb.png); trains on them instead of synthetic batches')
parser.add_argument('--val_list', default='', help='Text file of validation image paths (with --train_list)')
parser.add_argument('--gt_dir', default='', help='Directory with <base>_label.png for every listed image (with --train_list)')
parser.add_argument('--target_format', default='compact', choices=['compact', 'reference'],
                    help='compact: uint8 class / label maps (15 MB per 16-image batch); reference: the int64 one-hot tensors of '
                         'lib/dataset.py:354-376 (298 MB), distilled on the device')
parser.add_argument('--count_head', action='store_true', help='Train the instance-count head as well (count loss added to the cost)')
parser.add_argument('--cuda_graph', action='store_true', help='Replay forward+backward of the training step from a CUDA graph (fixed batch shape)')
parser.add_argument('--score_every', type=int, default=0, help='Score the --val_list images by SBD, |DiC| and FG dice every N epochs '
                    'and after the last one, as pred_list.py + evaluate.py --empty_as_zero would (0 = off) [Default: 0]')
parser.add_argument('--select_by', default='cost', choices=['cost', 'sbd'], help='Keep the checkpoints of the best validation '
                    'cost, or of the best mean SBD of the scored epochs (needs --score_every) [Default: cost]')


class SyntheticLoader(object):
    """Yields (images, sem, ins, n_objects): `reference` = int64 one-hot tensors like AlignCollate
    (lib/dataset.py:354-379), `compact` = uint8 class map / label map (isa_b200.data.compact_collate)."""

    def __init__(self, n_batches, batch, ts, seed, target_format='compact'):
        self.items = []
        for j in range(n_batches):
            d = synth.batch(seed + j, batch, 3, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, ts.MAX_N_OBJECTS)
            lab = d["labels"]
            if target_format == 'compact':
                sem, ins = (lab != 255).astype(np.uint8), lab
            else:
                sem = np.stack([(lab == 255), (lab != 255)], 1).astype(np.int64)
                ins = synth.onehot(lab, ts.MAX_N_OBJECTS, np.int64)
            self.items.append((torch.from_numpy(d["emb"]).pin_memory(), torch.from_numpy(sem).pin_memory(),
                               torch.from_numpy(ins).pin_memory(), torch.from_numpy(d["n_objects"])))

    def __iter__(self):
        return iter(self.items)

    def __len__(self):
        return len(self.items)


if __name__ == '__main__':
    opt = parser.parse_args()
    assert opt.dataset in ['CVPPP', 'Cityscapes']
    if opt.score_every < 0:
        parser.error('--score_every must be >= 0')
    if opt.score_every and not opt.train_list:
        parser.error('--score_every needs --train_list, --val_list and --gt_dir: the synthetic batches have no label files')
    if opt.select_by == 'sbd' and not opt.score_every:
        parser.error('--select_by sbd needs --score_every')
    ts = settings.CVPPPTrainingSettings() if opt.dataset == 'CVPPP' else settings.CityscapesTrainingSettings()
    rank, world, local_rank = parallel.init_from_env()
    torch.cuda.set_device(local_rank)
    random.seed(ts.SEED); np.random.seed(ts.SEED); torch.manual_seed(ts.SEED)
    model = Model(opt.dataset, ts.MODEL_NAME, ts.N_CLASSES, ts.MAX_N_OBJECTS,
                  use_instance_segmentation=ts.USE_INSTANCE_SEGMENTATION, use_coords=ts.USE_COORDINATES,
                  load_model_path=opt.model, usegpu=True, n_embedding=ts.D_MODEL, distributed=world > 1,
                  n_objects_prediction=ts.N_OBJECTS_PREDICTION,
                  device=torch.device('cuda', local_rank), count_head=opt.count_head or ts.COUNT_HEAD)
    if opt.cuda_graph:
        model.enable_cuda_graph()
    scorer = None
    if opt.train_list:
        if not (opt.val_list and opt.gt_dir):
            parser.error('--train_list needs --val_list and --gt_dir')
        from isa_b200 import augment
        flags = augment.flags_from_settings(ts)
        dev = torch.device('cuda', local_rank)
        stores = [augment.load_store(p, opt.gt_dir, ts.MAX_N_OBJECTS, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, ts.MEAN, ts.STD, dev)
                  for p in (opt.train_list, opt.val_list)]
        train_loader, test_loader = [augment.AugmentLoader(st, opt.batchsize * world, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, flags,
                                                           ts.SEED, train, rank, world)
                                     for st, train in zip(stores, (True, False))]
        if opt.score_every:
            from isa_b200.scoring import InstanceScorer
            # the k-means settings of pred_list.py (seed 0, 35 restarts, 500 iterations): the logged scores are the
            # ones pred_list.py + evaluate.py --empty_as_zero give for the same checkpoint
            scorer = InstanceScorer(opt.val_list, opt.gt_dir, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, ts.MEAN, ts.STD,
                                    ts.MAX_N_OBJECTS, dev, seed=0, n_init=35, max_iter=500, rank=rank, world=world)
    else:
        train_loader = SyntheticLoader(opt.synthetic, opt.batchsize, ts, 1000 * rank, opt.target_format)
        test_loader = SyntheticLoader(max(1, opt.synthetic // 4), opt.batchsize, ts, 500000 + 1000 * rank, opt.target_format)
    model.fit(ts.CRITERION, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM, ts.LEARNING_RATE, ts.WEIGHT_DECAY, ts.CLIP_GRAD_NORM,
              ts.LR_DROP_FACTOR, ts.LR_DROP_PATIENCE, ts.OPTIMIZE_BG, ts.OPTIMIZER, ts.TRAIN_CNN, opt.nepochs,
              ts.CLASS_WEIGHTS, train_loader, test_loader, os.path.join(opt.output, opt.dataset), opt.debug,
              scorer=scorer, score_every=max(opt.score_every, 1), select_by=opt.select_by)
