"""`Model`: orchestration with the reference's API (/root/reference/code/lib/model.py:21-499):

    Model(dataset, model_name, n_classes, max_n_objects, wae_opt=None, use_instance_segmentation=False,
          use_wae=True, use_coords=False, load_model_path='', load_decoder_model_path='', usegpu=True)
    .fit(criterion_type, delta_var, delta_dist, norm, learning_rate, weight_decay, clip_grad_norm,
         lr_drop_factor, lr_drop_patience, optimize_bg, optimizer, train_cnn, n_epochs, class_weights,
         train_loader, test_loader, model_save_path, debug, scorer=None, score_every=1, select_by='cost')
    .predict(images) -> (sem_probs (b,n_classes,h,w), embeddings (b,C,h,w), n_objects IntTensor (b,1))
    (n_objects: the trained count head's prediction with count_head=True, else the constant n_objects_prediction)

The reference file cannot be parsed by Python >= 3.7 (`cuda(async=True)`, model.py:221-225,476) and its
training step takes `ins_cost` from a NaN-producing decoder (SURVEY.md R3/R5); this is a rewrite with
the same surface where the step is the designed one (SURVEY.md section 3.1):
    sem_logits, emb = net(True, images); ins_cost, means = criterion_discriminative(emb, ins, n, K)
    cost = ins_cost + CE + Dice; backward; clip_grad_norm_; optimizer.step()
Extras: `train_step(...)` (the public face of the reference's private __minibatch), device-resident
`predict_device(...)` / `predict_device_with_counts(...)`, the optional instance-count head (`count_head=True`), and
single-node data parallelism (`distributed=True`): one process per GPU, parameters replicated, ONE flat-bucket NCCL
all-reduce of the gradients per step.
visdom plotting and the pickle dumps to a hard-coded path (model.py:55,454-457) are dropped.
"""
import os
import time

import numpy as np
import torch
import torch.distributed as dist
import torch.optim as optim
from torch.optim.lr_scheduler import ReduceLROnPlateau

from . import _lib, parallel, scoring
from .archs import ReSeg
from .losses import DiscriminativeLoss, label_fg_count, onehot_to_labels
from .seg_losses import DiceLoss, SegLosses, class_map


class Model(object):

    def __init__(self, dataset, model_name, n_classes, max_n_objects, wae_opt=None,
                 use_instance_segmentation=False, use_wae=False, use_coords=False,
                 load_model_path='', load_decoder_model_path='', usegpu=True,
                 n_input=3, n_embedding=24, n_objects_prediction=16, distributed=False, device=None, net_kwargs=None,
                 count_head=False):
        self.dataset = dataset
        self.model_name = model_name
        self.n_classes = n_classes
        self.max_n_objects = max_n_objects
        self.use_instance_segmentation = use_instance_segmentation
        self.use_coords = use_coords
        self.load_model_path = load_model_path
        self.load_decoder_model_path = load_decoder_model_path
        self.use_wae = use_wae
        self.usegpu = usegpu
        self.n_objects_prediction = int(n_objects_prediction)
        self.count_head = bool(count_head)
        assert self.dataset in ['CVPPP', 'Cityscapes']
        assert self.model_name in ['ReSeg']
        if not usegpu:
            raise _lib.IsaError("Model(usegpu=False): the hot path is sm_100a-only, there is no CPU fallback")
        _lib.load()
        self.device = torch.device(device) if device is not None else torch.device('cuda', torch.cuda.current_device())
        self.model = ReSeg(self.n_classes, self.use_instance_segmentation, pretrained=False,
                           use_coordinates=self.use_coords, use_wae=use_wae, usegpu=True,
                           n_input=n_input, n_embedding=n_embedding, count_head=self.count_head,
                           max_n_objects=self.max_n_objects, **(net_kwargs or {}))
        self.__load_weights()
        torch.backends.cudnn.benchmark = True          # model.py:50-52
        self.model.to(self.device).to(memory_format=torch.channels_last)
        self.distributed = bool(distributed) and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        if self.distributed:
            self.__broadcast_parameters()
        self._flat_grad = None
        self.optimizer = None
        self.lr_scheduler = None
        # CUDA-graph replay of the training step (static shapes): see enable_cuda_graph()
        self._graph_warmup = 0
        self._graphs = {}
        self._graph_seen = {}

    # ------------------------------------------------------------------ weights
    def __load_weights(self):
        """Partial-load semantics of model.py:62-79: state_dict.update(pretrained)."""
        if self.load_model_path != '':
            assert os.path.isfile(self.load_model_path), 'Model : {} does not exists!'.format(self.load_model_path)
            print('Loading model from {}'.format(self.load_model_path))
            model_state_dict = self.model.state_dict()
            pretrained_state_dict = torch.load(self.load_model_path, map_location='cpu')
            model_state_dict.update(pretrained_state_dict)
            self.model.load_state_dict(model_state_dict)

    def __broadcast_parameters(self):
        for t in list(self.model.parameters()) + list(self.model.buffers()):
            dist.broadcast(t.data, src=0)

    # ------------------------------------------------------------------ criterion / optimizer
    def define_criterion(self, class_weights, delta_var, delta_dist, norm=2, optimize_bg=False, criterion='CE'):
        """model.py:99-139"""
        assert criterion in ['CE', 'Dice', 'Multi', None]
        smooth = 1.0
        if self.use_instance_segmentation:
            self.criterion_discriminative = DiscriminativeLoss(delta_var, delta_dist, norm, usegpu=True)
        w = None
        if class_weights is not None:
            w = torch.as_tensor(class_weights, dtype=torch.float32, device=self.device)
        if criterion in ['CE', 'Multi']:
            self.criterion_ce = torch.nn.CrossEntropyLoss(w)
        if criterion in ['Dice', 'Multi']:
            self.criterion_dice = DiceLoss(optimize_bg=optimize_bg, weight=w, smooth=smooth)
        # what the step runs: cross entropy + Dice of the semantic head in one fused pass (csrc/seg_losses.cu)
        self.criterion_seg = SegLosses(w, optimize_bg=optimize_bg, smooth=smooth)
        self.criterion_type = criterion

    def define_optimizer(self, learning_rate, weight_decay, lr_drop_factor, lr_drop_patience, optimizer='Adam'):
        """model.py:141-160"""
        assert optimizer in ['RMSprop', 'Adam', 'Adadelta', 'SGD']
        parameters = [p for p in self.model.parameters() if p.requires_grad]
        if optimizer == 'RMSprop':
            self.optimizer = optim.RMSprop(parameters, lr=learning_rate, weight_decay=weight_decay)
        elif optimizer == 'Adadelta':
            # the shipped optimizer (training_settings.py): clip + update fused over flat buffers (optim.py)
            from .optim import FusedAdadelta
            self.optimizer = FusedAdadelta(parameters, lr=learning_rate, weight_decay=weight_decay)
            self._flat_grad = None
        elif optimizer == 'Adam':
            self.optimizer = optim.Adam(parameters, lr=learning_rate, weight_decay=weight_decay)
        else:
            self.optimizer = optim.SGD(parameters, lr=learning_rate, momentum=0.9, weight_decay=weight_decay)
        self.lr_scheduler = ReduceLROnPlateau(self.optimizer, mode='min', factor=lr_drop_factor, patience=lr_drop_patience)

    # ------------------------------------------------------------------ data-parallel gradient exchange
    def __allreduce_gradients(self):
        """One flat fp32 bucket, one NCCL all-reduce (sum) over NVLink, then / world_size."""
        flat = getattr(self.optimizer, 'flat_grad', None)
        if flat is not None:            # the fused optimizer's gradient buffer IS the bucket
            if parallel.is_distributed():
                dist.all_reduce(flat, op=dist.ReduceOp.SUM)
                flat.div_(dist.get_world_size())
            return
        if self._flat_grad is None:
            self._flat_grad = parallel.FlatGradBucket(self.model.parameters())
        self._flat_grad.allreduce(average=True)

    def __compact_targets(self, sem, ins):
        """Reference-format targets -> what the kernels read, ONE pass over the dense masks:
        sem one-hot (b,n_classes,h,w) -> uint8 class map (b,h,w);  ins one-hot int64/uint8 (b,K,h,w) -> uint8 label map
        (b,h,w), 255 = background (float masks may be soft: they stay dense);  uint8 maps pass through.  Also returns the
        data-parallel q-regulariser denominator (global foreground count / world size; None on a single process) -- the
        count comes out of the same distillation pass, nothing re-reads the masks."""
        dev = self.device
        sem_map = class_map(sem.to(dev, non_blocking=True))
        ins = ins.to(dev, non_blocking=True)
        count = None
        if ins.dim() == 4 and ins.dtype in (torch.int64, torch.uint8, torch.bool):
            ins, _flag, count = onehot_to_labels(ins, with_count=True)
        if not self.distributed:
            return sem_map, ins, None
        if count is None:
            count = label_fg_count(ins, self.max_n_objects) if ins.dim() == 3 else ins.sum()
        return sem_map, ins, parallel.global_q_denominator(count)

    # ------------------------------------------------------------------ CUDA-graph replay of the step
    def enable_cuda_graph(self, warmup_steps=3):
        """Capture the training step's forward, losses and backward (~800 launches at batch 16; the gradient all-reduce
        and the two launches of the fused clip + Adadelta update stay eager) in ONE CUDA graph per input signature after `warmup_steps` eager steps (cuDNN's algorithm
        search runs in those), then replay it: the step is launch-bound on the host otherwise (kernels 12.0 ms of a
        13.3 ms step).  Needs device-resident inputs of a fixed shape and the fused optimizer; anything else silently
        takes the eager path.  Metrics come back as the graph's static device scalars."""
        self._graph_warmup = max(int(warmup_steps), 1)

    def __graph_step(self, images, sem, ins, nobj, q_den, clip_grad_norm, criterion_type):
        """sem / ins are the COMPACT targets (uint8 maps, or dense float masks)."""
        key = (tuple(images.shape), tuple(sem.shape), sem.dtype, tuple(ins.shape), ins.dtype, tuple(nobj.shape), nobj.dtype,
               float(clip_grad_norm), criterion_type)
        g = self._graphs.get(key)
        if g is None:
            seen = self._graph_seen.get(key, 0)
            self._graph_seen[key] = seen + 1
            if seen < self._graph_warmup:
                return None                          # eager warm-up (also cuDNN autotuning)
            static = [t.clone() for t in (images, sem, ins, nobj)]
            # The graph holds forward + losses + backward.  The tail stays eager: (i) NCCL collectives captured in a
            # graph leave the process group's watchdog with events it can never complete (the process hangs at exit),
            # so the q-regulariser's global denominator is a static input and the gradient all-reduce runs after the
            # replay; (ii) the optimizer's learning rate is a kernel ARGUMENT that ReduceLROnPlateau changes between
            # epochs, so the two launches of the fused clip + Adadelta update are issued eagerly too.
            static_q = torch.zeros(1, device=self.device, dtype=torch.float32) if self.distributed else None
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            timer_was = _lib.TIMER.enabled
            _lib.TIMER.enabled = False               # event-timed C-ABI calls cannot be captured
            try:
                with torch.cuda.graph(graph):
                    out = self.__fwd_bwd(static[0], static[1], static[2], static[3], criterion_type, True, static_q)
            finally:
                _lib.TIMER.enabled = timer_was
            g = self._graphs[key] = (graph, static, static_q, out)
        graph, static, static_q, out = g
        for dst, src in zip(static, (images, sem, ins, nobj)):
            dst.copy_(src, non_blocking=True)
        if static_q is not None:
            static_q.copy_(q_den, non_blocking=True)
        graph.replay()
        self.__update(clip_grad_norm)
        return out

    # ------------------------------------------------------------------ one step (model.py:162-281)
    def train_step(self, images, sem_seg_annotations, ins_seg_annotations, n_objects, clip_grad_norm=10.0,
                   criterion_type=None, mode='training'):
        """images (b,c,h,w) float; sem one-hot (b,n_classes,h,w) or a (b,h,w) uint8 class map; ins one-hot (b,K,h,w)
        (float/int64/uint8) or a (b,h,w) uint8 label map (255 = background); n_objects (b,).  CPU tensors are copied with
        non_blocking=True as the reference does (.cuda(async=True)).  Returns the metrics dict of model.py:242-269
        (device scalars)."""
        criterion_type = criterion_type or self.criterion_type
        training = mode == 'training'
        dev = self.device
        images = images.to(dev, non_blocking=True)
        sem, ins, q_den = self.__compact_targets(sem_seg_annotations, ins_seg_annotations)
        nobj = torch.as_tensor(n_objects).to(dev, non_blocking=True).reshape(-1)
        if training and self._graph_warmup > 0 and hasattr(self.optimizer, 'flat_grad') and not _lib.TIMER.enabled:
            out = self.__graph_step(images, sem, ins, nobj, q_den, clip_grad_norm, criterion_type)
            if out is not None:
                return out
        out_metrics = self.__fwd_bwd(images, sem, ins, nobj, criterion_type, training, q_den)
        if training:
            self.__update(clip_grad_norm)
        return out_metrics

    def __fwd_bwd(self, images, sem_map, ins, nobj, criterion_type, training, q_den):
        """Forward, losses and (training) zero_grad + backward on COMPACT device targets; returns the metrics dict of
        model.py:242-269.  With the count head, cost += 'Count Cost' = mean_b (s_b - n_objects_b / K)^2 (weight 1) and
        'Count |DiC|' = mean_b |n_pred_b - n_objects_b| is reported; both stay device scalars (nothing synchronises, the
        step still captures in a CUDA graph).  Data parallel: the shards are equal-sized and the gradients are averaged,
        so the per-rank batch mean of the count loss gives the global-batch gradient with no collective of its own."""
        self.model.train(training)
        images = images.contiguous(memory_format=torch.channels_last)
        out_metrics = dict()
        with torch.set_grad_enabled(training):
            outputs = self.model(training, images)
            sem_seg_predictions, ins_seg_predictions = outputs[0], outputs[1]
            cost = 0
            if self.use_instance_segmentation:
                ins_cost, _means = self.criterion_discriminative(ins_seg_predictions, ins, nobj, self.max_n_objects,
                                                                 q_denominator=q_den)
                cost = cost + ins_cost
                out_metrics['INS Cost'] = ins_cost.detach()
            if criterion_type in ['CE', 'Dice', 'Multi']:
                ce_cost, dice_cost = self.criterion_seg(sem_seg_predictions, sem_map, time=1)   # model.py:255-269
                if criterion_type in ['CE', 'Multi']:
                    cost = cost + ce_cost
                    out_metrics['CE Cost'] = ce_cost.detach()
                if criterion_type in ['Dice', 'Multi']:
                    cost = cost + dice_cost
                    out_metrics['Dice Cost'] = dice_cost.detach()
            if self.count_head:
                count = outputs[2].evaluate(nobj)
                cost = cost + count.loss
                out_metrics['Count Cost'] = count.loss.detach()
                out_metrics['Count |DiC|'] = (count.n_pred - nobj).abs().float().mean()
            out_metrics['Cost'] = cost.detach()
        if training:
            if hasattr(self.optimizer, 'flat_grad'):
                self.optimizer.zero_grad()
            elif self._flat_grad is not None:
                self._flat_grad.zero()
            else:
                self.model.zero_grad()
            cost.backward()
        return out_metrics

    def loss_and_gradients(self, images, sem_seg_annotations, ins_seg_annotations, n_objects, criterion_type=None):
        """One forward + backward WITHOUT the optimizer update: returns (metrics, flat fp32 gradient) -- data parallel: the
        gradient after the all-reduce, i.e. what the update would consume.  Used to check that the data-parallel step
        equals the single-process step on the concatenated batch (bench.py `dp_parity`, tests)."""
        dev = self.device
        sem, ins, q_den = self.__compact_targets(sem_seg_annotations, ins_seg_annotations)
        nobj = torch.as_tensor(n_objects).to(dev, non_blocking=True).reshape(-1)
        m = self.__fwd_bwd(images.to(dev, non_blocking=True), sem, ins, nobj, criterion_type or self.criterion_type, True, q_den)
        if self.distributed:
            self.__allreduce_gradients()
        flat = getattr(self.optimizer, 'flat_grad', None)
        if flat is None:
            flat = torch.cat([p.grad.reshape(-1) for p in self.model.parameters() if p.grad is not None])
        return m, flat

    def __update(self, clip_grad_norm):
        """Gradient all-reduce (data parallel), global-norm clipping and the optimizer step (model.py:271-281)."""
        if self.distributed:
            self.__allreduce_gradients()
        if hasattr(self.optimizer, 'flat_grad'):
            self.optimizer.step(clip_grad_norm=clip_grad_norm)
        else:
            if clip_grad_norm != 0:
                torch.nn.utils.clip_grad_norm_(self.model.parameters(), clip_grad_norm)
            self.optimizer.step()

    # ------------------------------------------------------------------ fit (model.py:358-464)
    def fit(self, criterion_type, delta_var, delta_dist, norm, learning_rate, weight_decay, clip_grad_norm,
            lr_drop_factor, lr_drop_patience, optimize_bg, optimizer, train_cnn, n_epochs, class_weights,
            train_loader, test_loader, model_save_path, debug=False, scorer=None, score_every=1, select_by='cost'):
        """scorer (scoring.InstanceScorer): score the validation images by SBD, |DiC| and FG dice after the validation
        pass of every score_every-th epoch and of the last one, into model.score_history as (epoch, SBD, |DiC|,
        FgDice, unclustered); rank 0 also appends them to validation_scores.log.  select_by='sbd' keeps a checkpoint on each scored epoch whose mean SBD is >= the best so
        far, instead of each epoch whose validation cost is <= the best so far ('cost').  ReduceLROnPlateau steps on
        the validation cost either way."""
        assert criterion_type in ['CE', 'Dice', 'Multi']
        if select_by not in ('cost', 'sbd'):
            raise ValueError("select_by=%r: expected 'cost' or 'sbd'" % (select_by,))
        if select_by == 'sbd' and scorer is None:
            raise ValueError("select_by='sbd' needs a scorer")
        if int(score_every) < 1:
            raise ValueError("score_every=%r: must be >= 1" % (score_every,))
        rank0 = (not self.distributed) or dist.get_rank() == 0
        if rank0:
            os.makedirs(model_save_path, exist_ok=True)
            training_log_file = open(os.path.join(model_save_path, 'training.log'), 'w')
            validation_log_file = open(os.path.join(model_save_path, 'validation.log'), 'w')
            training_log_file.write('Epoch,Cost\n')
            validation_log_file.write('Epoch,Cost\n')
            if scorer is not None:
                scores_log_file = open(os.path.join(model_save_path, 'validation_scores.log'), 'w')
                scores_log_file.write('Epoch,' + ','.join(scoring.COLUMNS) + '\n')
        self.define_criterion(class_weights, delta_var, delta_dist, norm=norm, optimize_bg=optimize_bg, criterion=criterion_type)
        if not train_cnn:
            for p in self.model.base.parameters():
                p.requires_grad = False
        self.define_optimizer(learning_rate, weight_decay, lr_drop_factor, lr_drop_patience, optimizer=optimizer)
        best_val_cost = np.inf
        best_sbd = scoring.BestSBD()
        history = []
        self.score_history = []
        for epoch in range(n_epochs):
            t0 = time.time()
            train_metrics = self.__run_epoch(train_loader, clip_grad_norm, 'training')
            val_metrics = self.__run_epoch(test_loader, 0.0, 'test')
            train_cost, val_cost = train_metrics['Cost'], val_metrics['Cost']
            t_epoch = time.time() - t0
            scores = None
            if scorer is not None and scoring.is_scored_epoch(epoch, n_epochs, int(score_every)):
                t1 = time.time()
                scores = scoring.epoch_scores(scorer.score(self), scorer.n_images, self.device)
                self.score_history.append((epoch,) + scores)
            self.lr_scheduler.step(val_cost)
            history.append((epoch, train_cost, val_cost))
            if rank0:
                print('Epoch : [{}/{}] - [{:.1f}s]  Training Cost {:.5f} | Validation Cost {:.5f}'.format(
                    epoch, n_epochs, t_epoch, train_cost, val_cost))
                if scores is not None:
                    print('Epoch : [{}/{}] - [{:.1f}s]  Validation SBD {:.5f} | |DiC| {:.4f} | FG Dice {:.5f} | '
                          'unclustered {}/{}'.format(epoch, n_epochs, time.time() - t1, scores[0], scores[1], scores[2],
                                                     scores[3], scorer.n_images))
                    scores_log_file.write('{},{},{},{},{}\n'.format(epoch, *scores))
                    scores_log_file.flush()
                lr = self.optimizer.param_groups[0]['lr']
                if select_by == 'cost' and val_cost <= best_val_cost:
                    best_val_cost = val_cost
                    torch.save(self.model.state_dict(), os.path.join(model_save_path, 'model_{}_{}_{}.pth'.format(epoch, val_cost, lr)))
                if select_by == 'sbd' and scores is not None and best_sbd.keep(scores[0]):
                    torch.save(self.model.state_dict(), os.path.join(model_save_path, 'model_{}_sbd{}_{}.pth'.format(epoch, scores[0], lr)))
                training_log_file.write('{},{}\n'.format(epoch, train_cost))
                validation_log_file.write('{},{}\n'.format(epoch, val_cost))
                training_log_file.flush()
                validation_log_file.flush()
        if rank0:
            training_log_file.close()
            validation_log_file.close()
            if scorer is not None:
                scores_log_file.close()
        return history

    def __run_epoch(self, loader, clip_grad_norm, mode):
        """Mean metrics of one pass over `loader`.  Data parallel: every rank sees its own shard, so the sums are
        all-reduced -- ReduceLROnPlateau (whose learning rate is a per-rank kernel argument) and the best-checkpoint
        test then see the SAME validation cost on every rank and the replicas cannot drift apart."""
        from .data import CudaPrefetcher
        sums, n = {}, 0
        for images, sem, ins, nobj in CudaPrefetcher(loader, self.device):
            m = self.train_step(images, sem, ins, nobj, clip_grad_norm, mode=mode)
            for k, v in m.items():
                sums[k] = sums.get(k, 0.0) + v
            n += 1
        if self.distributed:
            return parallel.allreduce_epoch_metrics(sums, n, self.device)
        return {k: float(v) / max(n, 1) for k, v in sums.items()}

    # ------------------------------------------------------------------ predict (model.py:466-499)
    @torch.no_grad()
    def predict_device_with_counts(self, images):
        """-> (sem_probs, embeddings, n_pred) on the device, nothing synchronised; n_pred (b,) int32 is the count head's
        clamp(round(s K), 1, K), or None without the head."""
        assert len(images.size()) == 4  # b, c, h, w
        self.model.eval()
        images = images.to(self.device, non_blocking=True).contiguous(memory_format=torch.channels_last)
        outputs = self.model(False, images)
        sem_seg_predictions = torch.nn.functional.softmax(outputs[0], dim=1)
        n_pred = outputs[2].evaluate().n_pred if self.count_head else None
        return sem_seg_predictions, outputs[1], n_pred

    def predict_device(self, images):
        """-> (sem_probs, embeddings) on the device, nothing synchronised."""
        return self.predict_device_with_counts(images)[:2]

    def predict(self, images):
        sem, ins, n_pred = self.predict_device_with_counts(images)
        if self.use_instance_segmentation:
            if n_pred is not None:
                n_objects_predictions = n_pred.cpu().reshape(-1, 1)
            else:
                n_objects_predictions = torch.IntTensor([[self.n_objects_prediction]] * images.size(0))
            return sem.cpu(), ins.cpu(), n_objects_predictions
        return sem.cpu()
