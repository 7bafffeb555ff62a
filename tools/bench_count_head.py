"""What the instance-count head costs: the training step (CVPPP shape, batch 16, 256x256, CUDA-graph replay) and pred.py-shaped
inference per image, each with and without the head, alternating, plus the event-timed cost of the two tail entry points.

    python tools/bench_count_head.py [--runs 3] [--steps 30] [--images 20] [--json out.json]

Prints the GPU's name and power limit with the numbers.  The head model's linear layer is set to weight 0, bias 0 for
the inference leg (s = 0.5, so it predicts K / 2 = 16 = the head-less model's fixed count): both legs cluster with the
same k and differ only by the branch and the 4-byte read-back of the count.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from isa_b200 import _lib, settings, synth  # noqa: E402
from isa_b200.model import Model  # noqa: E402
from isa_b200.prediction import Prediction  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + " (power limit: nvidia-smi unavailable)"


def make_model(dev, count_head):
    ts = settings.CVPPPTrainingSettings()
    torch.manual_seed(23)
    m = Model('CVPPP', 'ReSeg', ts.N_CLASSES, ts.MAX_N_OBJECTS, use_instance_segmentation=True, n_embedding=ts.D_MODEL,
              n_objects_prediction=ts.N_OBJECTS_PREDICTION, device=dev, count_head=count_head)
    m.define_criterion(None, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM, ts.OPTIMIZE_BG, ts.CRITERION)
    m.define_optimizer(ts.LEARNING_RATE, ts.WEIGHT_DECAY, ts.LR_DROP_FACTOR, ts.LR_DROP_PATIENCE, ts.OPTIMIZER)
    return m, ts


def train_batch(dev, ts, bs=16):
    d = synth.batch(11, bs, 3, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, ts.MAX_N_OBJECTS)
    lab = torch.tensor(d["labels"], device=dev)
    return (torch.tensor(d["emb"], device=dev), (lab != 255).to(torch.uint8), lab, torch.tensor(d["n_objects"], device=dev))


def time_train(dev, count_head, steps):
    m, ts = make_model(dev, count_head)
    m.enable_cuda_graph(warmup_steps=3)
    b = train_batch(dev, ts)
    for _ in range(6):
        m.train_step(*b, clip_grad_norm=ts.CLIP_GRAD_NORM)
    torch.cuda.synchronize(dev)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        out = m.train_step(*b, clip_grad_norm=ts.CLIP_GRAD_NORM)
    e.record()
    torch.cuda.synchronize(dev)
    ms = s.elapsed_time(e) / steps
    assert all(np.isfinite(float(v)) for v in out.values())
    del m
    torch.cuda.empty_cache()
    return ms


def tail_call_times(dev, steps):
    """Event-timed isa_count_head_fwd / _bwd on eager steps (the timer turns graph capture off)."""
    m, ts = make_model(dev, True)
    b = train_batch(dev, ts)
    for _ in range(3):
        m.train_step(*b, clip_grad_norm=ts.CLIP_GRAD_NORM)
    _lib.TIMER.reset()
    _lib.TIMER.enabled = True
    try:
        for _ in range(steps):
            m.train_step(*b, clip_grad_norm=ts.CLIP_GRAD_NORM)
        summ = _lib.TIMER.summary()
    finally:
        _lib.TIMER.enabled = False
    out = {}
    for name in ("isa_count_head_fwd", "isa_count_head_bwd"):
        n, tot = summ.get(name, (0, 0.0))
        out[name] = {"calls": n, "us_per_call": 1e3 * tot / max(n, 1)}
    # the map the tail reads: batch 16, 256x256 -> conv4 output 16 x 64 x 16 x 16
    P, C = (ts.IMAGE_HEIGHT // 16) * (ts.IMAGE_WIDTH // 16), 64
    out["bytes"] = {"fwd": 16 * P * C * 4 * 2, "bwd": 16 * P * C * 4 * 2}
    del m
    torch.cuda.empty_cache()
    return out


def time_infer(dev, count_head, n_images):
    m, _ = make_model(dev, count_head)
    if count_head:
        with torch.no_grad():
            m.model.ins_cls_out.linear.weight.zero_()
            m.model.ins_cls_out.linear.bias.zero_()
    ms = settings.CVPPPModelSettings()
    pred = Prediction(ms.IMAGE_HEIGHT, ms.IMAGE_WIDTH, ms.MEAN, ms.STD, False, m, 1, seed=0, strict=False)
    raws = [synth.leaf_image(s, 530, 500) for s in range(4)]
    for r in raws:
        pred.predict_array(r)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    ns = []
    for i in range(n_images):
        ns.append(pred.predict_array(raws[i % len(raws)])[2])     # ends in the masks' device->host copy
    t = (time.perf_counter() - t0) / n_images * 1e3
    del m, pred
    torch.cuda.empty_cache()
    return t, sorted(set(ns))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--images", type=int, default=20)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.backends.cudnn.benchmark = True
    res = {"gpu": gpu_info(), "train_ms": {"head": [], "plain": []}, "infer_ms": {"head": [], "plain": []}}
    print("GPU (name, power limit, max SM clock):", res["gpu"])
    for r in range(a.runs):
        for head in ((False, True) if r % 2 == 0 else (True, False)):
            res["train_ms"]["head" if head else "plain"].append(time_train(dev, head, a.steps))
    res["tail_calls"] = tail_call_times(dev, 10)
    for r in range(a.runs):
        for head in ((False, True) if r % 2 == 0 else (True, False)):
            t, ns = time_infer(dev, head, a.images)
            res["infer_ms"]["head" if head else "plain"].append(t)
            res.setdefault("infer_counts", {})["head" if head else "plain"] = ns
    for leg in ("train_ms", "infer_ms"):
        p, h = res[leg]["plain"], res[leg]["head"]
        res[leg]["added_ms_median"] = float(np.median(h) - np.median(p))
        print("%s: without head %s, with head %s -> added %.3f ms (medians)" % (
            leg, " ".join("%.3f" % v for v in p), " ".join("%.3f" % v for v in h), res[leg]["added_ms_median"]))
    for name in ("isa_count_head_fwd", "isa_count_head_bwd"):
        c = res["tail_calls"][name]
        print("%s: %d calls, %.2f us per call" % (name, c["calls"], c["us_per_call"]))
    print("inference counts used (plain, head):", res["infer_counts"]["plain"], res["infer_counts"]["head"])
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
