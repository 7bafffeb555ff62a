"""What validation scoring costs per image (isa_b200.scoring.InstanceScorer.score): the network at batch 1, k-means on
the device, the upsampling and the SBD / foreground contingency tables, with and without the count head, at the CVPPP
shape (530x500 images, 256x256 network, k = 16, 35 restarts) and the Cityscapes shape (1024x2048, k = 64, --city_n_init
restarts).  For comparison, the same images through Prediction.predict_many (host resize and normalisation, masks copied
back) and the host metrics.calc_sbd / calc_dice / calc_dic, which is what pred_list.py + evaluate.py do.

    python tools/bench_scoring.py [--cvppp_images 25] [--city_images 3] [--city_n_init 2] [--reps 3] [--json out.json]

Prints the GPU's name and power limit with the numbers.  Untrained networks (seed 23); with the count head, its linear
layer is set so that every image predicts the head-less model's fixed k, so both legs cluster with the same k and differ
only by the branch and the 4-byte read of the count.  The timed scoring passes are bracketed by CUDA events and end in a
device synchronise; the images are a temporary directory written by this script.
"""
import argparse
import json
import math
import os
import sys
import tempfile
import time

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from bench_count_head import gpu_info  # noqa: E402
from isa_b200 import settings, synth  # noqa: E402
from isa_b200.metrics import calc_dic, calc_dice, calc_sbd  # noqa: E402
from isa_b200.model import Model  # noqa: E402
from isa_b200.prediction import Prediction  # noqa: E402
from isa_b200.scoring import InstanceScorer, list_order_means  # noqa: E402


def write_set(out, n, h, w, n_inst, scale):
    """n annotated images in the CVPPP layout; labels drawn at 1/scale and repeated (label_map is O(n_inst h w))."""
    gt = os.path.join(out, "gt")
    os.makedirs(gt, exist_ok=True)
    names = []
    for j in range(n):
        nm = "img%03d" % j
        Image.fromarray(synth.leaf_image(j, h, w)).save(os.path.join(out, nm + "_rgb.png"))
        lab = synth.label_map(np.random.RandomState(j), h // scale, w // scale, n_inst - j % 3).astype(np.int64) + 1
        lab = np.repeat(np.repeat(lab, scale, 0), scale, 1)
        lab[lab == 256] = 0
        Image.fromarray(lab.astype(np.uint8)).save(os.path.join(gt, nm + "_label.png"))
        Image.fromarray((lab > 0).astype(np.uint8)).save(os.path.join(gt, nm + "_fg.png"))
        names.append(os.path.join(out, nm + "_rgb.png"))
    return names, gt


def make_model(dev, ms, dataset, count_head):
    torch.manual_seed(23)
    m = Model(dataset, ms.MODEL_NAME, ms.N_CLASSES, ms.MAX_N_OBJECTS, use_instance_segmentation=True,
              n_embedding=ms.D_MODEL, n_objects_prediction=ms.N_OBJECTS_PREDICTION, device=dev, count_head=count_head,
              net_kwargs=dict(n_units=ms.N_RENET_UNITS, n_head=ms.N_HEAD, d_k=ms.D_K, d_v=ms.D_V))
    if count_head:      # s = (k - 1/4) / K for every image: clamp(round(s K), 1, K) = k = the fixed count
        s = (ms.N_OBJECTS_PREDICTION - 0.25) / ms.MAX_N_OBJECTS
        with torch.no_grad():
            m.model.ins_cls_out.linear.weight.zero_()
            m.model.ins_cls_out.linear.bias.fill_(math.log(s / (1 - s)))
    return m


def host_scores(pred, raws, names, gt):
    """pred_list.py + evaluate.py --empty_as_zero in memory: predict_many, then the host metrics per image."""
    rows = []
    for p, (sem, ins, n) in zip(names, pred.predict_many(iter(raws))):
        base = os.path.basename(p)[:-len("_rgb.png")]
        lab = np.array(Image.open(os.path.join(gt, base + "_label.png")))
        fg = np.array(Image.open(os.path.join(gt, base + "_fg.png"))) == 1
        sbd = 0.0 if ins.max() == 0 else calc_sbd(lab, ins)
        rows.append([sbd, calc_dic(len(np.unique(lab)) - 1, n), calc_dice(fg, (sem * 255).astype(np.uint8) == 255), n == 0])
    return rows


def leg(dev, dataset, ms, names, gt, n_init, reps):
    res = {}
    raws = [np.array(Image.open(p).convert('RGB')) for p in names]
    for head in (False, True):
        m = make_model(dev, ms, dataset, head)
        scorer = InstanceScorer(names, gt, ms.IMAGE_HEIGHT, ms.IMAGE_WIDTH, ms.MEAN, ms.STD, ms.MAX_N_OBJECTS, dev,
                                n_init=n_init)
        values = scorer.score(m)                 # warm-up: module loads, cuDNN's algorithm search at batch 1
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        times = []
        for _ in range(reps):
            s.record()
            values = scorer.score(m)
            e.record()
            torch.cuda.synchronize(dev)
            times.append(s.elapsed_time(e) / len(names))
        pred = Prediction(ms.IMAGE_HEIGHT, ms.IMAGE_WIDTH, ms.MEAN, ms.STD, False, m, 1, seed=0, n_init=n_init,
                          strict=False)
        rows = host_scores(pred, raws, names, gt)
        host = []
        for _ in range(reps):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            host_scores(pred, raws, names, gt)
            host.append((time.perf_counter() - t0) * 1e3 / len(names))
        key = "head" if head else "plain"
        res[key] = {"scorer_ms_per_image": times, "predict_many_host_metrics_ms_per_image": host,
                    "means": list_order_means(values),
                    "same_values_as_host": values.tolist() == [[float(v) for v in r] for r in rows]}
        del m, scorer, pred
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cvppp_images", type=int, default=25)
    ap.add_argument("--city_images", type=int, default=3)
    ap.add_argument("--city_n_init", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    out = {"gpu": gpu_info()}
    print("GPU (name, power limit, max SM clock):", out["gpu"])
    with tempfile.TemporaryDirectory() as tmp:
        cv = os.path.join(tmp, "cvppp")
        names, gt = write_set(cv, a.cvppp_images, 530, 500, 14, 1)
        out["cvppp"] = dict(shape="530x500 -> 256x256, k = 16, n_init = 35", images=len(names),
                            **leg(dev, "CVPPP", settings.CVPPPModelSettings(), names, gt, 35, a.reps))
        cs = os.path.join(tmp, "city")
        names, gt = write_set(cs, a.city_images, 1024, 2048, 48, 4)
        out["cityscapes"] = dict(shape="1024x2048 -> 1024x2048, k = 64, n_init = %d" % a.city_n_init, images=len(names),
                                 **leg(dev, "Cityscapes", settings.CityscapesModelSettings(), names, gt, a.city_n_init,
                                       a.reps))
    for name in ("cvppp", "cityscapes"):
        r = out[name]
        print("%s (%s, %d images):" % (name, r["shape"], r["images"]))
        for key in ("plain", "head"):
            v = r[key]
            print("  %-5s scorer %s ms/image (median %.2f); predict_many + host metrics %s ms/image (median %.2f); "
                  "identical to host: %s; means %s" % (
                      key, " ".join("%.2f" % t for t in v["scorer_ms_per_image"]), np.median(v["scorer_ms_per_image"]),
                      " ".join("%.2f" % t for t in v["predict_many_host_metrics_ms_per_image"]),
                      np.median(v["predict_many_host_metrics_ms_per_image"]), v["same_values_as_host"],
                      ["%.6f" % x for x in v["means"]]))
    print("scored epoch of a 25-image CVPPP validation split: %.3f s (plain), %.3f s (count head)" % (
        25e-3 * np.median(out["cvppp"]["plain"]["scorer_ms_per_image"]),
        25e-3 * np.median(out["cvppp"]["head"]["scorer_ms_per_image"])))
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
