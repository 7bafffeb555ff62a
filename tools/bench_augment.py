"""What the resident augmentation costs (isa_augment through isa_b200.augment):

- the kernel at batch 16, 530x500 -> 256x256 with the CVPPP flags, and at batch 2, Cityscapes-shaped 1024x2048 ->
  1024x2048 with a horizontal flip and a free rotation; the bytes it must move over its event time, against the
  7.7 TB/s HBM3e bandwidth of a B200's data sheet;
- the batch-16 training step (CUDA-graph replay) fed from the resident loader next to the same step fed from fixed
  device-resident synthetic tensors, alternating;
- a PIL implementation of the same augmentation on the host cores, in images/s;
- the mean difference between Prediction.image_to_tensor (PIL's antialiased resize) and the kernel's un-augmented view.

    python tools/bench_augment.py [--runs 3] [--steps 30] [--json out.json]

Prints the GPU's name and power limit with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from isa_b200 import augment as A  # noqa: E402
from isa_b200 import settings, synth  # noqa: E402
from isa_b200.model import Model  # noqa: E402
from isa_b200.prediction import Prediction  # noqa: E402

HBM_PEAK = 7.7e12


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or torch.cuda.get_device_name(0)
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + " (power limit: nvidia-smi unavailable)"


def cvppp_pairs(n, h=530, w=500):
    return [(synth.leaf_image(i, h, w), synth.label_map(np.random.RandomState(i), h, w, 12 + i % 12)) for i in range(n)]


def make_store(pairs, ts, dev):
    return A.ImageStore(["img%d" % i for i in range(len(pairs))], [p[0] for p in pairs], [p[1] for p in pairs],
                        ts.MEAN, ts.STD, dev)


def min_bytes(store, table, H, W):
    """14 B written per output pixel (12 of f32 image, class map, label map) + each source read once (3 B RGB + 1 B
    label per pixel): a lower bound on the traffic."""
    src = sum(4 * store.sizes[int(i)][0] * store.sizes[int(i)][1] for i in set(table[:, 0].tolist()))
    return table.shape[0] * H * W * 14 + src


def time_kernel(store, table, H, W, iters):
    params = torch.from_numpy(table).to(store.rgb.device)
    for _ in range(3):
        A.augment(store, params, H, W)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        A.augment(store, params, H, W)
    e.record()
    torch.cuda.synchronize()
    us = s.elapsed_time(e) * 1e3 / iters
    nb = min_bytes(store, table, H, W)
    return {"b": int(table.shape[0]), "us": us, "min_bytes": nb, "GB_per_s": nb / us * 1e-3,
            "share_of_hbm_peak": nb / (us * 1e-6) / HBM_PEAK}


def make_model(dev):
    ts = settings.CVPPPTrainingSettings()
    torch.manual_seed(23)
    m = Model('CVPPP', 'ReSeg', ts.N_CLASSES, ts.MAX_N_OBJECTS, use_instance_segmentation=True, n_embedding=ts.D_MODEL,
              n_objects_prediction=ts.N_OBJECTS_PREDICTION, device=dev)
    m.define_criterion(None, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM, ts.OPTIMIZE_BG, ts.CRITERION)
    m.define_optimizer(ts.LEARNING_RATE, ts.WEIGHT_DECAY, ts.LR_DROP_FACTOR, ts.LR_DROP_PATIENCE, ts.OPTIMIZER)
    m.enable_cuda_graph(warmup_steps=3)
    return m, ts


def time_train(dev, store, resident, steps):
    m, ts = make_model(dev)
    if resident:
        loader = A.AugmentLoader(store, 16, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, A.flags_from_settings(ts), ts.SEED, True)

        def batches():
            while True:
                for b in loader:
                    yield b
    else:
        d = synth.batch(11, 16, 3, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, ts.MAX_N_OBJECTS)
        lab = torch.tensor(d["labels"], device=dev)
        fixed = (torch.tensor(d["emb"], device=dev).contiguous(memory_format=torch.channels_last), (lab != 255).to(torch.uint8),
                 lab, torch.tensor(d["n_objects"], device=dev))

        def batches():
            while True:
                yield fixed
    it = batches()
    for _ in range(6):
        m.train_step(*next(it), clip_grad_norm=ts.CLIP_GRAD_NORM)
    torch.cuda.synchronize(dev)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        out = m.train_step(*next(it), clip_grad_norm=ts.CLIP_GRAD_NORM)
    e.record()
    torch.cuda.synchronize(dev)
    assert all(np.isfinite(float(v)) for v in out.values())
    del m
    torch.cuda.empty_cache()
    return s.elapsed_time(e) / steps


def pil_augment(rgb, lab, p, H, W, mean, std):
    """The same geometry with PIL on the host: D4 by transpose(), rotation with rotate(), resize to (W, H); bilinear
    RGB, nearest labels; then normalisation and the renumbering."""
    im, lb = Image.fromarray(rgb), Image.fromarray(lab)
    ops = []
    if p["hflip"]:
        ops.append(Image.FLIP_LEFT_RIGHT)
    if p["vflip"]:
        ops.append(Image.FLIP_TOP_BOTTOM)
    if p["transpose"]:
        ops.append(Image.TRANSPOSE)
    ops += [Image.ROTATE_90] * p["k"]
    for op in ops:
        im, lb = im.transpose(op), lb.transpose(op)
    if p["theta"] is not None:
        expand = not p["center_cut"]
        im = im.rotate(p["theta"], Image.BILINEAR, expand=expand)
        lb = lb.rotate(p["theta"], Image.NEAREST, expand=expand, fillcolor=255)
    x = np.asarray(im.resize((W, H), Image.BILINEAR), dtype=np.float32) / 255.0
    x = (x - mean) / std
    lab2 = np.asarray(lb.resize((W, H), Image.NEAREST))
    ids = np.unique(lab2[lab2 != 255])
    lut = np.full(256, 255, np.uint8)
    lut[ids] = np.arange(len(ids))
    return x, lut[lab2], len(ids)


def pil_rate(pairs, ts, n_images, workers):
    flags = A.flags_from_settings(ts)
    rs = np.random.RandomState(0)
    jobs = [(pairs[i % len(pairs)], A.draw(rs, flags)) for i in range(n_images)]
    mean, std = np.asarray(ts.MEAN, np.float32), np.asarray(ts.STD, np.float32)
    run = lambda j: pil_augment(j[0][0], j[0][1], j[1], ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, mean, std)  # noqa: E731
    with ThreadPoolExecutor(max_workers=workers) as ex:
        list(ex.map(run, jobs[:workers]))
        t0 = time.perf_counter()
        list(ex.map(run, jobs))
        t = time.perf_counter() - t0
    return n_images / t


def prediction_view_difference(store, pairs, ts):
    """mean |kernel plain view - Prediction.image_to_tensor| over the images, in normalised units and in 0..255 units."""
    pred = Prediction(ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, ts.MEAN, ts.STD, False, None, 1)
    params = torch.from_numpy(A.plain_table(store.sizes, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH)).to(store.rgb.device)
    img = A.augment(store, params, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH)[0].cpu().numpy()
    ref = np.stack([pred.image_to_tensor(p[0])[0].numpy() for p in pairs])
    d = np.abs(img - ref)
    std = np.asarray(ts.STD, np.float64).reshape(1, 3, 1, 1)
    return {"mean_abs_normalised": float(d.mean()), "mean_abs_uint8_steps": float((d * std * 255).mean()),
            "max_abs_uint8_steps": float((d * std * 255).max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--pil_images", type=int, default=256)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.backends.cudnn.benchmark = True
    res = {"gpu": gpu_info(), "host_cores": os.cpu_count()}
    print("GPU (name, power limit, max SM clock):", res["gpu"])
    ts = settings.CVPPPTrainingSettings()
    pairs = cvppp_pairs(64)
    store = make_store(pairs, ts, dev)
    table = A.epoch_table(store.sizes, 256, 256, A.flags_from_settings(ts), 23, 0)[:16]
    res["kernel_cvppp_b16"] = time_kernel(store, table, 256, 256, a.iters)
    cs = settings.CityscapesTrainingSettings()
    cpairs = [(np.random.RandomState(i).randint(0, 256, (1024, 2048, 3)).astype(np.uint8),
               synth.label_map(np.random.RandomState(i), 1024, 2048, 64)) for i in range(2)]
    cstore = make_store(cpairs, cs, dev)
    ctable = np.array([[i] + list(A.quantise(A.inverse_map(1024, 2048, 1024, 2048, hflip=i == 1, theta=10.0 + 20 * i,
                                                           center_cut=True))) for i in range(2)], dtype=np.int64)
    res["kernel_cityscapes_b2"] = time_kernel(cstore, ctable, 1024, 2048, a.iters // 4)
    for k in ("kernel_cvppp_b16", "kernel_cityscapes_b2"):
        r = res[k]
        print("%s: %.1f us per call, >= %.1f MB moved, %.0f GB/s = %.1f%% of 7.7 TB/s" % (
            k, r["us"], r["min_bytes"] / 1e6, r["GB_per_s"], 100 * r["share_of_hbm_peak"]))
    del cstore
    torch.cuda.empty_cache()
    res["train_ms"] = {"resident_loader": [], "synthetic": []}
    for r in range(a.runs):
        for resident in ((False, True) if r % 2 == 0 else (True, False)):
            res["train_ms"]["resident_loader" if resident else "synthetic"].append(time_train(dev, store, resident, a.steps))
    print("train step, batch 16, 256x256: synthetic %s ms, resident loader %s ms" % (
        " ".join("%.3f" % v for v in res["train_ms"]["synthetic"]),
        " ".join("%.3f" % v for v in res["train_ms"]["resident_loader"])))
    res["pil_images_per_s"] = pil_rate(pairs, ts, a.pil_images, os.cpu_count() or 1)
    print("PIL on %d host threads: %.0f images/s" % (os.cpu_count() or 1, res["pil_images_per_s"]))
    res["prediction_view_difference"] = prediction_view_difference(make_store(pairs[:16], ts, dev), pairs[:16], ts)
    print("plain view vs Prediction.image_to_tensor:", res["prediction_view_difference"])
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
