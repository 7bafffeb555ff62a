"""bench.py -- headline benchmark of the B200-native instance-embedding hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload train|infer|cityscapes|sweep]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Workloads (BASELINE.json `configs`):
  train (default, configs[1] / configs[2]):  one training step of the designed ReSeg path -- backbone, 2 x ReNet
        (GRU scan kernels), multi-head attention (tcgen05 kernel), heads, DiscriminativeLoss + CE + Dice,
        backward, clip, Adadelta -- on CVPPP-shaped synthetic batches of 16 images PER GPU (weak scaling;
        8 GPUs = the global batch 128 of configs[2]); data parallel = one flat NCCL gradient all-reduce.
  infer (configs[0]): pred.py: one 530x500 image -> resize 256x256 -> net -> softmax -> device clustering
        (k=16, n_init=35, max_iter=500) -> masks up-sampled to 530x500; N GPUs = N independent replicas.
  cityscapes (configs[3]): the same inference at 1024x2048 with k=64 (clustering-heavy, X no longer fits L2).
  sweep (configs[4]): discriminative-loss fwd/bwd and clustering over width 8-32, 1-128 instances, 256^2-1024^2 pixels.
The default run (N = 1) prints ONE JSON line for `train` that also carries the other three as the extra objects
"inference", "cityscapes" and "sweep", each with its own value / e2e / roofline / cpu_baseline.
`value` = whole-job images/s with inputs resident in HBM, `e2e` = the same through the public API with pinned HOST
buffers (H2D + D2H inside the timed region).  `--steps K` is the number of timed steps of every GPU leg.
`--dump-outputs DIR` writes what the timed path of the workload computed in its last step (train: the metrics, the
updated parameters and the gradient; infer / cityscapes: softmax, embedding, masks, k-means centres and inertias); the
inputs are seeded, so two builds run with the same arguments can be compared output for output.
`--impl reference` times the reference's CPU implementation of the same workload (oracle/model_ref.py: nn.GRU ReNet,
the reference's MultiHeadAttention math, its broadcast discriminative-loss graph, real scikit-learn KMeans, cv2) on
the box's host cores: the FULL batch-16 step as 8 micro-batches of 2 with gradient accumulation, every step it reports timed.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PER_GPU_BATCH = 16
NET_H = NET_W = 256
RAW_H, RAW_W = 530, 500
C_EMB, K_MAX, N_OBJ = 24, 32, 16
CITY_H, CITY_W, CITY_C, CITY_K = 1024, 2048, 32, 64
CPU_MICRO_BATCH = 2


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), bf16=float(d["bf16_tflops_sustained"]), src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1400.0, src="fallback (B200_PROFILING.md)")


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------- synthetic data
def train_batch(seed, bs, fmt="reference"):
    """(images, sem, ins, labels, n_objects): `reference` = the int64 one-hot tensors of the reference collate
    (dataset.py:354-376); `compact` = the uint8 class map / label map our collate emits (data.compact_collate)."""
    from isa_b200 import synth
    d = synth.batch(seed, bs, 3, NET_H, NET_W, K_MAX)          # d["emb"] doubles as the (b,3,H,W) image tensor
    labels = d["labels"]
    if fmt == "compact":
        sem, ins = (labels != 255).astype(np.uint8), labels
    else:
        sem = np.stack([(labels == 255), (labels != 255)], 1).astype(np.int64)
        ins = synth.onehot(labels, K_MAX, np.int64)
    return d["emb"], sem, ins, labels, d["n_objects"].astype(np.int32)


# ---------------------------------------------------------------------------------------------- rooflines
def algorithmic(name, cfg):
    """(bound, units per launch) used for roofline.achieved; formulas documented in DESIGN.md section 4."""
    bs, HW = cfg["bs"], NET_H * NET_W
    tok = cfg["bs"] * (NET_H // 4) * (NET_W // 4)
    n = 100
    if name == "isa_disc_loss_fwd":
        return "hbm", bs * HW * (4 * C_EMB + cfg["tgt_bytes"]) + bs * K_MAX * C_EMB * 4
    if name == "isa_disc_loss_bwd":     # emb read + grad write + the 1 B/pixel label map
        return "hbm", bs * HW * (8 * C_EMB + 1)
    if name == "isa_gru_scan_fwd":      # gx read + h write + stash write, both directions
        return "hbm", tok * 2 * (3 * n + n + 4 * n) * 4
    if name == "isa_gru_scan_bwd":      # dout + out + stash read, dgx + dghn write
        return "hbm", tok * 2 * (n + n + 4 * n + 3 * n + n) * 4
    if name == "isa_attention_fwd":     # 4 * BH * Lq * Lk * d flops
        L = (NET_H // 4) * (NET_W // 4)
        return "tensor", 4.0 * (2 * bs) * L * L * 12
    if name == "isa_attention_bwd":
        L = (NET_H // 4) * (NET_W // 4)
        return "tensor", 10.0 * (2 * bs) * L * L * 12
    # channels-last epilogues: 9 conv / transposed-conv outputs per step, E = bs*HW*315 elements in total
    if name == "isa_bias_act_fwd":      # read + write in place, averaged over the 9 calls
        return "hbm", bs * HW * 315 * 8 / 9.0
    if name == "isa_bias_act_bwd":      # gy read + y read + gx write
        return "hbm", bs * HW * 315 * 12 / 9.0
    if name in ("isa_pixel_heads_fwd", "isa_pixel_heads_bwd", "isa_pixel_heads_wgrad"):
        return "hbm", bs * HW * (114 + 26) * 4
    if name == "isa_add_layernorm_fwd":
        return "hbm", tok * 24 * 4 * 3
    if name == "isa_add_layernorm_bwd":
        return "hbm", tok * 24 * 4 * 4
    if name == "isa_seg_losses_fwd":    # 2 logits + 1 class byte per pixel
        return "hbm", bs * HW * 9
    if name == "isa_seg_losses_bwd":    # + 2 gradient planes written
        return "hbm", bs * HW * 17
    if name in cfg.get("gemm_flops", {}):   # ReNet projection GEMMs: 2*M*N*K useful flops per call (fp32-accurate bf16x3 = 3 MMAs per product)
        return "tensor", cfg["gemm_flops"][name]
    if name in cfg.get("bytes", {}):
        return "hbm", cfg["bytes"][name]
    return None, 0.0


def ncu_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel behind `name`, from the committed
    `ncu --set full` captures (profiles/r2_ncu_traffic.json, else round 1's); None when no capture exists for it."""
    for f in ("r2_ncu_traffic.json", "r1_ncu_traffic.json"):
        p = os.path.join(ROOT, "profiles", f)
        if os.path.exists(p):
            try:
                v = json.load(open(p)).get(name, {}).get("dram_bytes_per_launch")
                if v is not None:
                    return v
            except Exception:
                pass
    return None


def roofline_entry(name, n_calls, total_ms, cfg, peaks):
    bound, units = algorithmic(name, cfg)
    if bound is None or n_calls == 0 or total_ms <= 0 or units <= 0:
        return None
    per_launch_s = total_ms / n_calls * 1e-3
    if bound == "hbm":
        ach, peak, unit = units / per_launch_s / 1e9, peaks["hbm"], "GB/s"
    else:
        ach, peak, unit = units / per_launch_s / 1e12, peaks["bf16"], "TFLOP/s"
    return {"kernel": name, "bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
            "traffic": ncu_traffic(name), "peak_source": peaks["src"], "launches_timed": n_calls, "avg_launch_us": per_launch_s * 1e6}


METRIC = "images/sec (pred.py inference, train step at 1/2/4/8 B200) vs host-CPU ref"
INFER_WORKLOAD = ("pred.py inference: 530x500 RGB -> 256x256 -> ReSeg path -> softmax -> device k-means "
                  "(k=16, n_init=35, max_iter=500, seed 0) -> masks at 530x500; batch 1 per GPU, replicas only")
CITY_WORKLOAD = ("Cityscapes-shaped inference: 1024x2048 RGB -> ReSeg path (ReNet on the 256x512 map, attention L=131072, "
                 "width 32) -> softmax -> device k-means (k=64, n_init=35, max_iter=500, seed 0) -> masks; batch 1 per GPU")
TRAIN_WORKLOAD = ("CVPPP-shaped training step: backbone + 2xReNet(100) + MHA(2 heads, d_k=12, L=4096) + heads + "
                  "DiscriminativeLoss(C=24,K=32) + CE + Dice, fwd+bwd+clip+Adadelta, 256x256, batch 16 per GPU")
DTYPE = "f32 (hot path fp32-accurate: bf16x3 tensor-core products, fp32 accumulation; cuDNN backbone convolutions at PyTorch's default TF32)"


def _timed_plain(torch):
    def timed(step_fn, n_steps, n_warm):
        for i in range(n_warm):
            step_fn(i)
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(n_steps):
            step_fn(n_warm + i)
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e)
    return timed


DUMP_BUDGET_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes each of `arrays` (name -> tensor) as out_dir/<name>.npy, float64 kept, every other dtype as
    float32, at most DUMP_BUDGET_BYTES in all.  Smaller arrays are written whole; an array above its share of what is left
    becomes a fixed sample of its flattened elements (seed 0, indices ascending), so runs with the same arguments write
    files of the same shape that can be compared element for element."""
    os.makedirs(out_dir, exist_ok=True)
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
        host[name] = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
    left = DUMP_BUDGET_BYTES - 1024 * len(host)          # room for the .npy headers
    names = sorted(host, key=lambda n: host[n].nbytes)
    for i, name in enumerate(names):
        a = host[name]
        cap = left // (len(names) - i) // a.itemsize
        if a.size > cap:
            idx = np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))
            a = a.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


# ---------------------------------------------------------------------------------------------- clustering parity
def clustering_parity(pred, model, tens, k, raw_hw, max_images=4, budget_s=100.0, oracle_images=2):
    """Parity of the device clustering on the benchmark images, outside the timed region: bit-exact against the oracle
    (oracle/kmeans_oracle.c), against the real scikit-learn (labels up to permutation, SBD / |DiC| of the masks through
    metrics.calc_sbd / calc_dic), and -- where scikit-learn differs -- how stable scikit-learn itself is on that image
    (1 thread vs all threads; feature columns reversed): its fp32 BLAS sums depend on the thread count, so on near-tied
    random-init embeddings its own answer is not unique."""
    from oracle import kmeans as KM
    from isa_b200 import metrics
    t_start = time.time()
    per_image = []
    for ti in range(min(len(tens), max_images)):
        if time.time() - t_start > budget_s:
            break
        sem, emb = model.predict_device(tens[ti])
        fg, X = KM.gather_foreground(sem[0].cpu().numpy(), emb[0].cpu().numpy())
        if len(X) < k:
            continue
        got = pred.cluster_device(sem[0], emb[0], k)[1].cpu().numpy()
        ours = got[fg != 0]
        # the C oracle takes ~12 s of host time per image: bit-exactness is re-checked on the first images only (the GPU
        # tests assert it on every shape); None = not checked on this image
        o = KM.kmeans_oracle(X, k, seed=0) if ti < oracle_images else None
        sk = KM.sklearn_fit_predict(X, k, 0)
        sk_mask = KM.scatter_labels(fg, sk)
        rec = {"identical_to_oracle": bool(np.array_equal(got, KM.scatter_labels(fg, o["labels"]))) if o is not None else None,
               "identical_to_sklearn": bool(KM.same_up_to_permutation(ours, sk + 1)),
               "agreement_with_sklearn": round(float(KM.partition_agreement(ours, sk + 1)), 5),
               "sbd_ours_vs_sklearn_masks": round(float(metrics.calc_sbd(sk_mask, got)), 5),
               "dic_ours_vs_sklearn": int(metrics.calc_dic(len(np.unique(sk)), len(np.unique(ours))))}
        if not rec["identical_to_sklearn"]:
            x64 = X.astype(np.float64)

            def inertia(lab):
                return float(sum(((x64[lab == c] - x64[lab == c].mean(0)) ** 2).sum() for c in np.unique(lab)))
            rec["inertia_rel_diff_vs_sklearn"] = (inertia(ours) - inertia(sk + 1)) / inertia(sk + 1)
            try:
                from threadpoolctl import threadpool_limits
                with threadpool_limits(limits=1):
                    sk1 = KM.sklearn_fit_predict(X, k, 0)
                rec["sklearn_self_agreement_1_vs_all_threads"] = round(float(KM.partition_agreement(sk1, sk)), 5)
                rec["sbd_sklearn_1thread_vs_all_threads_masks"] = round(float(metrics.calc_sbd(sk_mask, KM.scatter_labels(fg, sk1))), 5)
                # the same points with the feature columns reversed: the identical problem in exact arithmetic (every
                # distance, mean and the k-means++ stream are unchanged), only the fp32 summation order differs
                skr = KM.sklearn_fit_predict(np.ascontiguousarray(X[:, ::-1]), k, 0)
                rec["sklearn_self_agreement_feature_order_reversed"] = round(float(KM.partition_agreement(skr, sk)), 5)
                rec["sbd_sklearn_feature_order_reversed_masks"] = round(float(metrics.calc_sbd(sk_mask, KM.scatter_labels(fg, skr))), 5)
            except Exception as e:   # threadpoolctl missing: the instability evidence is skipped, the mismatch stays reported
                rec["sklearn_self_agreement_error"] = repr(e)
        per_image.append(rec)
    flags = {"images_checked": len(per_image),
             "labels_identical_to_oracle": bool(per_image) and all(r["identical_to_oracle"] for r in per_image if r["identical_to_oracle"] is not None),
             "images_checked_against_oracle": int(sum(1 for r in per_image if r["identical_to_oracle"] is not None)),
             "images_identical_to_sklearn": int(sum(r["identical_to_sklearn"] for r in per_image)),
             "labels_identical_to_sklearn_up_to_permutation": bool(per_image) and all(r["identical_to_sklearn"] for r in per_image),
             "images_where_sklearn_disagrees_with_itself": int(sum(1 for r in per_image if min(
                 r.get("sklearn_self_agreement_1_vs_all_threads", 1.0),
                 r.get("sklearn_self_agreement_feature_order_reversed", 1.0)) < 1.0)),
             "sklearn_partition_agreement": min([r["agreement_with_sklearn"] for r in per_image]) if per_image else None,
             "per_image": per_image}
    return flags


def structured_parity(dev, n_cases=3):
    """The same check on STRUCTURED embeddings at the CVPPP size: planted clusters as tight as a network trained with this
    loss makes them (pull 0.9: within-cluster spread ~0.5 against centre distances ~1.3, cf. delta_var 0.5 / delta_dist
    1.5).  scikit-learn is stable there and the device labels must be identical to it."""
    import torch
    from isa_b200 import clustering, synth
    from oracle import kmeans as KM
    ident = []
    for j in range(n_cases):
        d = synth.batch(40 + j, 1, C_EMB, NET_H, NET_W, N_OBJ, n_min=N_OBJ, n_max=N_OBJ, pull=0.9)
        lab = d["labels"][0]
        sem = np.stack([(lab == 255).astype(np.float32) * 0.8 + 0.1, (lab != 255).astype(np.float32) * 0.8 + 0.1])
        fg, X = KM.gather_foreground(sem, d["emb"][0])
        got = clustering.cluster_embeddings(torch.tensor(sem, device=dev), torch.tensor(d["emb"][0], device=dev), N_OBJ)[1].cpu().numpy()
        sk = KM.sklearn_fit_predict(X, N_OBJ, 0)
        ident.append(bool(KM.same_up_to_permutation(got[fg != 0], sk + 1)))
    return {"structured_images_checked": len(ident), "structured_images_identical_to_sklearn": int(sum(ident))}


# ---------------------------------------------------------------------------------------------- inference legs
def inference_leg(model, dev, peaks, steps, warmup, rank=0, world=1, sampler=None, timed=None, with_cpu=True, shape="cvppp",
                  dump_dir=None):
    """pred.py inference: value (inputs in HBM), e2e (host image in, host masks out), per-kernel times, parity flags
    against the oracle / scikit-learn, and (N = 1) the host-CPU reference beside it.  shape: cvppp (configs[0]) or
    cityscapes (configs[3]).  dump_dir: rank 0 writes the last timed step's outputs there (dump_outputs)."""
    import torch
    from isa_b200 import _lib, synth
    from isa_b200.prediction import Prediction
    from isa_b200 import settings
    city = shape == "cityscapes"
    ms_ = settings.CityscapesModelSettings() if city else settings.CVPPPModelSettings()
    raw_h, raw_w = (CITY_H, CITY_W) if city else (RAW_H, RAW_W)
    k = CITY_K if city else N_OBJ
    C = CITY_C if city else C_EMB
    pred = Prediction(ms_.IMAGE_HEIGHT, ms_.IMAGE_WIDTH, ms_.MEAN, ms_.STD, False, model, 1, seed=0)
    n_img = 2 if city else 4
    raws = [synth.leaf_image(100 * rank + j, raw_h, raw_w) for j in range(n_img)]
    tens = [pred.image_to_tensor(r)[0].unsqueeze(0).to(dev) for r in raws]
    last = {}

    def step_dev(i):
        sem, emb = model.predict_device(tens[i % n_img])
        last["net"] = (sem, emb)
        last["o"] = pred.cluster_device(sem[0], emb[0], k, raw_h, raw_w)

    def _raw_cycle():
        j = 0
        while True:
            yield raws[j % n_img]
            j += 1

    e2e_results = pred.predict_many(_raw_cycle())    # the pipelined public path pred_list.py uses

    def step_e2e(i):
        last["masks"] = next(e2e_results)            # host image in -> host uint8 masks out

    if timed is None:
        timed = _timed_plain(torch)
    _lib.TIMER.reset()
    if sampler is not None:
        sampler.start()
    timed(step_dev, 0, warmup)
    _lib.TIMER.enabled = True
    ms = timed(step_dev, steps, 0)
    _lib.TIMER.enabled = False
    clocks = sampler.stop() if sampler is not None else None
    summ = _lib.TIMER.summary()
    launches = sum(_lib.KERNELS_PER_CALL[k_] * c for k_, (c, _) in summ.items())
    res = last["o"][4]
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"sem": last["net"][0], "emb": last["net"][1], "fg_mask": last["o"][3],
                                "ins_mask": last["o"][2], "centers": res.centers, "inertia": res.inertia})
    ms_e2e = timed(step_e2e, steps, 1)
    n_pts = int(res.info[2])
    it_sum = int(res.n_iter.sum())
    km = summ.get("isa_kmeans_fit", (1, 0.0))
    per_launch_s = km[1] / max(km[0], 1) * 1e-3
    units = it_sum * n_pts * (4 * C + 4)
    flops = 2.0 * it_sum * n_pts * k * C
    ach = units / max(per_launch_s, 1e-12) / 1e9
    total_img = world * steps
    flags = {}
    if rank == 0:
        if city:
            # the oracle needs ~10 minutes at this size: bit-exactness at 1024x2048 is covered with a bounded budget by
            # tests/test_cityscapes_shape_gpu.py; here only what fits the bench's time
            flags = {"parity": "see tests/test_cityscapes_shape_gpu.py (bit-exact vs the oracle with a bounded restart / iteration budget)"}
        else:
            flags = clustering_parity(pred, model, tens, k, (raw_h, raw_w))
            flags.update(structured_parity(dev))
    leg = {
        "value": total_img / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
        "config": {"workload": CITY_WORKLOAD if city else INFER_WORKLOAD,
                   "l2": ("X (n x 32 fp32 = %.0f MB) + labels exceed the L2 share of a restart: HBM/L2 streamed every iteration" % (n_pts * C * 4 / 1e6)) if city
                   else "%d alternating images; per-image working set (35 restarts x labels + X) < L2 by design" % n_img,
                   "fg_points": n_pts, "lloyd_restart_iterations": it_sum, "lloyd_grid_iterations": int(res.info[3]),
                   "kernel_ms_per_step": {k_: round(v[1] / steps, 4) for k_, v in sorted(summ.items())}, **flags},
        "e2e": {"value": total_img / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": 3 * ms_.IMAGE_HEIGHT * ms_.IMAGE_WIDTH * 4,
                "d2h_bytes_per_step": 2 * raw_h * raw_w},
        "gpu_launches": launches,
        "roofline": {"kernel": "isa_kmeans_fit", "bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s",
                     "frac": ach / peaks["hbm"], "traffic": ncu_traffic("isa_kmeans_fit_city" if city else "isa_kmeans_fit"), "peak_source": peaks["src"],
                     "note": "bytes = restart-iterations * n * (4C+4) (X re-read once per restart-iteration; at the CVPPP size it is "
                             "L2 resident, so the FP32-pipe figure next to it is the binding one)",
                     "fp32_tflops": flops / max(per_launch_s, 1e-12) / 1e12,
                     "fp32_pipe_frac_of_%s_tflops" % ("%.0f" % FP32_PEAK_TFLOPS): flops / max(per_launch_s, 1e-12) / 1e12 / FP32_PEAK_TFLOPS,
                     "restart_iterations_per_s": it_sum / max(per_launch_s, 1e-12),
                     "avg_launch_us": per_launch_s * 1e6},
    }
    if clocks is not None:
        leg["clocks"] = clocks
    if with_cpu and rank == 0:
        leg["cpu_baseline"] = cpu_reference("cityscapes" if city else "infer", steps=2 if city else 3, warmup=0 if city else 1,
                                            n_points=n_pts if city else None)
    return leg


FP32_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FMA lanes x 2 flop x 1.965 GHz = 74.4


# ---------------------------------------------------------------------------------------------- microbench sweep
def sweep_leg(dev, peaks, quick=True):
    """configs[4]: discriminative-loss forward / backward and clustering over embedding width 8-32, 1-128 instances,
    256^2-1024^2 pixels, through the raw C-ABI on preallocated buffers; CUDA events, L2 flushed between launches."""
    import torch
    from isa_b200 import _lib, clustering, synth
    lib = _lib.load()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def t_us(fn, iters=7, warm=2):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e) * 1e3)
        return float(np.median(ts))

    rows = []
    grid = [(16, 8, 256, 1), (16, 8, 256, 128), (16, 16, 256, 16), (16, 24, 256, 32), (16, 32, 256, 128),
            (16, 24, 512, 32), (16, 32, 512, 128), (1, 32, 1024, 64), (1, 8, 1024, 1), (16, 32, 1024, 128)]
    for bs, C, S, K in grid:
        d = synth.batch(7, bs, C, S, S, K, n_min=K, n_max=K)
        x = torch.tensor(d["emb"], device=dev)
        lab = torch.tensor(d["labels"], device=dev)
        n = torch.tensor(d["n_objects"], device=dev, dtype=torch.int32)
        loss, terms, means = torch.empty(1, device=dev), torch.empty(4, device=dev), torch.empty(bs, K, C, device=dev)
        grad, gl = torch.empty_like(x), torch.ones(1, device=dev)
        wsb = lib.isa_disc_loss_workspace_bytes(bs, C, K, S, S)
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)

        def fwd():
            rc = lib.isa_disc_loss_fwd(x.data_ptr(), lab.data_ptr(), 0, n.data_ptr(), bs, C, S, S, K, 0.5, 1.5, 2, 1, 1.0, 0.0, 0.0, 0.005,
                                       None, loss.data_ptr(), terms.data_ptr(), means.data_ptr(), ws.data_ptr(), wsb, st)
            assert rc == 0, lib.isa_last_error()

        def bwd():
            rc = lib.isa_disc_loss_bwd(x.data_ptr(), lab.data_ptr(), 0, n.data_ptr(), bs, C, S, S, K, 0.5, 1.5, 2, 1, 1.0, 0.0, 0.0, 0.005,
                                       None, means.data_ptr(), gl.data_ptr(), None, grad.data_ptr(), ws.data_ptr(), wsb, st)
            assert rc == 0, lib.isa_last_error()

        f, b = t_us(fwd), t_us(bwd)
        P = S * S
        fb, bb = bs * P * (4 * C + 1) + bs * K * C * 4, bs * P * (8 * C + 1)
        rows.append({"op": "disc_loss", "bs": bs, "C": C, "HW": "%d^2" % S, "K": K, "fwd_us": round(f, 1), "bwd_us": round(b, 1),
                     "fwd_frac_hbm": round(fb / f / 1e3 / peaks["hbm"], 3), "bwd_frac_hbm": round(bb / b / 1e3 / peaks["hbm"], 3)})
        del x, lab, grad, ws
    kgrid = [(8, 256, 1), (8, 256, 8), (32, 256, 128), (24, 512, 16), (32, 1024, 64)]
    for C, S, k in kgrid:
        d = synth.batch(9, 1, C, S, S, max(k, 2), n_min=k, n_max=k, pull=0.7)
        labm = d["labels"][0]
        X = d["emb"][0][:, labm != 255]
        Xt = torch.tensor(np.ascontiguousarray(X), device=dev)
        n_dev = torch.tensor([Xt.shape[1]], device=dev, dtype=torch.int32)
        res = {}

        def fit():
            res["r"] = clustering.kmeans_fit(Xt, n_dev, k, seed=0, n_init=35)

        t = t_us(fit, iters=3, warm=1)
        it = int(res["r"].n_iter.sum())
        npt = Xt.shape[1]
        rows.append({"op": "kmeans", "C": C, "HW": "%d^2" % S, "k": k, "n": npt, "ms": round(t / 1e3, 3), "restart_iterations": it,
                     "frac_hbm": round(it * npt * (4 * C + 4) / t / 1e3 / peaks["hbm"], 3),
                     "fp32_tflops": round(2.0 * it * npt * k * C / t / 1e6, 2)})
    dl = [r for r in rows if r["op"] == "disc_loss"]
    return {"config": {"workload": "configs[4] sweep: label-map targets, width 8-32, 1-128 instances, 256^2-1024^2, bs 1/16; "
                                   "clustering n_init=35, planted clusters (pull 0.7)", "l2": "256 MB flush between timed launches"},
            "disc_fwd_frac_hbm_min_max": [min(r["fwd_frac_hbm"] for r in dl), max(r["fwd_frac_hbm"] for r in dl)],
            "disc_bwd_frac_hbm_min_max": [min(r["bwd_frac_hbm"] for r in dl), max(r["bwd_frac_hbm"] for r in dl)],
            "rows": rows}


# ---------------------------------------------------------------------------------------------- our arm
def dp_parity(dev, rank, world, ts):
    """N > 1, before timing: the data-parallel forward+backward (each rank on its shard, gradients all-reduced) against
    the single-process forward+backward of the CONCATENATED batch on rank 0, same weights: loss and gradient."""
    import torch
    import torch.distributed as dist
    from isa_b200.model import Model
    bs = 4
    torch.manual_seed(ts.SEED)
    kw = dict(use_instance_segmentation=True, n_embedding=C_EMB, device=dev)
    m_dp = Model('CVPPP', 'ReSeg', ts.N_CLASSES, ts.MAX_N_OBJECTS, distributed=True, **kw)
    torch.manual_seed(ts.SEED)
    m_one = Model('CVPPP', 'ReSeg', ts.N_CLASSES, ts.MAX_N_OBJECTS, distributed=False, **kw)
    for m in (m_dp, m_one):
        m.define_criterion(ts.CLASS_WEIGHTS, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM, ts.OPTIMIZE_BG, ts.CRITERION)
        m.define_optimizer(ts.LEARNING_RATE, ts.WEIGHT_DECAY, ts.LR_DROP_FACTOR, ts.LR_DROP_PATIENCE, ts.OPTIMIZER)
    shards = [train_batch(7000 + r, bs, "compact") for r in range(world)]

    def dev_t(b):
        return [torch.from_numpy(a).to(dev) for a in (b[0], b[1], b[2], b[4])]

    mine = dev_t(shards[rank])
    met, g = m_dp.loss_and_gradients(*mine)
    loss_dp = met['Cost'].detach().clone().reshape(1)
    dist.all_reduce(loss_dp)
    loss_dp = float(loss_dp) / world
    out = None
    if rank == 0:
        cat = [np.concatenate([s[i] for s in shards]) for i in (0, 1, 2, 4)]
        met1, g1 = m_one.loss_and_gradients(*[torch.from_numpy(a).to(dev) for a in cat])
        loss_one = float(met1['Cost'])
        gn, gn1 = float(g.double().norm()), float(g1.double().norm())
        out = {"global_batch": bs * world, "loss_dp": loss_dp, "loss_single_process": loss_one,
               "loss_rel_diff": abs(loss_dp - loss_one) / abs(loss_one),
               "grad_norm_dp": gn, "grad_norm_single_process": gn1, "grad_norm_rel_diff": abs(gn - gn1) / gn1,
               "grad_max_abs_diff_over_max": float((g - g1).abs().max() / g1.abs().max())}
        out["ok"] = bool(out["loss_rel_diff"] < 1e-5 and out["grad_norm_rel_diff"] < 1e-4)
    dist.barrier()
    del m_dp, m_one
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from isa_b200 import _lib, parallel
    from isa_b200.model import Model
    from isa_b200.settings import CVPPPTrainingSettings, CityscapesTrainingSettings

    rank, world, local_rank = parallel.init_from_env("nccl")
    assert torch.cuda.is_available(), "bench.py needs a B200: there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, world)
    peaks = measured_peaks()
    ts = CVPPPTrainingSettings()
    sampler = ClockSampler(local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps, warmup):
        for i in range(warmup):
            step_fn(i)
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for i in range(steps):
            step_fn(warmup + i)
        e.record()
        barrier()
        return parallel.max_over_ranks(s.elapsed_time(e), dev)

    def fresh_model(dataset='CVPPP'):
        torch.manual_seed(ts.SEED)
        if dataset == 'Cityscapes':
            from isa_b200 import settings
            ms_ = settings.CityscapesModelSettings()
            return Model('Cityscapes', 'ReSeg', ms_.N_CLASSES, ms_.MAX_N_OBJECTS, use_instance_segmentation=True, n_embedding=ms_.D_MODEL,
                         n_objects_prediction=ms_.N_OBJECTS_PREDICTION, device=dev,
                         net_kwargs=dict(n_units=ms_.N_RENET_UNITS, n_head=ms_.N_HEAD, d_k=ms_.D_K, d_v=ms_.D_V))
        return Model('CVPPP', 'ReSeg', ts.N_CLASSES, ts.MAX_N_OBJECTS, use_instance_segmentation=True, n_embedding=C_EMB, device=dev)

    def extra_legs(out):
        """N = 1: the other BASELINE.json configs ride on the default line."""
        if args.no_inference:
            return
        m = fresh_model()
        out["inference"] = inference_leg(m, dev, peaks, steps=args.steps, warmup=args.warmup)
        del m
        torch.cuda.empty_cache()
        try:
            m = fresh_model('Cityscapes')
            out["cityscapes"] = inference_leg(m, dev, peaks, steps=args.steps, warmup=1, shape="cityscapes")
            del m
        except Exception as e:          # the leg must not take the headline down with it
            out["cityscapes"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        try:
            out["sweep"] = sweep_leg(dev, peaks)
        except Exception as e:
            out["sweep"] = {"error": repr(e)}

    out = {}
    if args.workload == "train":
        parity = dp_parity(dev, rank, world, ts) if world > 1 else None
        torch.manual_seed(ts.SEED)
        model = Model('CVPPP', 'ReSeg', ts.N_CLASSES, ts.MAX_N_OBJECTS, use_instance_segmentation=True,
                      n_embedding=C_EMB, distributed=world > 1, device=dev)
        model.define_criterion(ts.CLASS_WEIGHTS, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM, ts.OPTIMIZE_BG, ts.CRITERION)
        model.define_optimizer(ts.LEARNING_RATE, ts.WEIGHT_DECAY, ts.LR_DROP_FACTOR, ts.LR_DROP_PATIENCE, ts.OPTIMIZER)
        bs = PER_GPU_BATCH
        n_host = 2
        host, host_ref = [], []
        for j in range(n_host):
            img, sem, ins, labels, nobj = train_batch(1000 * rank + j, bs, "compact")
            host.append([torch.from_numpy(a).pin_memory() for a in (img, sem, ins, nobj)])
        devb = [[t.to(dev) for t in hb] for hb in host]
        clip = ts.CLIP_GRAD_NORM
        last = {}

        def step_dev(i):
            b = devb[i % n_host]
            last["m"] = model.train_step(b[0], b[1], b[2], b[3], clip)

        from isa_b200.data import CudaPrefetcher

        class _Cycle(object):                        # an endless loader over the pinned host batches
            def __init__(self, batches):
                self.batches = batches

            def __iter__(self):
                j = 0
                while True:
                    yield self.batches[j % len(self.batches)]
                    j += 1

            def __len__(self):
                return 1 << 30

        e2e_batches = iter(CudaPrefetcher(_Cycle(host), dev))   # the public staging path Model.fit uses (data.py)

        def step_e2e(i):
            b = next(e2e_batches)                    # H2D of this step's pinned inputs (overlaps the previous step)
            m = model.train_step(b[0], b[1], b[2], b[3], clip)
            last["loss"] = float(m['Cost'])          # device -> host read of the step's result

        # (a) per-kernel times: an EAGER pass with CUDA events around every C-ABI call (explains the step, is not the value)
        _lib.TIMER.reset()
        timed(step_dev, 0, args.warmup)              # warm-up outside the kernel timers
        _lib.TIMER.enabled = True
        ms_eager = timed(step_dev, args.steps, 0)
        _lib.TIMER.enabled = False
        summ = _lib.TIMER.summary()
        launches = sum(_lib.KERNELS_PER_CALL[k] * c for k, (c, _) in summ.items())
        # (b) value: inputs resident in HBM, the step replayed from its CUDA graph (Model.enable_cuda_graph: the same
        #     launches per step, submitted by one cudaGraphLaunch instead of one by one from Python)
        use_graph = not args.no_graph
        if use_graph:
            model.enable_cuda_graph(warmup_steps=1)
        sampler.start()
        ms = timed(step_dev, args.steps, 3)          # the first warm-up step here captures the graph
        clocks = sampler.stop()
        if args.dump_outputs and rank == 0:
            # the step's metrics (the graph's static scalars, overwritten by the next replay) and the parameters and
            # gradient it left in the optimizer's flat buffers
            dump = {name.lower().replace(" ", "_"): v for name, v in last["m"].items()}
            dump.update(params=model.optimizer.flat_param, grad=model.optimizer.flat_grad)
            dump_outputs(args.dump_outputs, dump)
        ms_e2e = timed(step_e2e, args.steps, 1)
        h2d = sum(t.numel() * t.element_size() for t in host[0])
        # (c) the same step fed the reference collate's int64 one-hot tensors (distilled to label maps on the device)
        img, sem, ins, labels, nobj = train_batch(1000 * rank, bs, "reference")
        ref_fmt = [torch.from_numpy(a).to(dev) for a in (img, sem, ins, nobj)]
        ms_ref_fmt = timed(lambda i: model.train_step(ref_fmt[0], ref_fmt[1], ref_fmt[2], ref_fmt[3], clip), args.steps, 2)
        h2d_ref = sum(t.numel() * t.element_size() for t in ref_fmt)
        del ref_fmt
        total_img = bs * world * args.steps
        tok = bs * (NET_H // 4) * (NET_W // 4)
        cfg = {"bs": bs, "tgt_bytes": 1, "gemm_flops": {}, "bytes": {}}
        for name, (cnt, _) in summ.items():
            pass
        from isa_b200 import renet as _renet
        cfg["gemm_flops"].update(getattr(_renet, "bench_gemm_flops", lambda tok_: {})(tok))
        dom = max(summ.items(), key=lambda kv: kv[1][1])
        dom_roof = roofline_entry(dom[0], dom[1][0], dom[1][1], cfg, peaks)
        all_roof = [r for r in (roofline_entry(k_, v_[0], v_[1], cfg, peaks) for k_, v_ in sorted(summ.items())) if r]
        kernel_ms = {k: round(v[1] / args.steps, 4) for k, v in sorted(summ.items())}
        out = {
            "metric": METRIC,
            "value": total_img / (ms * 1e-3), "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": TRAIN_WORKLOAD,
                       "per_gpu_batch": bs, "global_batch": bs * world, "parallelism": "dp%d" % world,
                       "l2": "working set (activations) >> 126 MB L2, two alternating input batches",
                       "target_format": "uint8 class map + uint8 instance label map (data.compact_collate)",
                       "ms_per_step_with_reference_int64_onehot_targets": ms_ref_fmt / args.steps,
                       "h2d_bytes_per_step_reference_format": h2d_ref,
                       "kernel_ms_per_step": kernel_ms,
                       "cuda_graph": bool(use_graph), "ms_per_step_eager_with_kernel_timers": ms_eager / args.steps},
            "clocks": clocks,
            "e2e": {"value": total_img / (ms_e2e * 1e-3), "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
            "gpu_launches": launches,
            "roofline": dom_roof,
            "rooflines": all_roof,
        }
        if parity is not None:
            out["dp_parity"] = parity
        if world == 1 and not args.no_inference:
            # strict fp32 for the backbone as well (cuDNN TF32 off): what the step costs when NOTHING runs below fp32 accuracy
            torch.backends.cudnn.allow_tf32 = False
            model._graphs.clear(); model._graph_seen.clear()
            ms_strict = timed(step_dev, args.steps, 3)
            torch.backends.cudnn.allow_tf32 = True
            out["config"]["ms_per_step_cudnn_tf32_off"] = ms_strict / args.steps
            del model, devb
            torch.cuda.empty_cache()
            extra_legs(out)
    elif args.workload in ("infer", "cityscapes"):
        city = args.workload == "cityscapes"
        model = fresh_model('Cityscapes' if city else 'CVPPP')
        leg = inference_leg(model, dev, peaks, steps=args.steps, warmup=args.warmup, rank=rank, world=world, sampler=sampler,
                            timed=timed, with_cpu=False, shape="cityscapes" if city else "cvppp", dump_dir=args.dump_outputs)
        out = {
            "metric": METRIC,
            "value": leg["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": leg["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": leg["config"], "clocks": leg["clocks"], "e2e": leg["e2e"], "gpu_launches": leg["gpu_launches"],
            "roofline": leg["roofline"],
        }
    else:
        sw = sweep_leg(dev, peaks)
        out = {"metric": METRIC, "value": None, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
               "config": sw["config"], "sweep": sw}
    if rank == 0 and world == 1 and args.workload != "sweep":
        out["cpu_baseline"] = cpu_reference(args.workload, steps=3 if args.workload != "cityscapes" else 2, warmup=1 if args.workload != "cityscapes" else 0)
    if rank == 0:
        emit(out)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------- reference arm (CPU)
def cpu_reference(workload, steps=3, warmup=1, n_points=None):
    """Times the reference's CPU implementation of the workload; returns the cpu_baseline dict.  `steps` steps are timed
    after `warmup` untimed ones, and that is what the dict reports.
    train: the FULL batch-16 step -- 8 micro-batches of 2 with gradient accumulation (one batch of 16 would materialise the
    reference loss's (bs, HW, K, C) broadcast temporaries: 3.2 GB each), clip + Adadelta once per step."""
    import torch
    from oracle import kmeans as KM
    from oracle.model_ref import ReSegRef, discriminative_loss_torch
    from isa_b200 import synth
    from isa_b200.settings import CVPPPTrainingSettings
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ts = CVPPPTrainingSettings()
    torch.manual_seed(ts.SEED)
    if workload == "train":
        net = ReSegRef(ts.N_CLASSES, n_embedding=C_EMB)
        bs, mb = PER_GPU_BATCH, CPU_MICRO_BATCH
        img, sem, ins, labels, nobj = train_batch(0, bs, "reference")
        img, sem, ins = torch.from_numpy(img), torch.from_numpy(sem), torch.from_numpy(ins).float()
        opt = torch.optim.Adadelta(net.parameters(), lr=ts.LEARNING_RATE, weight_decay=ts.WEIGHT_DECAY)
        ce = torch.nn.CrossEntropyLoss()

        def step():
            net.train()
            opt.zero_grad()
            for lo in range(0, bs, mb):
                sl = slice(lo, lo + mb)
                sem_out, emb = net(True, img[sl])
                ins_cost, _ = discriminative_loss_torch(emb, ins[sl], nobj[sl], K_MAX, ts.DELTA_VAR, ts.DELTA_DIST, ts.NORM)
                probs = torch.softmax(sem_out, 1)
                semf = sem[sl].float()
                dice = (2 * (probs * semf).sum((2, 3)) + 1.0) / (probs.sum((2, 3)) + semf.sum((2, 3)) + 1.0)
                cost = ins_cost + ce(sem_out, sem[sl].max(1)[1]) + (1 - dice[:, 1:].mean(1)).mean()
                (cost * (float(mb) / bs)).backward()
            torch.nn.utils.clip_grad_norm_(net.parameters(), ts.CLIP_GRAD_NORM)
            opt.step()

        for _ in range(warmup):
            step()
        t0 = time.time()
        for _ in range(steps):
            step()
        dt = (time.time() - t0) / steps
        return {"value": bs / dt, "unit": "images/s", "cores": cores, "kind": "port", "steps_timed": steps, "warmup_steps": warmup,
                "sample": "%d full batch-%d step(s) after %d warm-up: %d micro-batches of %d with gradient accumulation, one clip + Adadelta "
                          "update per step (same graph from reference ops on the CPU: nn.GRU ReNet, reference MHA math, the reference's "
                          "broadcast discriminative-loss graph + autograd)" % (steps, bs, warmup, bs // mb, mb),
                "seconds_per_step": dt}
    if workload == "cityscapes":
        # The CPU reference cannot run the network at this shape: its dense attention materialises the L x L scores
        # (L = 131072: 68 GB per head).  What is timed is the clustering it would run (prediction.py:72-74) on a planted
        # Cityscapes-shaped point set, with a bounded n_init, extrapolated linearly to n_init = 35.
        d = synth.batch(3, 1, CITY_C, 512, 1024, CITY_K, n_min=CITY_K, n_max=CITY_K, pull=0.5)
        lab = d["labels"][0]
        X = np.ascontiguousarray(d["emb"][0][:, lab != 255].T)
        n_init = 1
        t0 = time.time()
        for _ in range(max(1, steps)):
            KM.sklearn_fit_predict(X, CITY_K, 0, n_init=n_init)
        dt = (time.time() - t0) / max(1, steps)
        # the image's foreground size: what the GPU leg clustered (a random-init net calls every pixel foreground), else 30 %
        n_full = int(n_points) if n_points else int(0.3 * CITY_H * CITY_W)
        est = dt * (35.0 / n_init) * (n_full / float(len(X)))
        return {"value": 1.0 / est, "unit": "images/s", "cores": cores, "kind": "port", "steps_timed": max(1, steps), "warmup_steps": 0,
                "sample": "clustering only (the CPU reference cannot materialise L=131072 attention scores): scikit-learn KMeans(k=64, "
                          "n_init=%d, max_iter=500) on %d points x %d, %.1f s measured; extrapolated x35/%d restarts and x%d/%d points "
                          "to the 1024x2048 image" % (n_init, len(X), CITY_C, dt, n_init, n_full, len(X)),
                "seconds_per_step": est, "measured_seconds": dt}
    net = ReSegRef(ts.N_CLASSES, n_embedding=C_EMB)
    net.eval()
    raws = [synth.leaf_image(j, RAW_H, RAW_W) for j in range(4)]
    from PIL import Image
    from isa_b200.settings import CVPPPModelSettings
    ms_ = CVPPPModelSettings()

    def step(i):
        img = Image.fromarray(raws[i % 4]).resize((NET_W, NET_H), Image.BILINEAR)
        x = (np.asarray(img, dtype=np.float32).transpose(2, 0, 1) / 255.0 - np.asarray(ms_.MEAN, np.float32).reshape(3, 1, 1)) / np.asarray(ms_.STD, np.float32).reshape(3, 1, 1)
        with torch.no_grad():
            sem_out, emb = net(False, torch.from_numpy(x).unsqueeze(0))
            sem_p = torch.softmax(sem_out, 1)
        fg, mask = KM.cluster_reference(sem_p[0].numpy(), emb[0].numpy(), N_OBJ, seed=0, impl="sklearn")
        return KM.upsample_nearest(fg, RAW_H, RAW_W), KM.upsample_nearest(mask, RAW_H, RAW_W)

    for i in range(warmup):
        step(i)
    t0 = time.time()
    for i in range(steps):
        step(warmup + i)
    dt = (time.time() - t0) / steps
    return {"value": 1.0 / dt, "unit": "images/s", "cores": cores, "kind": "port", "steps_timed": steps, "warmup_steps": warmup,
            "sample": "%d whole image(s) after %d warm-up: CPU net forward (reference ops) + real scikit-learn KMeans(k=16, n_init=35, "
                      "max_iter=500) + numpy scatter + cv2 INTER_NEAREST" % (steps, warmup),
            "seconds_per_step": dt}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if args.workload == "sweep":
        emit({"impl": "reference", "unavailable": "the sweep has no single images/s figure; see the sweep rows of the default line"})
        return
    # every step the line reports is run and timed in full; the count is bounded so the arm ends within a few minutes
    steps = max(1, min(args.steps, 3))
    warmup = max(0, min(args.warmup, 1))
    cb = cpu_reference(args.workload, steps=steps, warmup=warmup)
    wl = {"train": TRAIN_WORKLOAD, "infer": INFER_WORKLOAD, "cityscapes": CITY_WORKLOAD}[args.workload]
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": cb["value"], "unit": "images/s", "n_gpus": args.gpus, "steps": cb["steps_timed"], "warmup": cb["warmup_steps"],
        "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": cb["seconds_per_step"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl, "per_gpu_batch": PER_GPU_BATCH if args.workload == "train" else 1,
                   "arm": "host-CPU reference implementation of this workload (see cpu_baseline.sample); rank 0 only"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_REAL_STDOUT = None


def _quarantine_stdout():
    """Libraries print to fd 1 (NCCL's version banner, cuDNN notes): point fd 1 at stderr for the run and keep the
    real stdout for the ONE JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "infer", "cityscapes", "sweep"])
    ap.add_argument("--no-graph", dest="no_graph", action="store_true", help="keep the training step eager (no CUDA-graph replay)")
    ap.add_argument("--no-inference", dest="no_inference", action="store_true",
                    help="train workload: skip the extra legs (inference, cityscapes, sweep, strict fp32) reported at N = 1")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path computed in its last step as DIR/<name>.npy "
                         "(float32 / float64, at most 64 MB; larger outputs as a fixed seeded sample)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload == "sweep"):
        ap.error("--dump-outputs needs --impl ours and the train, infer or cityscapes workload")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    _quarantine_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
