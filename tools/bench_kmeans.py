"""Micro-benchmark of the clustering kernels: python tools/bench_kmeans.py [n C k n_init pull]"""
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from isa_b200 import clustering  # noqa: E402


def main():
    a = sys.argv[1:]
    n, C, k, n_init = [int(v) for v in a[:4]] if len(a) >= 4 else (40000, 24, 16, 35)
    pull = float(a[4]) if len(a) > 4 else 0.7
    rs = np.random.RandomState(0)
    cent = rs.standard_normal((k, C))
    cent /= np.linalg.norm(cent, axis=1, keepdims=True)
    X = ((1 - pull) * rs.standard_normal((n, C)) + pull * cent[rs.randint(0, k, n)]).astype(np.float32)
    dev = torch.device("cuda:0")
    Xt = torch.tensor(X, device=dev).t().contiguous()
    n_dev = torch.tensor([n], device=dev, dtype=torch.int32)
    ts = []
    for it in range(6):
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        res = clustering.kmeans_fit(Xt, n_dev, k, seed=0, n_init=n_init)
        e.record()
        torch.cuda.synchronize()
        ts.append(s.elapsed_time(e))
    it_sum = int(res.n_iter.sum())
    out = {"n": n, "C": C, "k": k, "n_init": n_init, "ms_median": float(np.median(ts[1:])), "ms_min": float(np.min(ts)),
           "lloyd_iters_total": it_sum, "lloyd_iters_max": int(res.n_iter.max()), "grid_iters": int(res.info[3])}
    out["lloyd_phase_us(estep,bar1,update,bar2,loop,tail)"] = [int(v) for v in res.info[4:10].cpu()]
    med = out["ms_median"] * 1e-3
    out["restart_iters_per_s"] = it_sum / med
    out["GFMA_per_s"] = it_sum * n * k * C / med / 1e9
    out["algo_GBs"] = it_sum * n * (4 * C + 4) / med / 1e9
    if "--cpu" in a:
        from sklearn.cluster import KMeans
        t = time.time()
        KMeans(n_clusters=k, n_init=n_init, max_iter=500, random_state=0).fit_predict(X)
        out["sklearn_s"] = time.time() - t
    print(json.dumps(out))


if __name__ == "__main__":
    main()
