"""KMeans.fit(X, sample_weight=w) on one GPU.  Prints one JSON line per measurement, each with the GPU's name and power
limit (read in the same run):

* per shape, the time of a whole Lloyd fit from the same initial centres: unweighted, with weights of all ones (the
  same iterations: the cost of the weighted kernels alone -- the 8 B/row weight read and, for uint8 rows at d <= 32,
  the two-kernel iteration in place of the fused step) and with real-valued weights (a different trajectory, so its
  n_iter is printed too);
* the colour de-duplication use: the flow visualisation of one 32-pair 1080p chunk of synthetic.synthetic_clip,
  clustered by a full unweighted KMeans(8) over every pixel against its unique colours with their counts (found on the
  device) followed by a weighted KMeans(8).  It prints both times, the number of unique colours and the share of
  pixels whose label agrees with the full fit's (after matching the two fits' cluster numbers).

    python tools/kmeans_weighted_bench.py [--runs 5]

Times come from a host clock around work that ends in a device synchronise, after one warm-up run; the median of
--runs runs is reported."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opticalflowclustering_b200 import flow as fl       # noqa: E402
from opticalflowclustering_b200 import kmeans as km     # noqa: E402
from opticalflowclustering_b200.synthetic import synthetic_clip   # noqa: E402

SHAPES = [  # (n, d, dtype, k): the shapes of tests/test_gpu_kmeans_weighted.py
    (1_000_000, 4, torch.uint8, 8),
    (200_000, 16, torch.float32, 16),
    (1_000_000, 64, torch.float32, 64),
    (1_000_000, 352, torch.uint8, 256),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
    except Exception:
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def rows(n, d, dt, k, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    cen = torch.rand((k + 2, d), generator=g, device="cuda", dtype=torch.float64) * 210 + 20
    X = cen[torch.randint(0, k + 2, (n,), generator=g, device="cuda")] + torch.randn((n, d), generator=g, device="cuda",
                                                                                       dtype=torch.float64) * 15
    return X.round().clamp(0, 255).to(torch.uint8) if dt == torch.uint8 else X.to(dt)


def median_time(fn, runs):
    fn()
    ts = []
    for _ in range(runs):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t)
    return out, float(np.median(ts))


def fit_shapes(runs, info):
    for n, d, dt, k in SHAPES:
        X = rows(n, d, dt, k)
        g = torch.Generator(device="cuda").manual_seed(1)
        init = X[torch.randperm(n, generator=g, device="cuda")[:k]].to(torch.float64)
        ones = torch.ones(n, dtype=torch.float64, device="cuda")
        w = torch.rand(n, generator=g, device="cuda", dtype=torch.float64) * 2
        u, tu = median_time(lambda: km.lloyd(X, init), runs)
        o, to = median_time(lambda: km.lloyd(X, init, sample_weight=ones), runs)
        r, tr = median_time(lambda: km.lloyd(X, init, sample_weight=w), runs)
        print(json.dumps({"gpu": info[0], "power_limit": info[1], "n": n, "d": d, "dtype": str(dt).split(".")[-1], "k": k,
                          "tensor_cores": km._tc_wanted(X.unsqueeze(0), k), "unweighted_ms": round(tu * 1e3, 3),
                          "unit_weights_ms": round(to * 1e3, 3), "unit_weights_bit_identical": all(torch.equal(a, b) for a, b in zip(u, o)),
                          "n_iter": int(u[3]), "real_weights_ms": round(tr * 1e3, 3), "real_weights_n_iter": int(r[3])}), flush=True)
        del X, ones, w


def dedup(runs, info, k=8):
    """the visualisation colours of one 32-pair 1080p chunk: full fit against unique colours + counts + weighted fit"""
    H, W, P = 1080, 1920, 32
    frames = synthetic_clip(P + 1, H, W, seed=0, device="cuda")
    gray = fl.bgr2gray(frames)
    plan = fl.FarnebackPlan(W, H, max_frames=P + 1)
    flow = plan.sequence(gray)
    bgr = fl.flow_to_bgr(flow)
    X = bgr.reshape(-1, 3).contiguous()                                         # 66 M pixels

    def full():
        return km.KMeans(n_clusters=k, random_state=0).fit(X)

    def unique_weighted():
        key = (X[:, 0].to(torch.int32) << 16) | (X[:, 1].to(torch.int32) << 8) | X[:, 2].to(torch.int32)
        u, counts = torch.unique(key, return_counts=True)
        U = torch.stack([(u >> 16) & 255, (u >> 8) & 255, u & 255], dim=1).to(torch.uint8).contiguous()
        return km.KMeans(n_clusters=k, random_state=0).fit(U, sample_weight=counts.to(torch.float64)), int(u.numel())

    a, t_full = median_time(full, runs)
    (b, n_unique), t_dedup = median_time(unique_weighted, runs)
    la = a.labels_
    lb = b.predict(X)
    conf = np.zeros((k, k), np.int64)
    np.add.at(conf, (la, lb), 1)
    from scipy.optimize import linear_sum_assignment
    r, c = linear_sum_assignment(-conf)
    agree = conf[r, c].sum() / la.size
    print(json.dumps({"gpu": info[0], "power_limit": info[1], "dedup": f"{P} pairs {W}x{H}", "k": k, "pixels": int(X.shape[0]),
                      "unique_colours": n_unique, "full_fit_ms": round(t_full * 1e3, 2), "unique_plus_weighted_fit_ms": round(t_dedup * 1e3, 2),
                      "label_agreement": round(float(agree), 6), "full_n_iter": a.n_iter_, "weighted_n_iter": b.n_iter_}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("a CUDA device is required")
    info = gpu_info()
    fit_shapes(args.runs, info)
    dedup(args.runs, info)


if __name__ == "__main__":
    main()
