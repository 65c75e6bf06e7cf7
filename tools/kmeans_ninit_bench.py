"""KMeans(n_init=R).fit on one GPU: one batched fit of R starts over a single copy of the rows against R single starts
run one after another from the same initial centres.  Prints one JSON line per shape: the GPU's name and power limit
(read in the same run), the median seeding and Lloyd times of both forms, whether the two give the same result, and
(--sklearn) scikit-learn's time on the host.

    python tools/kmeans_ninit_bench.py [--runs 5] [--sklearn]

Seeding is k-means++ in both forms: the lockstep seeding of every start (kmeans_plusplus_starts) against R calls of
kmeans_plusplus.  Times come from a host clock around work that ends in a device synchronise, after one warm-up
run of every form; the median of --runs runs is reported."""
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
from opticalflowclustering_b200 import kmeans as km   # noqa: E402

SHAPES = [  # (n, d, dtype, k, R)
    (5852, 4, torch.uint8, 8, 10),          # one 1080p grid cell of pixels
    (1_000_000, 4, torch.uint8, 8, 10),
    (200_000, 16, torch.float32, 16, 10),
    (1_000_000, 64, torch.float32, 64, 3),  # tensor-core regime: the starts run one after another
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


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t


def batched(X, k, R, seed):
    cen, t_seed = timed(lambda: km.kmeans_plusplus_starts(X, k, R, np.random.RandomState(seed))[0])
    res, t_lloyd = timed(lambda: km.lloyd(X, cen))
    return res, t_seed, t_lloyd


def sequential(X, k, R, seed):
    def seeds():
        rs = np.random.RandomState(seed)
        return [km.kmeans_plusplus(X, k, rs)[0] for _ in range(R)]
    cens, t_seed = timed(seeds)
    runs, t_lloyd = timed(lambda: [km.lloyd(X, c) for c in cens])
    return tuple(torch.stack(t) for t in zip(*runs)), t_seed, t_lloyd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--sklearn", action="store_true")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    name, power = gpu_info()
    for n, d, dt, k, R in SHAPES:
        X = rows(n, d, dt, k)
        batched(X, k, R, 0)
        sequential(X, k, R, 0)                                 # warm-up of both forms
        b_seed, b_lloyd, s_seed, s_lloyd = [], [], [], []
        equal = True
        for i in range(args.runs):                             # the two forms alternate
            rb, ts, tl = batched(X, k, R, i)
            b_seed.append(ts)
            b_lloyd.append(tl)
            rq, ts, tl = sequential(X, k, R, i)
            s_seed.append(ts)
            s_lloyd.append(tl)
            equal = equal and all(torch.equal(a, b) for a, b in zip(rb, rq))
        line = dict(gpu=name, power_limit=power, n=n, d=d, dtype=str(dt).replace("torch.", ""), k=k, n_init=R,
                    batched_seed_ms=1e3 * float(np.median(b_seed)), batched_lloyd_ms=1e3 * float(np.median(b_lloyd)),
                    sequential_seed_ms=1e3 * float(np.median(s_seed)), sequential_lloyd_ms=1e3 * float(np.median(s_lloyd)),
                    same_result=bool(equal), runs=args.runs)
        if args.sklearn:
            from sklearn.cluster import KMeans
            Xh = X.cpu().numpy()
            ts = []
            for i in range(args.runs):
                t = time.perf_counter()
                KMeans(n_clusters=k, n_init=R, random_state=i).fit(Xh)
                ts.append(time.perf_counter() - t)
            line["sklearn_host_ms"] = 1e3 * float(np.median(ts))
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
