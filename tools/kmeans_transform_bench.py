"""KMeans.transform on one GPU (kmeans.transform -> ofc_kmeans_distances).  Prints one JSON line per shape, each with the
GPU's name and power limit (read in the same run):

* write-bound shapes (the small form): achieved bytes/s, (n d sizeof(x) + n k sizeof(out)) over the call's time, next to
  a device-to-device copy of the same byte count;
* dense shapes: FP64 instructions/s, 2 n k d over the call's time, next to a torch float64 matmul of the same n x d x k
  (the practical FP64 ceiling; the direct difference needs a subtract and an fma where the product needs one fma);
* both: torch.cdist on float64 copies, its time and its largest difference from the library.

    python tools/kmeans_transform_bench.py [--runs 5]

Times come from a host clock around work that ends in a device synchronise, after one warm-up run; the median of --runs
runs is reported.  Before every timed run a 512 MB buffer is overwritten, so no run starts from a warm L2 (126 MB)."""
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
from opticalflowclustering_b200 import kmeans as km     # noqa: E402

SHAPES = [  # (n, d, dtype, k, what): the shapes of tests/test_gpu_kmeans_transform.py
    (2_073_600, 3, torch.uint8, 8, "1080p Lab pixels (quant.py)"),
    (2_073_600, 4, torch.uint8, 8, "the reference's 4-channel pixels"),
    (1_000_000, 16, torch.float32, 16, ""),
    (1_000_000, 128, torch.float32, 256, ""),
    (1_000_000, 512, torch.float32, 256, "BASELINE configs[4] corner"),
]

_FLUSH = None


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
    except Exception:
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def median_time(fn, runs):
    global _FLUSH
    if _FLUSH is None:
        _FLUSH = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")
    fn()
    ts = []
    out = None
    for _ in range(runs):
        _FLUSH.fill_(1)
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t)
    return out, float(np.median(ts))


def rows(n, d, dt, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.randn((n, d), generator=g, device="cuda", dtype=torch.float64) * 40 + 120
    return X.round().clamp(0, 255).to(torch.uint8) if dt == torch.uint8 else X.to(dt)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("a CUDA device is required")
    name, power = gpu_info()
    for n, d, dt, k, what in SHAPES:
        X = rows(n, d, dt, d)
        Cc = rows(k, d, torch.float64, k)
        if dt == torch.float32:
            Cc = Cc.to(torch.float32)
        out, t = median_time(lambda: km.transform(X, Cc), args.runs)
        rec = {"gpu": name, "power_limit": power, "n": n, "d": d, "dtype": str(dt).split(".")[-1], "k": k,
               "out": str(out.dtype).split(".")[-1], "what": what, "form": "small" if d <= 16 and k <= 64 else "dense",
               "ms": round(t * 1e3, 4)}
        if rec["form"] == "small":
            nbytes = n * d * X.element_size() + n * k * out.element_size()
            src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            dst = torch.empty_like(src)
            _, tc = median_time(lambda: dst.copy_(src), args.runs)
            del src, dst
            rec.update({"bytes": nbytes, "GB_per_s": round(nbytes / t / 1e9, 1), "copy_ms": round(tc * 1e3, 4),
                        "copy_GB_per_s": round(nbytes / tc / 1e9, 1), "share_of_copy": round(tc / t, 3)})
        else:
            Xd, Cd = X.to(torch.float64), Cc.to(torch.float64).t().contiguous()
            _, tm = median_time(lambda: Xd @ Cd, args.runs)
            del Xd, Cd
            rec.update({"fp64_Tinst_per_s": round(2.0 * n * k * d / t / 1e12, 3), "matmul_ms": round(tm * 1e3, 4),
                        "matmul_fma_per_s_T": round(1.0 * n * k * d / tm / 1e12, 3), "time_over_matmul": round(t / tm, 3)})
        Xd, Cd = X.to(torch.float64), Cc.to(torch.float64)
        cd, tcd = median_time(lambda: torch.cdist(Xd, Cd), args.runs)
        rec.update({"cdist_ms": round(tcd * 1e3, 4), "cdist_max_abs_diff": float((cd - out.to(torch.float64)).abs().max())})
        del Xd, Cd, cd, out
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
