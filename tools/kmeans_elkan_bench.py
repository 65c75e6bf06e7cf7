"""KMeans(algorithm="elkan") against Lloyd on one GPU: whole fits of ``kmeans.lloyd`` from the same seeds.  Prints one JSON
line per shape and writes them all to --out, each with the GPU's name and power limit (read in the same run):

* time per fit and per iteration of both algorithms (Lloyd as ``lloyd`` picks it: fused uint8 step, tensor cores for
  float32 at d > 32, CUDA-core E-step otherwise), their iteration counts and whether the labels agree;
* distances Elkan evaluates per row and iteration (init excluded), against Lloyd's k;
* the bound pass (ofc_kmeans_elkan_bounds, 2 n k sizeof(W) bytes plus the upper bounds) against a device-to-device copy
  of the n k lower bounds (the same bytes read and written).

    python tools/kmeans_elkan_bench.py [--runs 3] [--out profiles/kmeans_elkan_bench.json]

Fit times come from a host clock around work that ends in a device synchronise, after one warm-up fit; the median of
--runs fits is reported.  The seeds are k rows drawn without replacement from a fixed RandomState (``init="random"``), so
both algorithms start from the same centres.  Bound-pass and copy times are CUDA events over 20 launches each."""
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

SHAPES = [  # (name, n, d, dtype, k, starts)
    ("cell 5852x4 u8 k8 x10 starts", 5852, 4, torch.uint8, 8, 10),
    ("1080p 2073600x3 u8 k16", 2_073_600, 3, torch.uint8, 16, 1),
    ("1Mx32 f64 k256", 1_000_000, 32, torch.float64, 256, 1),
    ("1Mx128 f64 k256", 1_000_000, 128, torch.float64, 256, 1),
    ("1Mx64 f32 k64", 1_000_000, 64, torch.float32, 64, 1),
]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
    except Exception:
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def rows(n, d, dtype, k, seed):
    """blobs: k + 3 centres with Gaussian spread (uint8: rounded and clipped to bytes)"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    cen = torch.rand((k + 3, d), generator=g, device="cuda", dtype=torch.float64) * 210 + 20
    pick = torch.randint(0, k + 3, (n,), generator=g, device="cuda")
    X = cen[pick] + torch.randn((n, d), generator=g, device="cuda", dtype=torch.float64) * 14
    if dtype == torch.uint8:
        return X.round().clamp(0, 255).to(torch.uint8)
    return X.to(dtype)


def timed_fit(X, init, algorithm, runs):
    km.lloyd(X, init, algorithm=algorithm)
    ts, out = [], None
    for _ in range(runs):
        torch.cuda.synchronize()
        t = time.perf_counter()
        out = km.lloyd(X, init, algorithm=algorithm)
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t)
    return float(np.median(ts)), out


def event_time(fn, reps=20):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def bound_pass(X, init):
    """time of one ofc_kmeans_elkan_bounds call on a fit's buffers, and of a copy of its lower bounds"""
    Xb, _ = km._as_batch(X)
    ctx = km._Ctx(Xb.device)
    k = int(init.shape[-2])
    st = km.LloydState(ctx, Xb, k)
    centres = init.reshape(1, k, -1).to(torch.float64).contiguous()
    el = km.ElkanSteps(st, torch.zeros((1, st.d), dtype=torch.float64, device="cuda"))
    el.upper.zero_()
    el.lower.zero_()
    el.old.copy_(centres + 0.5)
    st.labels[0].zero_()
    t_bounds = event_time(lambda: el.bounds(centres, st.labels[0]))
    dst = torch.empty_like(el.lower)
    t_copy = event_time(lambda: dst.copy_(el.lower))
    nbytes = 2 * el.lower.numel() * el.lower.element_size()
    return t_bounds, t_copy, nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default="profiles/kmeans_elkan_bench.json")
    args = ap.parse_args()
    gpu, power = gpu_info()
    results = []
    for name, n, d, dtype, k, starts in SHAPES:
        X = rows(n, d, dtype, k, seed=n + d + k)
        idx = np.stack([np.random.RandomState(r).choice(n, k, replace=False) for r in range(starts)])
        init = X[torch.from_numpy(idx).cuda()].to(torch.float64)
        if starts == 1:
            init = init[0]
        t_l, (lab_l, _, _, it_l) = timed_fit(X, init, "lloyd", args.runs)
        t_e, (lab_e, _, _, it_e) = timed_fit(X, init, "elkan", args.runs)
        cnt = torch.zeros(starts, dtype=torch.int64, device="cuda")
        km.lloyd(X, init, algorithm="elkan", _n_dist=cnt)
        it_l_s, it_e_s = int(it_l.sum()), int(it_e.sum())
        t_b, t_c, nbytes = bound_pass(X, init if starts == 1 else init[0])
        r = dict(shape=name, gpu=gpu, power_limit=power, n=n, d=d, k=k, dtype=str(dtype).replace("torch.", ""), starts=starts,
                 lloyd_ms_per_fit=1e3 * t_l, elkan_ms_per_fit=1e3 * t_e, lloyd_iterations=it_l_s, elkan_iterations=it_e_s,
                 lloyd_ms_per_iteration=1e3 * t_l / it_l_s, elkan_ms_per_iteration=1e3 * t_e / it_e_s,
                 elkan_over_lloyd=t_e / t_l, labels_agree=float((lab_l == lab_e).double().mean()),
                 elkan_distances_per_row_iteration=int(cnt.sum()) / (n * (it_e_s + starts)), lloyd_distances_per_row_iteration=k,
                 bound_pass_ms=1e3 * t_b, bound_pass_GBps=nbytes / t_b / 1e9, copy_same_bytes_ms=1e3 * t_c,
                 copy_GBps=nbytes / t_c / 1e9, bound_pass_over_copy=t_b / t_c)
        print(json.dumps(r), flush=True)
        results.append(r)
        del X
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
