#!/usr/bin/env python
"""Benchmark of the flow -> grid -> k-means hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]

A step = one pass of the hot path over one chunk of a synthetic 1080p clip:
`chunk` consecutive BGR frames (default 33) -> chunk-1 frame pairs through bgr2gray, Farneback
flow (levels=3, winsize=15, iterations=3), HSV visualisation, the 14x25 grid means
and the per-cell k-means(1) hues.  The clip (larger than L2) is resident in HBM
for `value`; steps walk through it so no step re-reads the previous step's inputs.
`e2e` is the same work through ClipPipeline with HOST (pinned) frames: H2D copy of
the step's new frames and D2H of its hue rows / magnitudes inside the timed region.

Under torchrun (N > 1) every rank processes its own clip shard (weak scaling, no
data-path collective); timing is max over ranks, value the aggregate.

`extras` carries the other BASELINE.json configs measured in the same run: the 720p and 4K sizes,
`-c 8` (per-cell KMeans(8), configs[1]) at 720p and 1080p with the CPU reference at k = 8, the literal
drop-in calls (numpy in / numpy out, one pair per call), the k-means / cosine sweep of configs[4], and --
on every N -- the one collective of the path: whole Lloyd fits over row-sharded vectors with the NCCL
all-reduce (`dist_kmeans`), plus the host-link ceiling with all ranks uploading at once.

`--dump-outputs DIR` writes what the last timed step computed (rank 0) as DIR/<name>.npy.  The clip is
generated from a fixed seed, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "1080p frame-pairs/sec (flow+grid+k-means)"
UNIT = "frame-pairs/s"
H, W = 1080, 1920
LEVELS = 3
SIZE_NAME = "1080p"
# other BASELINE.json configs (parity-test / documentation runs, not the headline): --size 720p | 4k
SIZES = {"720p": (720, 1280, 3, 422.8e6), "1080p": (1080, 1920, 3, 951.4e6), "4k": (2160, 3840, 5, 3836.6e6)}
ROWS, COLS = 14, 25
LANES = 3                        # chunks in flight in the timed loops (--lanes)
# SURVEY.md §8(d): algorithmic bytes per 1080p pair (levels=3) for flow+viz+grid, and
# per flow_iter launch per pixel (update-matrices 68 B + blur/solve 28 B)
ALGO_BYTES_PER_PAIR = 951.4e6
ITER_BYTES_PER_PX = 96.0
FUSED_ITER_BYTES_PER_PX = 56.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chunk", type=int, default=33, help="frames per step (pairs = chunk-1)")
    ap.add_argument("--clip-frames", type=int, default=129)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--size", default="1080p", choices=sorted(SIZES), help="frame size (the metric is quoted on 1080p)")
    ap.add_argument("--k", type=int, default=1, help="the reference's -c: clusters per grid cell (every documented command uses 1)")
    ap.add_argument("--no-extras", action="store_true", help="only the headline workload")
    ap.add_argument("--lanes", type=int, default=3, help="chunks in flight on separate streams (LanedPipeline); 1 = one chain of kernels")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 / "
                         "float64; flow and visualisation as a fixed, seeded sample of pixels) to compare two builds")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    global H, W, LEVELS, ALGO_BYTES_PER_PAIR, SIZE_NAME, METRIC
    H, W, LEVELS, ALGO_BYTES_PER_PAIR = SIZES[args.size]
    SIZE_NAME = args.size
    if args.size != "1080p" or args.k != 1:
        METRIC = f"{args.size} frame-pairs/sec (flow+grid+k-means{'' if args.k == 1 else ', k=%d' % args.k})"
        if args.size == "4k" and args.clip_frames == 129 and args.chunk == 33:
            args.clip_frames, args.chunk = 33, 9           # 25 MB frames: keep the resident and pinned clips small
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi-equivalent clock / throttle sampling through NVML during the timed region."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample_now(self):
        """one sample from the calling thread (the timed loop calls it while the GPU is still working through the
        enqueued steps, so a starved sampler thread cannot leave the record empty)"""
        if not self.nv:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for bit, name in self.REASONS.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _run(self):
        while not self._stop.is_set():
            self.sample_now()
            self._stop.wait(0.01)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        if self._t:
            self._stop.set()
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def bind_to_gpu_numa(index):
    """Pin this rank to the CPUs NVML reports as local to its GPU, BEFORE the pinned staging buffers are allocated: first
    touch then places them on the GPU's NUMA node and the copy-issuing thread runs next to it (with 8 ranks uploading
    ~27 GB/s each, remote-node staging is what the host memory system cannot sustain).  Returns the CPU count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [w * 64 + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        cpus = [c for c in cpus if c < (os.cpu_count() or 0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def cpu_reference_throughput(frames_np, workers, pairs_per_worker, n_clusters=1):
    from oracle import reference_chain
    return reference_chain.timed_throughput(frames_np, workers, pairs_per_worker, n_clusters, ROWS, COLS)


def run_reference(args):
    """--impl reference: the reference's own CPU path (cv2 + sklearn as the reference calls
    them, restated in oracle/reference_chain.py because /root/reference is not a package and
    does not travel) on all host cores, process-parallel over frame ranges."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from opticalflowclustering_b200.synthetic import synthetic_clip
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 64))
    ppw = 2 if args.k == 1 else 1
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    frames = synthetic_clip(min(args.clip_frames, 33), H, W, seed=0, device=dev).cpu().numpy()
    times = []
    for i in range(args.warmup + args.steps):
        v, wall = cpu_reference_throughput(frames, workers, ppw, args.k)
        if i >= args.warmup:
            times.append((v, wall))
    value = sum(workers * ppw for _ in times) / sum(w for _, w in times)
    ms = 1e3 * sum(w for _, w in times) / len(times)
    sample = f"{workers} processes x {ppw} consecutive {SIZE_NAME} pairs per step, cv2.setNumThreads(1), k={args.k}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"synthetic {SIZE_NAME} clip, Farneback levels={LEVELS} winsize=15 iters=3, 14x25 grid, k={args.k}",
                   "impl": "oracle/reference_chain.py: cv2 4.13 calcOpticalFlowFarneback + sklearn KMeans, as the reference calls them"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), file=_claim_stdout(), flush=True)


def kmeans_cosine_extras(dev, peak):
    """Secondary numbers for BASELINE.json configs[4] (k-means / cosine over 1M grid vectors): one Lloyd
    iteration (E-step + M-step kernels) and the row-cosine kernel, CUDA-event timed, against their
    algorithmic bytes (SURVEY.md §8d: N*D*sizeof(x) + 4N per iteration; N*D*sizeof(x) for cosine)."""
    import torch
    from opticalflowclustering_b200 import cosine as cosm
    from opticalflowclustering_b200 import kmeans as km
    out = {}
    g = torch.Generator().manual_seed(0)
    for name, (N, D, K, dt) in {"u8_d4_k8": (1_000_000, 4, 8, torch.uint8), "u8_d4_k8_64M": (64_000_000, 4, 8, torch.uint8),
                                "u8_d16_k8_16M": (16_000_000, 16, 8, torch.uint8), "u8_d350_k8": (200_000, 350, 8, torch.uint8),
                                "f32_d32_k16": (1_000_000, 32, 16, torch.float32)}.items():
        X = torch.randint(0, 180, (N, D), device=dev, dtype=torch.uint8).to(dt)          # generated on the device
        ctx = km._Ctx(dev)
        st = km.LloydState(ctx, X.unsqueeze(0).contiguous(), K)
        centres = X[:K].double().unsqueeze(0).contiguous()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fused = st.step_supported()          # uint8 rows with small [k][d]: E-step + exact sums in one pass over X
        for it in range(6):
            if it == 1:
                e0.record()
            if fused:
                st.step(None, centres, st.labels[it & 1], st.labels[(it & 1) ^ 1], st.n_changed, st.sums, st.counts)
            else:
                st.assign(None, centres, st.labels[0])
                st.sums_(None, st.labels[0], st.sums, st.counts, K)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        # algorithmic bytes (SURVEY 8d): X once + labels written (+ previous labels read by the fused step);
        # the two-kernel form reads X and the labels a second time
        nbytes = (N * D * X.element_size() + 2 * 4 * N) if fused else (2 * (N * D * X.element_size()) + 2 * 4 * N)
        out["kmeans_iter_" + name] = {"ms": ms, "rows_per_s": N / (ms / 1e3), "gb_s": nbytes / (ms / 1e3) / 1e9,
                                      "frac_of_hbm_peak": nbytes / (ms / 1e3) / 1e9 / peak, "fused_step": bool(fused), "rows": N}
    # dense corner of configs[4] (float32, d > 32): one Lloyd iteration on the tensor-core path -- 3xTF32 tcgen05
    # E-step (filter + float32 re-evaluation of near-ties) and the CSR M-step.  `tflops` counts the 2 N k D flop of the
    # distance GEMM once; the tensor cores execute three TF32 MMAs per product term (`tf32_tflops`), whose peak is
    # half the measured bf16 one.
    bf16_peak = None
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            bf16_peak = float(json.load(f).get("bf16_tflops"))
    except Exception:
        pass
    for name, (N, D, K) in {"f32_d64_k256": (1_000_000, 64, 256), "f32_d512_k256": (1_000_000, 512, 256),
                            "f32_d128_k1024": (1_000_000, 128, 1024), "u8_d352_k256": (1_000_000, 352, 256)}.items():
        gd = torch.Generator(device=dev).manual_seed(1)
        is_u8 = name.startswith("u8")          # uint8 hue vectors: float64 semantics, tensor-core filter + float64 re-evaluation
        cen = torch.rand((K, D), device=dev, generator=gd) * (200 if is_u8 else 8)
        X = cen[torch.randint(0, K, (N,), device=dev, generator=gd)] + (12 if is_u8 else 1) * torch.randn((N, D), device=dev, generator=gd)
        X = X.round().clamp(0, 255).to(torch.uint8) if is_u8 else X.float()
        ctx = km._Ctx(dev)
        st = km.LloydState(ctx, X.unsqueeze(0).contiguous(), K, ws_k=1)
        mean = X.double().mean(0).contiguous() if is_u8 else X.double().mean(0).float().double().contiguous()
        tc = km.TensorCoreSteps(st, mean)
        centres = (X[:K].double() - mean).unsqueeze(0).contiguous()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        t_assign = t_sums = 0.0
        for it in range(6):
            ev[0].record()
            tc.assign(centres, st.labels[0], prev=st.labels[1], n_changed=st.n_changed)
            ev[1].record()
            tc.sums_(st.labels[0], st.sums, st.counts)
            ev[2].record()
            torch.cuda.synchronize()
            if it >= 1:
                t_assign += ev[0].elapsed_time(ev[1]) / 5
                t_sums += ev[1].elapsed_time(ev[2]) / 5
        flop = 2.0 * N * K * D
        rec = {"ms_assign": t_assign, "ms_sums": t_sums, "rows_per_s": N / ((t_assign + t_sums) / 1e3),
               "tflops": flop / (t_assign / 1e3) / 1e12, "tf32_tflops": 3 * flop / (t_assign / 1e3) / 1e12,
               "rechecked_rows": int(tc.n_rechecked.item()),
               "sums_gb_s": ((N * D if is_u8 else 2 * N * D * 4) + 8 * N) / (t_sums / 1e3) / 1e9}
        if bf16_peak:
            rec["tf32_frac_of_peak"] = rec["tf32_tflops"] / (bf16_peak / 2)
        out["kmeans_iter_tc_" + name] = rec
        del tc, st, X
    # the reference's per-cell KMeans(n_clusters=8) over one 1080p frame (350 cells x 5852 px x 4 channels),
    # k-means++ seeding included, as ONE device-resident launch (kmeans.lloyd_cells)
    cells = torch.randint(0, 256, (350, 76 * 77, 4), generator=g).to(torch.uint8).to(dev)
    km.lloyd_cells(cells, 8, seed=1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _, _, _, n_it, _ = km.lloyd_cells(cells, 8, seed=1)
    e1.record()
    torch.cuda.synchronize()
    out["per_cell_kmeans_k8_1080p_frame"] = {"ms": e0.elapsed_time(e1), "mean_lloyd_iterations": float(n_it.float().mean().item()),
                                             "cells": 350, "rows_per_cell": 76 * 77}
    # host link: what a pinned 50 MB upload (one step's frames) achieves on this box
    hbuf = torch.empty(50 * 1024 * 1024, dtype=torch.uint8).pin_memory()
    dbuf = torch.empty_like(hbuf, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dbuf.copy_(hbuf, non_blocking=True)
    e0.record()
    for _ in range(4):
        dbuf.copy_(hbuf, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    out["h2d_pinned_gb_s"] = 4 * hbuf.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9
    X = torch.randint(0, 180, (1_000_000, 16), generator=g).to(torch.uint8).to(dev)
    q = torch.randint(0, 180, (16,), generator=g).double()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(6):
        if it == 1:
            e0.record()
        cosm.row_cosine(X, q)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    out["row_cosine_u8_1Mx16"] = {"ms": ms, "rows_per_s": 1e6 / (ms / 1e3), "gb_s": (16e6 + 8e6) / (ms / 1e3) / 1e9}
    # the rest of SURVEY 8(d)'s cosine sweep: a wide float32 row cosine (HBM-bound) and the sliding-window form of
    # findCosineDifferentVectors.py (n = 16 over m = 1 M; the call includes its 8-byte result read-back)
    Xw = torch.rand((1_000_000, 512), device=dev, dtype=torch.float32)
    qw = torch.rand(512, dtype=torch.float64)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(6):
        if it == 1:
            e0.record()
        cosm.row_cosine(Xw, qw)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    nb = 1e6 * 512 * 4 + 8e6
    out["row_cosine_f32_1Mx512"] = {"ms": ms, "rows_per_s": 1e6 / (ms / 1e3), "gb_s": nb / (ms / 1e3) / 1e9,
                                    "frac_of_hbm_peak": nb / (ms / 1e3) / 1e9 / peak}
    del Xw
    short = torch.randint(0, 180, (16,), generator=g).double().to(dev)
    long_ = torch.randint(0, 180, (1_000_000,), generator=g).double().to(dev)
    cosm.sliding_cosine(short, long_)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        cosm.sliding_cosine(short, long_)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    out["sliding_cosine_n16_m1M"] = {"ms": ms, "windows_per_s": (1e6 - 15) / (ms / 1e3), "gb_s": 16e6 / (ms / 1e3) / 1e9}
    return out


def _timed_steps(pipe, clip, F, steps, warmup):
    """device-resident steps over `clip` (walking through it), CUDA-event timed; returns ms per step"""
    import torch
    P, T = F - 1, int(clip.shape[0])
    starts = [(i * P) % (T - F + 1) for i in range(warmup + steps)]
    for i in range(warmup):
        pipe.run_chunk(clip[starts[i]:starts[i] + F])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(warmup, warmup + steps):
        pipe.run_chunk(clip[starts[i]:starts[i] + F])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _timed_steps_laned(lp, clip, F, steps, warmup):
    """the same over a LanedPipeline (chunks in flight on several streams)"""
    import torch
    P, T = F - 1, int(clip.shape[0])
    starts = [(i * P) % (T - F + 1) for i in range(warmup + steps)]
    for i in range(warmup):
        lp.submit(clip[starts[i]:starts[i] + F])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    main = torch.cuda.current_stream()
    e0.record()
    for i in range(warmup, warmup + steps):
        lp.submit(clip[starts[i]:starts[i] + F])
    for l in range(lp.n_lanes):
        main.wait_event(lp.done_event(l))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _kind_ms(pipe, clip, F, kinds, steps=3):
    """per-kernel-kind device time (ms per step) of `steps` steps, events around every launch"""
    import ctypes as C
    from opticalflowclustering_b200 import _lib
    L = _lib.lib()
    _lib.check(L.ofc_profile_begin())
    for _ in range(steps):
        pipe.run_chunk(clip[:F])
    ms_k, n_k = (C.c_float * 20)(), (C.c_int * 20)()
    _lib.check(L.ofc_profile_end(ms_k, n_k, 20))
    return {name: ms_k[k] / steps for k, name in kinds.items() if n_k[k]}


def other_sizes_leg(dev, peak):
    """BASELINE configs at 720p (levels=3) and 4K (levels=5), k = 1, device-resident, a few steps each"""
    import torch
    from opticalflowclustering_b200.pipeline import LanedPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    out = {}
    for name, F, T in (("720p", 33, 65), ("4k", 9, 17)):
        h, w, levels, algo = SIZES[name]
        clip = synthetic_clip(T, h, w, seed=7, device=dev)
        pipe = LanedPipeline(w, h, lanes=LANES, chunk_frames=F, rows=ROWS, cols=COLS, device=dev, levels=levels)
        ms = _timed_steps_laned(pipe, clip, F, 9, 3)
        out[name] = {"value": (F - 1) / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "pairs_per_step": F - 1, "levels": levels,
                     "lanes": LANES, "step_frac": algo * (F - 1) / (ms / 1e3) / 1e9 / peak, "algorithmic_bytes_per_pair": algo}
        del pipe, clip
        torch.cuda.empty_cache()
    return out


def k8_leg(dev, with_cpu):
    """`-c 8` (BASELINE configs[1]: 720p, k = 8; and the 1080p metric at k = 8): every cell of every pair gets its own
    KMeans(8) fit on the device (ofc_grid_kmeans_cells), straight from the visualisation"""
    import torch
    from opticalflowclustering_b200.pipeline import LanedPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    out = {}
    for name, F, T in (("720p", 33, 65), ("1080p", 17, 33)):
        h, w, levels, _ = SIZES[name]
        clip = synthetic_clip(T, h, w, seed=5, device=dev)
        rec = {}
        for k in (1, 8):
            lp = LanedPipeline(w, h, lanes=LANES, chunk_frames=F, rows=ROWS, cols=COLS, device=dev, levels=levels, n_clusters=k)
            ms = _timed_steps_laned(lp, clip, F, 9, 3)
            pipe = lp.lane(0)
            rec[f"k{k}"] = {"value": (F - 1) / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "pairs_per_step": F - 1, "lanes": LANES}
            if k == 8:
                kinds = _kind_ms(pipe, clip, F, {8: "kmeans_cells"})
                rec["k8"]["kmeans_ms_per_frame"] = kinds.get("kmeans_cells", 0.0) / (F - 1)
                rec["k8"]["mean_lloyd_iterations"] = float(pipe.km_n_iter.float().mean().item())
                rec["k8"]["max_lloyd_iterations"] = int(pipe.km_n_iter.max().item())
            del pipe, lp
        rec["k8_over_k1_time"] = rec["k8"]["ms_per_step"] / rec["k1"]["ms_per_step"]
        if with_cpu and name == "720p":
            cores = os.cpu_count() or 1
            workers = max(1, min(cores, 64))
            v, wall = cpu_reference_throughput(clip[:9].cpu().numpy(), workers, 1, 8)
            rec["cpu_reference_k8"] = {"value": v, "unit": UNIT, "cores": workers, "kind": "port",
                                       "sample": f"{workers} processes x 1 pair of the same 720p clip, cv2 Farneback + grid loop + "
                                                 f"sklearn KMeans(8) per cell, {wall:.1f} s wall"}
        out[name] = rec
        del clip
        torch.cuda.empty_cache()
    return out


def dropin_leg(host_clip):
    """The literal drop-in calls, numpy in / numpy out, one pair per call (what a user of the reference types):
    ComputeOpticalFLow(first).compute(frame) (computeOpticalFlowModule.py:6-36) and the cv2-signature
    calc_optical_flow_farneback(prev, next, None, 0.5, 3, 15, 3, 5, 1.2, 0).  Wall clock per call, host copies included."""
    import numpy as np
    import torch
    from opticalflowclustering_b200.computeOpticalFlowModule import ComputeOpticalFLow
    from opticalflowclustering_b200.flow import calc_optical_flow_farneback
    from oracle import reference_chain
    frames = host_clip[:8].numpy()
    cf = ComputeOpticalFLow(frames[0])
    cf.compute(frames[1])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for f in frames[2:8]:
        out = cf.compute(f)
    t_compute = (time.perf_counter() - t0) / 6
    gray = np.stack([reference_chain._cv2().cvtColor(f, reference_chain._cv2().COLOR_BGR2GRAY) for f in frames[:4]])
    calc_optical_flow_farneback(gray[0], gray[1], None, 0.5, 3, 15, 3, 5, 1.2, 0)
    t0 = time.perf_counter()
    for i in range(1, 3):
        fl = calc_optical_flow_farneback(gray[i], gray[i + 1], None, 0.5, 3, 15, 3, 5, 1.2, 0)
    t_flow = (time.perf_counter() - t0) / 2
    ref = reference_chain.FlowState(frames[0])
    t0 = time.perf_counter()
    ref.compute(frames[1])
    t_cv2 = time.perf_counter() - t0
    return {"ComputeOpticalFLow.compute_ms_per_call": 1e3 * t_compute, "calc_optical_flow_farneback_ms_per_call": 1e3 * t_flow,
            "reference_compute_ms_per_call_cv2": 1e3 * t_cv2, "frame": f"{W}x{H} BGR uint8 numpy in, numpy out",
            "out_shape": list(out.shape), "flow_shape": list(fl.shape)}


def dist_kmeans_leg(dev, world, rank):
    """The one collective of the path (north_star: NCCL all-reduce of k-means centroid sums and counts per iteration):
    WHOLE Lloyd fits over vectors sharded by row across the ranks (kmeans.lloyd(group=...)), timed on the device
    (max over ranks).  Total rows are fixed, so across N this leg is strong scaling; `rows_iter_per_s` = rows x
    iterations / fit time."""
    import torch
    import torch.distributed as dist
    from opticalflowclustering_b200 import kmeans as km
    from opticalflowclustering_b200.sharding import shard_range
    out = {}
    cases = {"u8_8Mx4_k8": (8_000_000, 4, 8, True), "u8_64Mx4_k8": (64_000_000, 4, 8, True), "f32_1Mx128_k1024": (1_000_000, 128, 1024, False)}
    for name, (N, D, K, is_u8) in cases.items():
        gd = torch.Generator(device=dev).manual_seed(11)
        cen = torch.rand((K, D), device=dev, generator=gd) * (200 if is_u8 else 8) + (25 if is_u8 else 0)
        lo, hi = shard_range(N, rank, world)
        # every rank draws the whole label / noise stream in blocks and keeps its rows: identical data for every N
        rows = []
        init = None
        blk = 4_000_000 if is_u8 else 250_000
        for s0 in range(0, N, blk):
            nb = min(blk, N - s0)
            lab = torch.randint(0, K, (nb,), device=dev, generator=gd)
            x = cen[lab] + (12 if is_u8 else 1) * torch.randn((nb, D), device=dev, generator=gd)
            if s0 == 0:                          # initial centres: the first K rows of the whole set (same on every rank)
                init = (x[:K].round().clamp(0, 255) if is_u8 else x[:K].float()).double()
            a, b = max(lo, s0), min(hi, s0 + nb)
            if a < b:
                x = x[a - s0:b - s0]
                rows.append(x.round().clamp(0, 255).to(torch.uint8) if is_u8 else x.float())
            del lab, x
        X = torch.cat(rows).contiguous()
        del rows
        group = dist.group.WORLD if world > 1 else None
        km.lloyd(X, init, group=group)           # warm-up fit
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        labels, centres, inertia, n_iter = km.lloyd(X, init, group=group)
        e1.record()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        it = int(n_iter)
        rec = {"rows": N, "d": D, "k": K, "n_iter": it, "fit_ms": ms, "host_wall_ms": 1e3 * wall, "ms_per_iteration": ms / max(it, 1),
               "rows_iter_per_s": N * it / (ms / 1e3), "inertia": float(inertia)}
        if world > 1:
            # which exchange the fit above used, and the same fit with the library collectives (NCCL all-reduce x 2 +
            # all-gather per iteration) for comparison
            from opticalflowclustering_b200.peer import PeerExchange
            peer = any(v not in (None, False) for v in PeerExchange._cache.values())
            rec["exchange"] = "one peer-memory kernel per iteration over NVLink (csrc/peer_exchange.cu)" if peer else "NCCL collectives"
            if peer:
                os.environ["OFC_KMEANS_PEER"] = "0"
                km.lloyd(X, init, group=group)
                dist.barrier()
                torch.cuda.synchronize()
                e0.record()
                _, c_n, _, it_n = km.lloyd(X, init, group=group)
                e1.record()
                torch.cuda.synchronize()
                os.environ.pop("OFC_KMEANS_PEER")
                tn = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
                dist.all_reduce(tn, op=dist.ReduceOp.MAX)
                rec["fit_ms_nccl"] = float(tn.item())
                rec["same_result_as_nccl"] = bool(torch.equal(c_n, centres) and int(it_n) == it)
        if world == 1:
            # same fit with events around every kernel: how much of the fit is kernel time (host-free loop)
            import ctypes as C
            from opticalflowclustering_b200 import _lib
            L = _lib.lib()
            os.environ["OFC_KMEANS_GRAPH"] = "0"          # per-kernel events cannot be recorded inside a graph capture
            _lib.check(L.ofc_profile_begin())
            km.lloyd(X, init)
            ms_k, n_k = (C.c_float * 20)(), (C.c_int * 20)()
            _lib.check(L.ofc_profile_end(ms_k, n_k, 20))
            os.environ.pop("OFC_KMEANS_GRAPH")
            rec["sum_of_kernel_ms"] = float(sum(ms_k[i] for i in range(20)))
            rec["kernel_launches"] = int(sum(n_k[i] for i in range(20)))
            rec["fit_over_kernel_time"] = ms / max(rec["sum_of_kernel_ms"], 1e-9)
        out[name] = rec
        del X, labels
        torch.cuda.empty_cache()
    return out


def h2d_concurrent_leg(dev, world):
    """Host-link ceiling of the end-to-end number: pinned 50 MB uploads (one step's frames) on EVERY rank at the same
    time -- what each rank's copy engine gets when all N share the host's memory system / PCIe roots."""
    import torch
    import torch.distributed as dist
    hbuf = torch.empty(50 * 1024 * 1024, dtype=torch.uint8).pin_memory()
    dbuf = torch.empty_like(hbuf, device=dev)
    dbuf.copy_(hbuf, non_blocking=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(8):
        dbuf.copy_(hbuf, non_blocking=True)
    e1.record()
    torch.cuda.synchronize()
    gbs = torch.tensor([8 * hbuf.numel() / (e0.elapsed_time(e1) / 1e3) / 1e9], dtype=torch.float64, device=dev)
    lo, tot = gbs.clone(), gbs.clone()
    if world > 1:
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    return {"per_rank_min_gb_s": float(lo.item()), "all_ranks_gb_s": float(tot.item()), "ranks": world}


DUMP_SAMPLE_PX = 1 << 20           # --dump-outputs: (pair, pixel) positions kept of the per-pixel outputs
DUMP_SAMPLE_SEED = 0


def dump_sample_index(n_px):
    """the positions (flat index over pairs x rows x columns, ascending) at which --dump-outputs keeps the per-pixel
    outputs: every position when there are at most DUMP_SAMPLE_PX, else DUMP_SAMPLE_PX drawn from a fixed seed"""
    import torch
    if n_px <= DUMP_SAMPLE_PX:
        return torch.arange(n_px)
    g = torch.Generator().manual_seed(DUMP_SAMPLE_SEED)
    return torch.randint(n_px, (DUMP_SAMPLE_PX,), generator=g).sort().values


def dump_outputs(out_dir, pipe, P):
    """--dump-outputs: what the last timed step computed, i.e. what a caller of LanedPipeline.submit reads from the lane
    that ran it, as out_dir/<name>.npy.  Per-cell rows and magnitudes are written whole; the flow and the visualisation
    (0.7 GB at 1080p) at the positions of dump_sample_index.  Integer outputs are widened to float32 (exact), the mean
    magnitude stays float64 (the host division of ClipPipeline.process_clip).  At most about 20 MB at any size."""
    import numpy as np
    idx = dump_sample_index(P * pipe.H * pipe.W).to(pipe.device)
    out = {"avg_hue": pipe.avg_hue[:P], "km_hue": pipe.km_hue[:P], "km_centre": pipe.km_centre[:P], "avg_bgr": pipe.avg_bgr[:P],
           "mean_magnitude": pipe.mag_sum[:P].cpu() / float(pipe.H * pipe.W),
           "flow_sample": pipe.flow[:P].reshape(-1, 2)[idx], "viz_sample": pipe.viz[:P].reshape(-1, 3)[idx]}
    if pipe.km_n_iter is not None:
        out["km_n_iter"] = pipe.km_n_iter[:P]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in out.items():
        a = t.cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float32))
    return sorted(out)


_JSON_OUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL writes its version banner to stdout
    under torchrun), so file descriptor 1 is pointed at stderr for the rest of the process and the JSON line goes to
    a private duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _JSON_OUT


def main():
    args = parse()
    _claim_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from opticalflowclustering_b200 import _lib
    from opticalflowclustering_b200.pipeline import ClipPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    import ctypes as C

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = None
    if world > 1:
        if os.environ.get("OFC_BENCH_NUMA", "1") != "0":
            numa_cpus = bind_to_gpu_numa(local)
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    F = args.chunk
    P = F - 1
    T = max(args.clip_frames, F)
    clip = synthetic_clip(T, H, W, seed=rank, device=dev)              # resident in HBM, > L2
    pipe = ClipPipeline(W, H, chunk_frames=F, rows=ROWS, cols=COLS, device=dev, levels=LEVELS, n_clusters=args.k)
    # the timed loops deal their chunks over `lanes` pipelines on their own streams (one chunk's gaps and tails are
    # filled by another's CTAs); `pipe` alone serves the per-kernel breakdown, which wants one chain of kernels
    from opticalflowclustering_b200.pipeline import LanedPipeline
    global LANES
    n_lanes = LANES = max(1, args.lanes)
    lp = LanedPipeline(W, H, lanes=n_lanes, chunk_frames=F, rows=ROWS, cols=COLS, device=dev, levels=LEVELS, n_clusters=args.k)
    starts = [(i * P) % (T - F + 1) for i in range(args.warmup + args.steps)]
    main_stream = torch.cuda.current_stream()

    # ---- value: inputs resident in HBM --------------------------------------
    for _ in range(n_lanes):                                   # every lane's buffers touched once, whatever --warmup is
        lp.submit(clip[0:F])
    for i in range(args.warmup):
        lp.submit(clip[starts[i]:starts[i] + F])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # profiler range = the timed steps: `ncu --profile-from-start off` then lists exactly these launches (no-ops otherwise)
    torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    for i in range(args.warmup, args.warmup + args.steps):
        last_lane, _ = lp.submit(clip[starts[i]:starts[i] + F])   # each lane's stream waits for e0 through the current stream
    for l in range(n_lanes):
        main_stream.wait_event(lp.done_event(l))
    e1.record()
    torch.cuda.cudart().cudaProfilerStop()
    sampler.sample_now()        # after the last enqueue: the GPU is still working, and a slow NVML call cannot stall the timed steps
    barrier()
    clocks = sampler.stop()
    dumped = None
    if args.dump_outputs and rank == 0:          # before the e2e loop below reuses the lanes
        dumped = {"dir": os.path.abspath(args.dump_outputs), "arrays": dump_outputs(args.dump_outputs, lp.lane(last_lane), P),
                  "step": args.warmup + args.steps - 1, "frames": [starts[-1], starts[-1] + F]}
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * args.steps * P / (ms_total / 1e3)

    # ---- per-kernel breakdown (same steps again, events around every launch) --
    L = _lib.lib()
    _lib.check(L.ofc_profile_begin())
    prof_steps = min(args.steps, 5)
    for i in range(args.warmup, args.warmup + prof_steps):
        pipe.run_chunk(clip[starts[i]:starts[i] + F])
    ms_k = (C.c_float * 20)()
    n_k = (C.c_int * 20)()
    _lib.check(L.ofc_profile_end(ms_k, n_k, 20))
    names = {0: "bgr2gray", 1: "prefilter", 2: "polyexp", 3: "minmax_init", 4: "flow_encode_grid" if pipe.fuse_grid else "flow_encode",
             5: "grid_cells", 8: "kmeans_cells", 10: "flow_upsample"}
    names.update({12 + l: f"flow_iter_L{l}" for l in range(8)})
    kernels = {names[k]: {"ms_per_step": ms_k[k] / prof_steps, "launches_per_step": n_k[k] // prof_steps}
               for k in names if n_k[k]}
    launches_per_step = sum(v["launches_per_step"] for v in kernels.values())
    peak, peak_kind = measured_peak()
    it0 = kernels.get("flow_iter_L0")
    roofline = None
    if it0:
        per_launch_ms = it0["ms_per_step"] / it0["launches_per_step"]
        algo = ITER_BYTES_PER_PX * H * W * P
        achieved = algo / (per_launch_ms / 1e3) / 1e9
        # DRAM bytes of this launch are not measurable inside the run: the figure comes from the committed ncu capture of
        # the same launch (profiles/r02_flow_iter_traffic.json: dram__bytes_read.sum + dram__bytes_write.sum, --set full),
        # scaled by the pairs per launch, and is labelled as such
        traffic, traffic_source = None, None
        try:
            if SIZE_NAME != "1080p":
                raise KeyError("the ncu capture is of the 1080p launch")
            with open(os.path.join(ROOT, "profiles", "r02_flow_iter_traffic.json")) as f:
                tj = json.load(f)
            traffic = tj["dram_bytes_per_launch"] * P / float(tj.get("pairs_per_launch", P))
            traffic_source = "ncu capture committed as profiles/r02_flow_iter_traffic.json (not measured in this run), scaled by pairs per launch"
        except Exception:
            pass
        total_ms = sum(v["ms_per_step"] for v in kernels.values())
        # the fused kernel never writes or re-reads the update matrices M that SURVEY 8(d)'s 96 B/px charges: what it must
        # move is R of both frames (2 x 20 B), the flow in (8 B) and the flow out (8 B) = 56 B/px
        fused = FUSED_ITER_BYTES_PER_PX * H * W * P / (per_launch_ms / 1e3) / 1e9
        roofline = {"bound": "hbm", "kernel": f"flow_iter_tmem_kernel<R=7,TW=240> @{W}x{H} (update-matrices + 15x15 box + 2x2 solve fused, "
                              "persistent strip walk, ring in TMEM, cp.async tap landing, float32 error-free solve, pair-aligned grid for L2 "
                              "sharing of the expansions; 3 launches per step)",
                    "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_source": traffic_source,
                    "algorithmic_bytes_per_launch": algo, "ms_per_launch": per_launch_ms,
                    "achieved_fused_model": fused, "frac_fused": fused / peak,
                    "dram_frac_of_peak": (traffic / (per_launch_ms / 1e3) / 1e9 / peak) if traffic else None,
                    "note": "`frac` follows SURVEY 8(d)'s unfused dataflow (96 B/px incl. writing and re-reading M); the kernel keeps M "
                            "on the SM, so `frac_fused` (56 B/px: R0 + R1 + flow in + flow out) and `dram_frac_of_peak` (measured DRAM "
                            "bytes / time) say how far from the HBM bound it really runs: it is issue / latency bound",
                    "share_of_step": it0["ms_per_step"] / total_ms,
                    "step_achieved_gbs": ALGO_BYTES_PER_PAIR * P / (ms_total / args.steps / 1e3) / 1e9,
                    "step_frac": ALGO_BYTES_PER_PAIR * P / (ms_total / args.steps / 1e3) / 1e9 / peak}

    # ---- e2e: host frames in, hue rows out ----------------------------------
    # The public call a user makes: ClipPipeline.run_chunk(new frames, carry=True) -- every step uploads
    # the P new frames of its chunk from pinned host memory (the frame shared with the previous chunk
    # stays on the device as prev_gray, like the reference's ComputeOpticalFLow state) and reads back
    # the hue rows and magnitudes.
    # walk the clip forwards then backwards so that consecutive chunks are always consecutive frames
    host_clip = clip.cpu()
    host = torch.cat([host_clip[1:], host_clip[:-1].flip(0)]).pin_memory()
    res_avg = torch.empty((P, ROWS * COLS), dtype=torch.uint8).pin_memory()
    res_km = torch.empty((P, ROWS * COLS), dtype=torch.uint8).pin_memory()
    res_mag = torch.empty(P, dtype=torch.float64).pin_memory()
    NBUF = n_lanes + 2   # a staging buffer is busy until its chunk has run; `lanes` chunks are in flight and one upload ahead
    NRES = n_lanes + 1   # result snapshots on the device / pinned read-back buffers
    stage = [torch.empty((P, H, W, 3), dtype=torch.uint8, device=dev) for _ in range(NBUF)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(NBUF)]
    freed = [torch.cuda.Event() for _ in range(NBUF)]
    n_chunks = host.shape[0] // P               # consecutive P-frame chunks of the there-and-back walk

    d2h_stream = torch.cuda.Stream(device=dev)
    done_ev = [torch.cuda.Event() for _ in range(NRES)]
    read_ev = [torch.cuda.Event() for _ in range(NRES)]
    no_upload = os.environ.get("OFC_E2E_NO_UPLOAD", "0") == "1"        # diagnostic only: what the uploads cost the kernels
    res_pin = [(torch.empty_like(res_avg).pin_memory(), torch.empty_like(res_km).pin_memory(), torch.empty_like(res_mag).pin_memory())
               for _ in range(NRES)]
    dev_res = [(torch.empty((P, ROWS * COLS), dtype=torch.uint8, device=dev), torch.empty((P, ROWS * COLS), dtype=torch.uint8, device=dev),
                torch.empty(P, dtype=torch.float64, device=dev)) for _ in range(NRES)]

    def e2e_loop(lo, hi):
        """every step: upload the P new frames of the chunk from pinned host memory (copy stream), run the chunk on the
        next lane (carry: the frame shared with the previous chunk stays on the device), snapshot its hue rows and
        magnitudes on the lane's stream and read the snapshot back to pinned host memory on a third stream"""
        main = torch.cuda.current_stream()
        for b in range(NBUF):
            freed[b].record(main)
        for j in range(NRES):
            read_ev[j].record(d2h_stream)

        def upload(i):
            b = i % NBUF
            c = i % n_chunks
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[b])
                if not no_upload:
                    stage[b].copy_(host[c * P:(c + 1) * P], non_blocking=True)
                ready[b].record(copy_stream)
        # frame 0 of the clip seeds prev_gray (outside the steady state, like the reference's first cap.read())
        lp.submit(clip[0:2])
        upload(lo)
        for i in range(lo, hi):
            b = i % NBUF
            if i + 1 < hi:
                upload(i + 1)
            l, _ = lp.submit(stage[b], carry=True, wait=ready[b])
            s, lane = lp.lane_stream(l), lp.lane(l)
            freed[b].record(s)
            # snapshot the step's rows on the device (the lane's buffers are rewritten by its next chunk), then read the
            # snapshot back beside the following kernels
            j = i % NRES
            with torch.cuda.stream(s):
                s.wait_event(read_ev[j])
                dev_res[j][0].copy_(lane.avg_hue[:P], non_blocking=True)
                dev_res[j][1].copy_(lane.km_hue[:P], non_blocking=True)
                dev_res[j][2].copy_(lane.mag_sum[:P], non_blocking=True)
                done_ev[j].record(s)
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(done_ev[j])
                for k in range(3):
                    res_pin[j][k].copy_(dev_res[j][k], non_blocking=True)
                read_ev[j].record(d2h_stream)
        for l in range(n_lanes):
            main.wait_event(lp.done_event(l))
        main.wait_stream(d2h_stream)

    e2e_loop(0, args.warmup)
    barrier()
    t0 = time.perf_counter()
    e0.record()
    e2e_loop(args.warmup, args.warmup + args.steps)
    e1.record()
    barrier()
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * args.steps * P / (float(t.item()) / 1e3)
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": P * H * W * 3,
           "d2h_bytes_per_step": P * (2 * ROWS * COLS + 8),
           "api": f"LanedPipeline.submit(new frames, carry=True) on pinned host frames, {n_lanes} lanes, staged upload on a copy "
                  "stream, result rows read back to pinned host memory every step"}

    extras = None
    if not args.no_extras:
        dk = dist_kmeans_leg(dev, world, rank)                 # every rank takes part
        hl = h2d_concurrent_leg(dev, world)
        if rank == 0:
            extras = kmeans_cosine_extras(dev, peak)
            extras["dist_kmeans"] = dk
            extras["h2d_pinned_all_ranks"] = hl
            if SIZE_NAME == "1080p" and args.k == 1:
                extras["sizes"] = other_sizes_leg(dev, peak)
                extras["k8"] = k8_leg(dev, with_cpu=(world == 1 and not args.no_cpu_baseline))
                extras["dropin_latency"] = dropin_leg(host_clip)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and LEVELS == 3:
        cores = os.cpu_count() or 1
        workers = max(1, min(cores, 64))
        frames_np = host_clip[:min(T, 33)].numpy()
        ppw = 2 if args.k == 1 else 1
        v, wall = cpu_reference_throughput(frames_np, workers, ppw, args.k)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": workers, "kind": "port",
                        "sample": f"{workers} processes x {ppw} consecutive {SIZE_NAME} pairs of the same clip "
                                  f"(cv2 Farneback + grid loop + sklearn KMeans({args.k}) per cell), {wall:.1f} s wall"}

    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"synthetic {SIZE_NAME} clip, Farneback levels={LEVELS} winsize=15 iters=3, 14x25 grid, k={args.k}",
                       "frames_per_step": F, "pairs_per_step": P, "clip_frames": T, "rank_cpu_affinity": numa_cpus,
                       "lanes": n_lanes,
                       "l2": f"steps walk a {T}-frame clip ({T * H * W * 3 / 1e6:.0f} MB > L2); intermediates "
                             f"({pipe.plan.workspace_bytes / 1e6:.0f} MB workspace) are rewritten every step"},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline, "cpu_baseline": cpu_baseline, "kernels": kernels, "extras": extras,
            **({"dump_outputs": dumped} if dumped else {}),
        }), file=_claim_stdout(), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
