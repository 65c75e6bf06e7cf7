"""Time MiniBatchKMeans on the GPU: the centre update on both paths of its streaming kernel with CUDA events, partial_fit per 1080p frame end to end and by part, fit on all pixels against fit on the unique colours with
their counts, and scikit-learn on the host cores for the same calls.  Prints the card and its power limit and writes
one JSON file.

    python tools/minibatch_bench.py --out profiles/minibatch_bench.json
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opticalflowclustering_b200 import _lib, kmeans as km                     # noqa: E402
from opticalflowclustering_b200.minibatch import MiniBatchKMeans              # noqa: E402
from opticalflowclustering_b200.synthetic import synthetic_clip               # noqa: E402

DT = {torch.uint8: 0, torch.float32: 1, torch.float64: 2}


def _vp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def host_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / reps


def update_paths(rows_list, reps):
    """ofc_minibatch_update[_weighted] per batch size, k and input kind (uint8 unit / integer weights take the
    exact-integer path, real weights and non-integer float32 rows the sequential path)"""
    lib, out = _lib.lib(), []
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(0)
    for n in rows_list:
        for k in (8, 64):
            for kind in ("u8_unit", "u8_int", "u8_real", "f32_unit"):
                dt = torch.float32 if kind.startswith("f32") else torch.uint8
                X = torch.randint(0, 256, (n, 3), generator=g, device="cuda").to(dt)
                if dt == torch.float32:
                    X += torch.rand((n, 3), generator=g, device="cuda")
                labels = torch.randint(0, k, (n,), generator=g, device="cuda", dtype=torch.int32)
                w = None
                if kind == "u8_int":
                    w = torch.randint(0, 5, (n,), generator=g, device="cuda").to(torch.float64)
                elif kind == "u8_real":
                    w = torch.rand((n,), generator=g, device="cuda", dtype=torch.float64) * 3
                c_old = torch.rand((k, 3), generator=g, device="cuda", dtype=torch.float64) * 255
                c_new = torch.empty_like(c_old)
                ws0 = torch.full((k,), 1000.0, device="cuda", dtype=torch.float64)
                ws = ws0.clone()
                head = (_vp(X), DT[dt], n, 3, k, _vp(labels))
                tail = (_vp(c_old), _vp(c_new), _vp(ws), stream)

                def run():
                    ws.copy_(ws0)
                    _lib.check(lib.ofc_minibatch_update(*head, *tail) if w is None
                               else lib.ofc_minibatch_update_weighted(*head, _vp(w), *tail))
                reset = events_ms(lambda: ws.copy_(ws0), reps)
                ms = events_ms(run, reps) - reset
                out.append(dict(rows=n, k=k, kind=kind, path="sequential" if kind in ("u8_real", "f32_unit") else "integer",
                                ms=round(ms, 5)))
                print(json.dumps(out[-1]), flush=True)
    return out


def partial_fit_1080p(frames, reps_frames):
    """partial_fit per 1080p uint8 frame (k = 8) end to end, and its parts on the same frame: E-step, update, count
    read-back, label pass (the reassignment's host permutation is inside end to end when it fires)"""
    clip = synthetic_clip(frames, 1080, 1920, seed=1).cuda()
    px = [f.reshape(-1, 3).contiguous() for f in clip]
    m = MiniBatchKMeans(n_clusters=8, random_state=0)
    m.partial_fit(px[0])
    torch.cuda.synchronize()
    t = []
    for i in range(reps_frames):
        s = time.perf_counter()
        m.partial_fit(px[(i + 1) % frames])
        torch.cuda.synchronize()
        t.append((time.perf_counter() - s) * 1e3)
    ctx = km._Ctx(px[0].device)
    Xb = px[0].unsqueeze(0)
    st = km.LloydState(ctx, Xb, 8)
    cen = m._centres_t.clone()
    c_new = torch.empty_like(cen)
    ws = m._counts_t.clone()
    lib = ctx.lib
    e = events_ms(lambda: st.assign(None, cen.view(1, 8, 3), st.labels[0]), 20)
    u = events_ms(lambda: ctx.check(lib.ofc_minibatch_update(_vp(Xb), 0, Xb.shape[1], 3, 8, _vp(st.labels[0]), _vp(cen),
                                                             _vp(c_new), _vp(ws), ctx.stream())), 20)
    r = host_ms(lambda: ws.cpu(), 50)
    lp = events_ms(lambda: st.assign(None, cen.view(1, 8, 3), st.labels[1], inertia=st.inertia), 20)
    return dict(frame="1080p uint8", k=8, end_to_end_ms_median=round(float(np.median(t)), 3),
                end_to_end_ms_all=[round(x, 3) for x in t], e_step_ms=round(e, 4), update_ms=round(u, 4),
                readback_ms=round(r, 4), label_pass_ms=round(lp, 4))


def fit_unique(reps):
    px = synthetic_clip(1, 1080, 1920, seed=2)[0].reshape(-1, 3).numpy()
    uniq, counts = np.unique(px, axis=0, return_counts=True)
    Xa, Xu = torch.from_numpy(px).cuda(), torch.from_numpy(uniq).cuda()
    wu = counts.astype(np.float64)
    all_ms = host_ms(lambda: MiniBatchKMeans(n_clusters=8, random_state=0).fit(Xa), reps)
    uniq_ms = host_ms(lambda: MiniBatchKMeans(n_clusters=8, random_state=0).fit(Xu, sample_weight=wu), reps)
    return dict(pixels=int(px.shape[0]), unique_colours=int(uniq.shape[0]), fit_all_pixels_ms=round(all_ms, 3),
                fit_unique_with_counts_ms=round(uniq_ms, 3))


def sklearn_baseline():
    try:
        from sklearn.cluster import MiniBatchKMeans as SK
    except ImportError:
        return "not measured (scikit-learn not installed)"
    clip = synthetic_clip(3, 1080, 1920, seed=1)
    px = [f.reshape(-1, 3).numpy() for f in clip]
    m = SK(n_clusters=8, random_state=0).partial_fit(px[0])
    t = []
    for i in range(4):
        s = time.perf_counter()
        m.partial_fit(px[(i + 1) % 3])
        t.append((time.perf_counter() - s) * 1e3)
    p0 = synthetic_clip(1, 1080, 1920, seed=2)[0].reshape(-1, 3).numpy()
    uniq, counts = np.unique(p0, axis=0, return_counts=True)
    s = time.perf_counter()
    SK(n_clusters=8, random_state=0).fit(p0)
    fa = (time.perf_counter() - s) * 1e3
    s = time.perf_counter()
    SK(n_clusters=8, random_state=0).fit(uniq, sample_weight=counts.astype(np.float64))
    fu = (time.perf_counter() - s) * 1e3
    return dict(host_cpus=os.cpu_count(), partial_fit_1080p_ms_median=round(float(np.median(t)), 2),
                fit_all_pixels_ms=round(fa, 2), fit_unique_with_counts_ms=round(fu, 2))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/minibatch_bench.json")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("a CUDA device is required")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0]
    print("card:", card, flush=True)
    res = dict(card=card, update=update_paths([1024, 4096, 16384, 51200, 2073600], args.reps))
    res["partial_fit_1080p"] = partial_fit_1080p(3, 10)
    print(json.dumps(res["partial_fit_1080p"]), flush=True)
    res["fit_unique"] = fit_unique(3)
    print(json.dumps(res["fit_unique"]), flush=True)
    res["sklearn_host"] = sklearn_baseline()
    print(json.dumps(res["sklearn_host"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
