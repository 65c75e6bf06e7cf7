"""Batched clip pipeline: the hot path end to end on one GPU.

    BGR frames -> gray -> Farneback flow -> HSV visualisation -> 14x25 grid
    -> per-cell mean hue + per-cell k-means(1) hue

i.e. what the reference's KmeanGrids.py main loop (:180-231, :376-399) does
frame by frame in Python, run for a chunk of consecutive frames per launch
sequence.  Frame pairs are independent given both frames, so a chunk of n
frames yields n-1 pairs in one set of kernel launches (grid.z = pair); the
pre-filter and polynomial expansion of every frame are computed once and used
by both pairs it belongs to.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from .flow import FarnebackPlan, _ptr, _stream_ptr


class ClipPipeline:
    def __init__(self, width: int, height: int, chunk_frames: int = 9, rows: int = 14, cols: int = 25,
                 draw_lines: bool = True, threshold: int = 30, device=None, keep_viz: bool = False,
                 pyr_scale: float = 0.5, levels: int = 3, winsize: int = 15, iterations: int = 3,
                 poly_n: int = 5, poly_sigma: float = 1.2, n_clusters: int = 1, kmeans_seed: int = 0,
                 kmeans_max_iter: int = 300, kmeans_tol: float = 1e-4):
        """``n_clusters``: the reference's ``-c`` (KmeanGrids.py:248-250).  1 (every documented command): the per-cell
        k-means centre is the cell mean and rides the grid pass.  k > 1: every cell of every pair gets its own
        ``KMeans(n_clusters=k)`` fit (k-means++ from ``kmeans_seed`` -- the reference leaves ``random_state`` unset)
        on the device, straight from the visualisation (``ofc_grid_kmeans_cells``); ``km_centre`` / ``km_hue`` then
        hold the largest cluster's rounded centre and its hue (KmeanGrids.py:299-339), ``km_n_iter`` the Lloyd
        iterations per cell."""
        self.W, self.H, self.F = int(width), int(height), int(chunk_frames)
        if self.F < 2:
            raise ValueError("chunk_frames must be >= 2")
        self.rows, self.cols = int(rows), int(cols)
        self.cells = self.rows * self.cols
        self.draw_lines, self.threshold = int(bool(draw_lines)), int(threshold)
        self.plan = FarnebackPlan(width, height, self.F, pyr_scale, levels, winsize, iterations, poly_n, poly_sigma,
                                  0, device=device)
        dev = self.device = self.plan.device
        P = self.F - 1
        self.gray = torch.empty((self.F, self.H, self.W), dtype=torch.uint8, device=dev)
        self.flow = torch.empty((P, self.H, self.W, 2), dtype=torch.float32, device=dev)
        self.minmax = torch.empty((P, 2), dtype=torch.int32, device=dev)
        self.viz = torch.empty((P, self.H, self.W, 3), dtype=torch.uint8, device=dev)
        self.mag_sum = torch.empty(P, dtype=torch.float64, device=dev)
        self.avg_bgr = torch.empty((P, self.cells, 3), dtype=torch.uint8, device=dev)
        self.avg_hue = torch.empty((P, self.cells), dtype=torch.uint8, device=dev)
        self.km_centre = torch.empty((P, self.cells, 4), dtype=torch.uint8, device=dev)
        self.km_hue = torch.empty((P, self.cells), dtype=torch.uint8, device=dev)
        self.keep_viz = keep_viz
        self.fuse_grid = True            # False runs the visualisation and the grid pass as two kernels (same bytes)
        self.n_clusters = int(n_clusters)
        if self.n_clusters < 1:
            raise ValueError("n_clusters must be >= 1")
        self.kmeans_seed, self.kmeans_max_iter, self.kmeans_tol = int(kmeans_seed), int(kmeans_max_iter), float(kmeans_tol)
        self.km_n_iter = None
        self._km_ws = None
        self._pairs_done = 0             # pairs processed so far: the k-means++ stream is indexed by absolute pair number
        if self.n_clusters > 1:
            L = _lib.lib()
            self.km_n_iter = torch.empty((P, self.cells), dtype=torch.int32, device=dev)
            nb = int(L.ofc_grid_kmeans_cells_workspace_bytes(P, self.H, self.W, self.rows, self.cols, self.n_clusters))
            self._km_ws = torch.empty(max(nb, 8), dtype=torch.uint8, device=dev)
        self._last_gray_index = None     # where the last processed frame's gray image sits in self.gray
        self._gray_event = None          # LanedPipeline: recorded once the chunk's gray frames exist (another lane carries the last)
        #: kernels launched by one full-chunk call of :meth:`run_chunk`
        self.launches_per_chunk = 1 + 2 * self.plan.num_levels + 1 + self.plan.num_levels * iterations + 1 + 1

    def run_chunk(self, frames: torch.Tensor, n_frames: int | None = None, carry: bool = False):
        """frames: CUDA uint8 [n,H,W,3] (n <= chunk_frames).  Results stay in the
        pipeline's buffers (``avg_hue``, ``km_hue``, ``km_centre``, ``mag_sum``, ``viz``,
        ``flow``) for pairs 0..n-2; returns n-1.

        ``carry=True``: ``frames`` are the m NEW frames that follow the previous call's last
        frame (m <= chunk_frames - 1); the pipeline keeps that frame's gray image on the device
        (the reference's ``prev_gray``, computeOpticalFlowModule.py:34), so the one-frame halo
        between chunks is neither uploaded nor converted again.  Returns m pairs."""
        m = int(frames.shape[0]) if n_frames is None else int(n_frames)
        n = m + 1 if carry else m
        if n < 2 or n > self.F:
            raise ValueError(f"n_frames={n} outside [2, {self.F}]")
        if carry and self._last_gray_index is None:
            raise ValueError("carry=True needs a previous run_chunk call on this pipeline")
        if tuple(frames.shape[1:]) != (self.H, self.W, 3) or frames.dtype != torch.uint8 or not frames.is_cuda:
            raise ValueError("frames must be CUDA uint8 [n,H,W,3] of the pipeline's size")
        if not frames.is_contiguous():
            frames = frames.contiguous()
        L = _lib.lib()
        s = _stream_ptr()
        P = n - 1
        with torch.cuda.device(self.device):
            if carry:
                if self._last_gray_index != 0:
                    self.gray[0].copy_(self.gray[self._last_gray_index])
                _lib.check(L.ofc_bgr2gray(_ptr(frames), _ptr(self.gray[1:]), m * self.H * self.W, s))
            else:
                _lib.check(L.ofc_bgr2gray(_ptr(frames), _ptr(self.gray), n * self.H * self.W, s))
            self._last_gray_index = n - 1
            if self._gray_event is not None:
                self._gray_event.record(torch.cuda.current_stream(self.device))
            _lib.check(L.ofc_farneback_sequence(self.plan._ptr, _ptr(self.gray), n, _ptr(self.flow), _ptr(self.minmax),
                                                _ptr(self.plan.workspace), self.plan.workspace_bytes, s))
            k1 = self.n_clusters == 1
            kc = _ptr(self.km_centre) if k1 else C.c_void_p(0)
            kh = _ptr(self.km_hue) if k1 else C.c_void_p(0)
            if self.fuse_grid:
                # visualisation + grid pass in one kernel: the BGR bytes are written once and not read back
                _lib.check(L.ofc_flow_to_bgr_grid(_ptr(self.flow), P, self.H, self.W, _ptr(self.minmax), _ptr(self.viz),
                                                  _ptr(self.mag_sum), self.rows, self.cols, self.draw_lines, self.threshold,
                                                  _ptr(self.avg_bgr), _ptr(self.avg_hue), kc, kh, s))
            else:
                _lib.check(L.ofc_flow_to_bgr(_ptr(self.flow), P, self.H, self.W, _ptr(self.minmax), _ptr(self.viz),
                                             _ptr(self.mag_sum), s))
                _lib.check(L.ofc_grid_cells(_ptr(self.viz), P, self.H, self.W, self.rows, self.cols, self.draw_lines,
                                            self.threshold, _ptr(self.avg_bgr), _ptr(self.avg_hue), kc, kh, C.c_void_p(0), s))
            if not k1:
                first = 0 if not carry else self._pairs_done
                _lib.check(L.ofc_grid_kmeans_cells(_ptr(self.viz), P, self.H, self.W, self.rows, self.cols, self.draw_lines,
                                                   self.threshold, 0, self.n_clusters, C.c_uint64(self.kmeans_seed),
                                                   C.c_uint64(first), self.kmeans_max_iter, C.c_double(self.kmeans_tol),
                                                   _ptr(self.km_centre), _ptr(self.km_hue), C.c_void_p(0), C.c_void_p(0),
                                                   _ptr(self.km_n_iter), _ptr(self._km_ws), C.c_size_t(self._km_ws.numel()), s))
            self._pairs_done = (self._pairs_done if carry else 0) + P
        return P

    def process_clip(self, frames, pinned_out: torch.Tensor | None = None):
        """Whole clip ``[T,H,W,3]`` uint8 (host numpy / pinned torch / CUDA) ->
        dict of host tensors: ``avg_hue`` ``[T-1,cells]``, ``km_hue`` ``[T-1,cells]``,
        ``mean_magnitude`` ``[T-1]``.  Chunks overlap by one frame (the halo)."""
        import numpy as np
        if isinstance(frames, np.ndarray):
            frames = torch.from_numpy(frames)
        T = int(frames.shape[0])
        avg = torch.empty((T - 1, self.cells), dtype=torch.uint8)
        km = torch.empty((T - 1, self.cells), dtype=torch.uint8)
        mag = torch.empty(T - 1, dtype=torch.float64)
        t = 0
        while t < T - 1:
            # the first chunk carries its own first frame; later chunks only the new frames
            first = t == 0
            n = min(self.F, T - t) if first else min(self.F - 1, T - 1 - t)
            chunk = frames[t:t + n] if first else frames[t + 1:t + 1 + n]
            if not chunk.is_cuda:
                chunk = chunk.to(self.device, non_blocking=True)
            P = self.run_chunk(chunk, carry=not first)
            avg[t:t + P] = self.avg_hue[:P].cpu()
            km[t:t + P] = self.km_hue[:P].cpu()
            mag[t:t + P] = self.mag_sum[:P].cpu() / float(self.H * self.W)     # IEEE division on the host
            t += P
        return {"avg_hue": avg, "km_hue": km, "mean_magnitude": mag}

    def seed(self, first_frame):
        """Start a stream: ``first_frame`` (BGR uint8 [H,W,3], host or device) becomes ``prev_gray``
        (the reference's ``ComputeOpticalFLow.__init__``, computeOpticalFlowModule.py:7-16)."""
        import numpy as np
        f = torch.from_numpy(np.ascontiguousarray(first_frame)) if isinstance(first_frame, np.ndarray) else first_frame
        f = f.to(self.device).contiguous()
        if tuple(f.shape) != (self.H, self.W, 3) or f.dtype != torch.uint8:
            raise ValueError("first_frame must be uint8 [H,W,3] of the pipeline's size")
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().ofc_bgr2gray(_ptr(f), _ptr(self.gray), self.H * self.W, _stream_ptr()))
        self._last_gray_index = 0
        self._pairs_done = 0

    def process_stream(self, frames, on_pairs=None, want_viz: bool = False, nbuf: int = 3):
        """Streaming ingest (SURVEY.md §8f-1): ``frames`` is any iterable of host BGR uint8 frames
        ``[H,W,3]`` (e.g. a ``cv2.VideoCapture`` read loop).  Frames are packed into pinned staging
        chunks and uploaded on a copy stream while the previous chunk computes; results come back
        through pinned buffers.  ``on_pairs(first_pair_index, result_dict)`` is called per chunk with
        host tensors ``avg_hue [p,cells]``, ``km_hue [p,cells]``, ``mean_magnitude [p]`` (and ``viz
        [p,H,W,3]`` when ``want_viz``); without a callback the chunks are concatenated and returned."""
        import numpy as np
        P = self.F - 1
        dev = self.device
        pin = [torch.empty((P, self.H, self.W, 3), dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
        stage = [torch.empty((P, self.H, self.W, 3), dtype=torch.uint8, device=dev) for _ in range(nbuf)]
        out_avg = [torch.empty((P, self.cells), dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
        out_km = [torch.empty((P, self.cells), dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
        out_mag = [torch.empty(P, dtype=torch.float64).pin_memory() for _ in range(nbuf)]
        out_viz = [torch.empty((P, self.H, self.W, 3), dtype=torch.uint8).pin_memory() for _ in range(nbuf)] if want_viz else None
        done = [None] * nbuf                      # event after which slot b's results are on the host / its buffers free
        pending = []                              # (slot, first_pair, n_pairs) in flight
        copy_stream = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        collected = []

        def deliver(upto_all=False):
            while pending and (upto_all or len(pending) >= nbuf - 1):
                b, first, n = pending.pop(0)
                done[b].synchronize()
                res = {"avg_hue": out_avg[b][:n].clone(), "km_hue": out_km[b][:n].clone(),
                       "mean_magnitude": out_mag[b][:n].clone() / float(self.H * self.W)}
                if want_viz:
                    res["viz"] = out_viz[b][:n].clone()
                if on_pairs is not None:
                    on_pairs(first, res)
                else:
                    collected.append(res)

        def submit(b, n, first_pair):
            up = torch.cuda.Event()
            with torch.cuda.stream(copy_stream):
                stage[b][:n].copy_(pin[b][:n], non_blocking=True)
                up.record(copy_stream)
            main.wait_event(up)
            self.run_chunk(stage[b][:n], carry=True)
            out_avg[b][:n].copy_(self.avg_hue[:n], non_blocking=True)
            out_km[b][:n].copy_(self.km_hue[:n], non_blocking=True)
            out_mag[b][:n].copy_(self.mag_sum[:n], non_blocking=True)
            if want_viz:
                out_viz[b][:n].copy_(self.viz[:n], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(main)
            done[b] = ev
            pending.append((b, first_pair, n))

        it = iter(frames)
        try:
            self.seed(next(it))
        except StopIteration:
            raise ValueError("empty frame stream")
        b, fill, n_pairs = 0, 0, 0
        for fr in it:
            if fill == 0 and done[b] is not None:
                deliver()                          # make sure slot b's previous use has been handed over
                done[b].synchronize()
            pin[b][fill].copy_(torch.from_numpy(np.ascontiguousarray(fr)))
            fill += 1
            if fill == P:
                submit(b, P, n_pairs)
                n_pairs += P
                b, fill = (b + 1) % nbuf, 0
        if fill:
            submit(b, fill, n_pairs)
            n_pairs += fill
        deliver(upto_all=True)
        if on_pairs is not None:
            return n_pairs
        if not collected:
            return {"avg_hue": torch.empty((0, self.cells), dtype=torch.uint8),
                    "km_hue": torch.empty((0, self.cells), dtype=torch.uint8),
                    "mean_magnitude": torch.empty(0, dtype=torch.float64)}
        return {k: torch.cat([c[k] for c in collected]) for k in collected[0]}


class LanedPipeline:
    """Several :class:`ClipPipeline` lanes on their own streams, chunks dealt to them in turn.

    A chunk is a chain of kernels of very different character -- the level-0 / level-1 walks own every register and
    tensor-memory column of an SM and are latency-bound, the stage-1 kernels are issue-bound, the coarse levels and the
    tails of every launch leave SMs idle.  With two or three independent chunks in flight the hardware fills one chain's
    gaps with another's CTAs: 5 570 -> 5 995 pairs/s with two lanes, 6 087 with three (1080p, chunks of 33 frames,
    ``tools/two_lane.py``, r03h).  Every lane has its own plan workspace and result buffers (4.5 GB per lane at 1080p).

    ``submit`` enqueues one chunk and returns ``(lane, n_pairs)``; the lane's buffers (``lane.avg_hue`` ...) hold the chunk's
    results once ``lane_stream(lane)`` has run that far.  Work that reads them belongs on that stream (or behind
    ``done_event(lane)``) and must be enqueued before the lane's next ``submit`` -- ``lanes`` chunks later -- overwrites them.
    With ``carry=True`` the chunk's first pair starts at the previous chunk's last frame, whose gray image is taken over
    from the lane that converted it (the reference's ``prev_gray``, computeOpticalFlowModule.py:34)."""

    def __init__(self, width: int, height: int, lanes: int = 2, device=None, **kw):
        if lanes < 1:
            raise ValueError("lanes must be >= 1")
        self.pipes = [ClipPipeline(width, height, device=device, **kw) for _ in range(int(lanes))]
        self.device = self.pipes[0].device
        self.W, self.H, self.F = self.pipes[0].W, self.pipes[0].H, self.pipes[0].F
        self.cells = self.pipes[0].cells
        self.streams = [torch.cuda.Stream(device=self.device) for _ in self.pipes]
        self._done = [torch.cuda.Event() for _ in self.pipes]
        self._taken = [None for _ in self.pipes]        # event: the next lane has copied this lane's last gray frame
        for p in self.pipes:
            p._gray_event = torch.cuda.Event()
        self._next = 0
        self._last = None                                # lane of the previous chunk

    @property
    def n_lanes(self) -> int:
        return len(self.pipes)

    def lane_stream(self, lane: int):
        return self.streams[lane]

    def done_event(self, lane: int):
        return self._done[lane]

    def lane(self, lane: int) -> ClipPipeline:
        return self.pipes[lane]

    def submit(self, frames: torch.Tensor, carry: bool = False, wait=None):
        """Enqueue one chunk on the next lane.  ``wait``: an event after which ``frames`` are complete (default: whatever
        the caller's current stream has enqueued so far).  Returns ``(lane, n_pairs)``."""
        l = self._next
        pipe, s = self.pipes[l], self.streams[l]
        if wait is None:
            s.wait_stream(torch.cuda.current_stream(self.device))
        else:
            s.wait_event(wait)
        if self._taken[l] is not None:                   # the lane's gray buffer is about to be rewritten
            s.wait_event(self._taken[l])
            self._taken[l] = None
        with torch.cuda.stream(s):
            if carry:
                if self._last is None:
                    raise ValueError("carry=True needs a previous chunk")
                prev = self.pipes[self._last]
                if self._last != l:
                    s.wait_event(prev._gray_event)
                    pipe.gray[0].copy_(prev.gray[prev._last_gray_index])
                    pipe._last_gray_index = 0
                    pipe._pairs_done = prev._pairs_done
                    ev = torch.cuda.Event()
                    ev.record(s)
                    self._taken[self._last] = ev
            P = pipe.run_chunk(frames, carry=carry)
            self._done[l].record(s)
        self._last = l
        self._next = (l + 1) % len(self.pipes)
        return l, P

    def seed(self, first_frame):
        """Start a stream of ``carry=True`` chunks: ``first_frame`` becomes ``prev_gray`` (see ClipPipeline.seed)."""
        with torch.cuda.stream(self.streams[0]):
            self.pipes[0].seed(first_frame)
            self.pipes[0]._gray_event.record(self.streams[0])
        self._last, self._next = 0, (1 % len(self.pipes))

    def synchronize(self):
        for s in self.streams:
            s.synchronize()

    def process_clip(self, frames):
        """Whole clip ``[T,H,W,3]`` uint8 on the device -> dict of host tensors like :meth:`ClipPipeline.process_clip`,
        with the chunks dealt over the lanes (results are read back one round of lanes late)."""
        T = int(frames.shape[0])
        avg = torch.empty((T - 1, self.cells), dtype=torch.uint8)
        km = torch.empty((T - 1, self.cells), dtype=torch.uint8)
        mag = torch.empty(T - 1, dtype=torch.float64)
        pending = []                                     # (lane, first_pair, n_pairs)

        def collect():
            l, t0, P = pending.pop(0)
            self._done[l].synchronize()
            pipe = self.pipes[l]
            avg[t0:t0 + P] = pipe.avg_hue[:P].cpu()
            km[t0:t0 + P] = pipe.km_hue[:P].cpu()
            mag[t0:t0 + P] = pipe.mag_sum[:P].cpu() / float(self.H * self.W)

        t = 0
        while t < T - 1:
            first = t == 0
            n = min(self.F, T - t) if first else min(self.F - 1, T - 1 - t)
            chunk = frames[t:t + n] if first else frames[t + 1:t + 1 + n]
            if not chunk.is_cuda:
                chunk = chunk.to(self.device, non_blocking=True)
            if len(pending) == len(self.pipes):          # the lane about to be reused still holds unread results
                collect()
            l, P = self.submit(chunk, carry=not first)
            pending.append((l, t, P))
            t += P
        while pending:
            collect()
        return {"avg_hue": avg, "km_hue": km, "mean_magnitude": mag}
