"""Host side of the k-means stage: the Lloyd loop around libofc's E-step / M-step kernels.

Mirrors what the reference gets from scikit-learn at
k-means-color-clustering/KmeanGrids.py:299-304 and color_kmeans.py:65-78::

    clt = KMeans(n_clusters = k); clt.fit(X); labels = clt.predict(X); clt.cluster_centers_

following sklearn 1.9.0's ``_kmeans_single_lloyd`` (sklearn/cluster/_kmeans.py:627-758,
SURVEY.md Appendix A.5): data centred on its column mean, ``tol_ = mean(var(X)) * tol``,
stop when the labels repeat (strict) or the squared centre shift is <= tol_, one more
E-step when the stop was not strict.  uint8 rows are worked in float64 like sklearn does.

Everything is batched: ``X`` may be ``[n, d]`` (one problem) or ``[B, n, d]`` (B independent
problems of equal shape -- the reference runs one fit per grid cell).  Problems that have
converged are frozen by an ``active`` mask while the others keep iterating.  ``X [n, d]`` with
``init [R, k, d]`` runs R starts of one fit (``KMeans(n_init=R)``) as R problems that read the
same rows (``OFC_KMEANS_SHARED_ROWS``: no copy of X per start).

Multi-GPU: rows sharded over the ranks of ``group``; the only exchange is an all-reduce
of ``[k*d sums | k counts | n_changed]`` per iteration (NCCL over NVLink on GPUs).  For
uint8 data the sums are integers held exactly in float64, so the result does not depend
on the number of ranks or the reduction order.

torch is used for device memory, streams and torch.distributed only.
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np
import torch

from . import _lib

_vp = C.c_void_p
_DT = {torch.uint8: 0, torch.float32: 1, torch.float64: 2}


#: set by tests only (tests/emu: the same .cu sources compiled for the host): the library every entry point of this
#: module and of cosine.py uses instead of libofc.so.  The product never sets it; there is no CPU fallback.
_TEST_LIBRARY = None


def _use_test_library(lib):
    """Private test hook: route this module through the host-side debug emulation (``None`` restores libofc.so)."""
    global _TEST_LIBRARY
    _TEST_LIBRARY = lib


class _Ctx:
    """Library handle + device.  The product path is always libofc.so on a CUDA device."""

    def __init__(self, device, lib=None):
        self.device = torch.device(device)
        if lib is None:
            lib = _TEST_LIBRARY
        if lib is None:
            if self.device.type != "cuda":
                raise _lib.OfcError("a CUDA device is required: this package has no CPU fallback")
            lib = _lib.lib()
            self.check = _lib.check
        else:
            def _check(rc, _l=lib):
                if rc != 0:
                    raise RuntimeError(f"libofc rc={rc}: {_l.ofc_last_error().decode()}")
            self.check = _check
        self.lib = lib

    def stream(self):
        if self.device.type == "cuda":
            return _vp(torch.cuda.current_stream(self.device).cuda_stream)
        return _vp(0)


def _ptr(t):
    return _vp(t.data_ptr()) if t is not None else _vp(0)


def _target_device(X, lib_override=None):
    """Where host inputs go: the current CUDA device (product) -- or the host when a test has installed
    the emulated library.  Fails loudly when neither the GPU nor the CUDA library is there."""
    lib_override = lib_override if lib_override is not None else _TEST_LIBRARY
    if lib_override is not None:
        return None if (isinstance(X, torch.Tensor) and X.is_cuda) else "cpu"
    if isinstance(X, torch.Tensor) and X.is_cuda:
        return None
    if not torch.cuda.is_available():
        raise _lib.OfcError("a CUDA device is required: this package has no CPU fallback")
    _lib.lib()
    return "cuda"


def _as_batch(X, device=None):
    if isinstance(X, np.ndarray):
        X = torch.from_numpy(np.ascontiguousarray(X))
    if X.dtype not in _DT:
        if X.dtype in (torch.int8, torch.int16, torch.int32, torch.int64, torch.bool, torch.float16, torch.bfloat16):
            X = X.to(torch.float64)                      # sklearn: validate_data(dtype=[float64, float32])
        else:
            raise TypeError(f"unsupported dtype {X.dtype}")
    if device is not None and X.device != torch.device(device):
        X = X.to(device)
    single = X.dim() == 2
    if single:
        X = X.unsqueeze(0)
    if X.dim() != 3:
        raise ValueError("X must be [n, d] or [batch, n, d]")
    return X.contiguous(), single


def _check_sample_weight(sample_weight, n: int, x_dtype, rows: int = 1):
    """sklearn's ``_check_sample_weight(sample_weight, X, dtype=X.dtype)`` as KMeans uses it: ``None`` stays None, a number
    is that weight for every row, anything else must be ``(n,)`` (or ``(rows, n)`` for a batch of problems).  The weights
    are cast to the working dtype (float32 for float32 rows, float64 otherwise, uint8 rows included).  All-zero weights,
    NaN and inf raise ValueError as in sklearn; negative weights raise ValueError too (sklearn accepts them in ``fit``,
    but its seeding then fails and an "empty" cluster means nothing).  Returns the numpy array in the working dtype."""
    if sample_weight is None:
        return None
    wdt = np.float32 if x_dtype in (torch.float32, np.float32) else np.float64
    if isinstance(sample_weight, torch.Tensor):
        sample_weight = sample_weight.detach().cpu().numpy()
    if np.ndim(sample_weight) == 0:
        return np.full(n, sample_weight, dtype=wdt)
    w = np.ascontiguousarray(np.asarray(sample_weight, dtype=wdt))
    if w.shape != (n,) and not (rows > 1 and w.shape == (rows, n)):
        raise ValueError(f"sample_weight.shape == {w.shape}, expected {(n,)}!")
    if not np.isfinite(w).all():
        raise ValueError("Input sample_weight contains NaN or infinity.")
    if (w < 0).any():
        raise ValueError("Negative values in sample_weight: KMeans takes non-negative weights.")
    if (w.reshape(-1, n) == 0).all(axis=1).any():
        raise ValueError("Sample weights must contain at least one non-zero number.")
    return w


class LloydState:
    """Buffers of one batched Lloyd run (all on the data's device)."""

    def __init__(self, ctx: _Ctx, X: torch.Tensor, k: int, ws_k: int | None = None, shared_batch: int | None = None,
                 weights: torch.Tensor | None = None):
        """``ws_k``: cluster count the stepwise workspace is sized for (1 when the tensor-core path does
        the E/M steps and only the column statistics run through the stepwise kernels).  ``shared_batch``: run that
        many problems over the one problem of ``X`` ([1, n, d]) without copying it (OFC_KMEANS_SHARED_ROWS).
        ``weights``: float64 sample weights (``[B, n]``, or ``[n]`` for a shared batch) -- every E-step's inertia is
        weighted, and ``wsum`` holds the clusters' weight sums for the weighted M-step."""
        self.ctx, self.X, self.k = ctx, X, int(k)
        self.w = weights
        self.B, self.n, self.d = (int(s) for s in X.shape)
        self.dtype = _DT[X.dtype]
        self.flags = 0                  # OR-ed into the dtype of the calls that read X
        per = self.B                    # problems the workspace queries are asked for; a shared batch needs B times one
        if shared_batch is not None:
            self.B, self.flags, per = int(shared_batch), _lib.OFC_KMEANS_SHARED_ROWS, 1
        dev = X.device
        lib = ctx.lib
        lib.ofc_kmeans_workspace_bytes.restype = C.c_size_t
        lib.ofc_kmeans_workspace_bytes.argtypes = [C.c_int, C.c_int64, C.c_int, C.c_int]
        mul = self.B // per
        self.ws_bytes = mul * int(lib.ofc_kmeans_workspace_bytes(per, self.n, self.d, max(self.k if ws_k is None else int(ws_k), 1)))
        if ws_k is not None and hasattr(lib, "ofc_kmeans_assign_workspace_bytes"):
            # the E-step / centre kernels still run for all k clusters (final inertia, relocation, new centres)
            lib.ofc_kmeans_assign_workspace_bytes.restype = C.c_size_t
            lib.ofc_kmeans_assign_workspace_bytes.argtypes = [C.c_int, C.c_int64, C.c_int, C.c_int]
            self.ws_bytes = max(self.ws_bytes, mul * int(lib.ofc_kmeans_assign_workspace_bytes(per, self.n, self.d, max(self.k, 1))))
        self.ws = torch.empty(max(self.ws_bytes, 256), dtype=torch.uint8, device=dev)
        self.labels = [torch.full((self.B, self.n), -1, dtype=torch.int32, device=dev) for _ in range(2)]
        # the kernels write straight into the buffers the all-reduces move: float64 sums, and ONE int64 buffer holding
        # the member counts followed by the label-change counts (two collectives per iteration, no staging copies)
        self.sums = torch.zeros((self.B, self.k, self.d), dtype=torch.float64, device=dev)
        self.icnt = torch.zeros(self.B * self.k + self.B, dtype=torch.int64, device=dev)
        self.counts = self.icnt[:self.B * self.k].view(self.B, self.k)
        self.n_changed = self.icnt[self.B * self.k:]
        self.shift = torch.zeros(self.B, dtype=torch.float64, device=dev)
        self.inertia = torch.zeros(self.B, dtype=torch.float64, device=dev)
        # device-side loop control (ofc_kmeans_update): which problems still run, who just stopped, iterations done
        self.active = torch.ones(self.B, dtype=torch.uint8, device=dev)
        self.just_done = torch.zeros(self.B, dtype=torch.uint8, device=dev)
        self.n_iter = torch.zeros(self.B, dtype=torch.int32, device=dev)
        self.wsum = torch.zeros((self.B, self.k), dtype=torch.float64, device=dev) if weights is not None else None

    # -- thin wrappers over the C-ABI -----------------------------------------------------
    def assign(self, mean, centres, labels, prev=None, n_changed=None, inertia=None, min_dist=None, active=None):
        c = self.ctx
        if self.w is not None:
            c.check(c.lib.ofc_kmeans_assign_weighted(_ptr(self.X), self.dtype | self.flags, self.B, C.c_int64(self.n), self.d,
                                                     int(centres.shape[1]), _ptr(mean), _ptr(centres), _ptr(self.w), _ptr(labels),
                                                     _ptr(prev), _ptr(n_changed), _ptr(inertia), _ptr(min_dist), _ptr(active),
                                                     _ptr(self.ws), C.c_size_t(self.ws.numel()), c.stream()))
            return
        c.check(c.lib.ofc_kmeans_assign(_ptr(self.X), self.dtype | self.flags, self.B, C.c_int64(self.n), self.d, int(centres.shape[1]),
                                        _ptr(mean), _ptr(centres), _ptr(labels), _ptr(prev), _ptr(n_changed),
                                        _ptr(inertia), _ptr(min_dist), _ptr(active), _ptr(self.ws),
                                        C.c_size_t(self.ws.numel()), c.stream()))

    def step_supported(self) -> bool:
        """uint8 rows whose [k][d] accumulators fit shared memory: E-step + M-step sums in one pass"""
        lib = self.ctx.lib
        return (os.environ.get("OFC_KMEANS_FUSED", "1") != "0" and hasattr(lib, "ofc_kmeans_step_supported")
                and bool(lib.ofc_kmeans_step_supported(self.dtype, self.d, self.k)))

    def step(self, mean, centres, labels, prev, n_changed, sums, counts, active=None):
        c = self.ctx
        c.check(c.lib.ofc_kmeans_step(_ptr(self.X), self.dtype | self.flags, self.B, C.c_int64(self.n), self.d, self.k, _ptr(mean),
                                      _ptr(centres), _ptr(labels), _ptr(prev), _ptr(n_changed), _ptr(sums), _ptr(counts),
                                      _ptr(active), _ptr(self.ws), C.c_size_t(self.ws.numel()), c.stream()))

    def sums_(self, mean, labels, sums, counts, k, square=0, active=None):
        c = self.ctx
        c.check(c.lib.ofc_kmeans_sums(_ptr(self.X), self.dtype | self.flags, self.B, C.c_int64(self.n), self.d, int(k), _ptr(mean),
                                      _ptr(labels), int(square), _ptr(sums), _ptr(counts), _ptr(active), _ptr(self.ws),
                                      C.c_size_t(self.ws.numel()), c.stream()))

    def sums_weighted(self, mean, labels, sums, wsum, active=None):
        """weighted M-step: sums of (x - mean) w and the clusters' weight sums (float64) in place of the counts"""
        c = self.ctx
        c.check(c.lib.ofc_kmeans_sums_weighted(_ptr(self.X), self.dtype | self.flags, self.B, C.c_int64(self.n), self.d, self.k,
                                               _ptr(mean), _ptr(labels), _ptr(self.w), _ptr(sums), _ptr(wsum), _ptr(active),
                                               _ptr(self.ws), C.c_size_t(self.ws.numel()), c.stream()))

    def centres_(self, sums, counts, mean_sub, use_reciprocal, centres, shift, active=None):
        c = self.ctx
        c.check(c.lib.ofc_kmeans_centres(self.B, self.d, int(centres.shape[1]), _ptr(sums), _ptr(counts), _ptr(mean_sub),
                                         int(use_reciprocal), _ptr(centres), _ptr(shift), _ptr(active), _ptr(self.ws),
                                         C.c_size_t(self.ws.numel()), c.stream()))

    def update_(self, sums, counts, mean_sub, use_reciprocal, round_f32, centres, n_changed, tol, it, n_active, lab, lab_other,
                it_counter=None):
        """new centres + sklearn's stopping rule on the device (no read-back): see ofc_kmeans_update.  float64 ``counts``
        are the weight sums of a weighted fit (ofc_kmeans_update_weighted)"""
        c = self.ctx
        fn = c.lib.ofc_kmeans_update_weighted if counts.dtype == torch.float64 else c.lib.ofc_kmeans_update
        c.check(fn(self.B, C.c_int64(self.n), self.d, int(centres.shape[1]), _ptr(sums), _ptr(counts), _ptr(mean_sub),
                   int(use_reciprocal), int(round_f32), _ptr(centres), _ptr(self.shift), _ptr(n_changed), _ptr(tol), int(it),
                   _ptr(self.active), _ptr(self.just_done), _ptr(self.n_iter), _ptr(n_active), _ptr(lab), _ptr(lab_other),
                   _ptr(it_counter), _ptr(self.ws), C.c_size_t(self.ws.numel()), c.stream()))

    def relocate(self, mean, labels, centres_old, sums, counts, raw_sums, active=None):
        c = self.ctx
        if counts.dtype == torch.float64:          # weight sums: a cluster is empty when its weight is 0
            c.check(c.lib.ofc_kmeans_relocate_weighted(_ptr(self.X), self.dtype | self.flags, self.B, C.c_int64(self.n), self.d, self.k,
                                                       _ptr(mean), _ptr(labels), _ptr(centres_old), _ptr(self.w), _ptr(sums),
                                                       _ptr(counts), int(raw_sums), _ptr(active), _ptr(self.row_scratch()),
                                                       c.stream()))
            return
        c.check(c.lib.ofc_kmeans_relocate(_ptr(self.X), self.dtype | self.flags, self.B, C.c_int64(self.n), self.d, self.k, _ptr(mean),
                                          _ptr(labels), _ptr(centres_old), _ptr(sums), _ptr(counts), int(raw_sums),
                                          _ptr(active), _ptr(self.row_scratch()), c.stream()))

    def row_scratch(self):
        """float64 [B, n]: the row distances of the empty-cluster relocation (allocated on first use)"""
        if getattr(self, "_row_scratch", None) is None:
            self._row_scratch = torch.empty((self.B, max(self.n, 1)), dtype=torch.float64, device=self.X.device)
        return self._row_scratch


class TensorCoreSteps:
    """E-step / M-step of ONE float32 or uint8 problem on the tensor-core path (libofc's ofc_kmeans_tc_*): the
    centred rows are split once into TF32-exact hi parts and exact remainders; every E-step is a
    3xTF32 tcgen05 distance GEMM used as a filter plus a re-evaluation of the near-ties in the working
    precision (float32 rows: float32; uint8 rows: float64 on the original bytes), so the labels are those
    of the CUDA-core E-step; the M-step walks a label-sorted member list (uint8: exact integer sums)."""

    def __init__(self, st: "LloydState", mean: torch.Tensor):
        self.st = st
        c = st.ctx
        dev = st.X.device
        n, d, k = st.n, st.d, st.k
        self.Xh = torch.empty((n, d), dtype=torch.float32, device=dev)
        self.Xl = torch.empty((n, d), dtype=torch.float32, device=dev)
        self.xnorm = torch.empty(n, dtype=torch.float32, device=dev)
        self.ws_bytes = int(c.lib.ofc_kmeans_tc_workspace_bytes(C.c_int64(n), d, k))
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.n_rechecked = torch.zeros(1, dtype=torch.int32, device=dev)
        self.u8 = st.dtype == 0
        self.mean = mean
        prep = c.lib.ofc_kmeans_tc_prepare_u8 if self.u8 else c.lib.ofc_kmeans_tc_prepare
        c.check(prep(_ptr(st.X), _ptr(mean), C.c_int64(n), d, _ptr(self.Xh), _ptr(self.Xl), _ptr(self.xnorm), c.stream()))

    def assign(self, centres, labels, prev=None, n_changed=None, inertia=None):
        st, c = self.st, self.st.ctx
        if self.u8:
            c.check(c.lib.ofc_kmeans_tc_assign_u8(_ptr(st.X), _ptr(self.mean), _ptr(self.Xh), _ptr(self.Xl), _ptr(self.xnorm),
                                                  C.c_int64(st.n), st.d, st.k, _ptr(centres), _ptr(labels), _ptr(prev),
                                                  _ptr(n_changed), _ptr(self.n_rechecked), _ptr(self.ws),
                                                  C.c_size_t(self.ws_bytes), c.stream()))
            if inertia is not None:
                # inertia of the final (centres, labels): the float64 CUDA-core E-step (idempotent on the labels)
                st.assign(self.mean.view(1, -1), centres, labels, inertia=inertia)
            return
        if st.w is not None:
            c.check(c.lib.ofc_kmeans_tc_assign_weighted(_ptr(self.Xh), _ptr(self.Xl), _ptr(self.xnorm), C.c_int64(st.n), st.d, st.k,
                                                        _ptr(centres), _ptr(st.w), _ptr(labels), _ptr(prev), _ptr(n_changed),
                                                        _ptr(inertia), _ptr(self.n_rechecked), _ptr(self.ws), C.c_size_t(self.ws_bytes),
                                                        c.stream()))
            return
        c.check(c.lib.ofc_kmeans_tc_assign(_ptr(self.Xh), _ptr(self.Xl), _ptr(self.xnorm), C.c_int64(st.n), st.d, st.k,
                                           _ptr(centres), _ptr(labels), _ptr(prev), _ptr(n_changed), _ptr(inertia),
                                           _ptr(self.n_rechecked), _ptr(self.ws), C.c_size_t(self.ws_bytes), c.stream()))

    def sums_(self, labels, sums, counts):
        """member counts into ``counts``; a weighted fit also writes the weight sums into ``st.wsum``"""
        st, c = self.st, self.st.ctx
        if st.w is not None:
            if self.u8:
                c.check(c.lib.ofc_kmeans_tc_sums_u8_weighted(_ptr(st.X), C.c_int64(st.n), st.d, st.k, _ptr(labels), _ptr(st.w),
                                                             _ptr(sums), _ptr(counts), _ptr(st.wsum), _ptr(self.ws),
                                                             C.c_size_t(self.ws_bytes), c.stream()))
            else:
                c.check(c.lib.ofc_kmeans_tc_sums_weighted(_ptr(self.Xh), _ptr(self.Xl), C.c_int64(st.n), st.d, st.k, _ptr(labels),
                                                          _ptr(st.w), _ptr(sums), _ptr(counts), _ptr(st.wsum), _ptr(self.ws),
                                                          C.c_size_t(self.ws_bytes), c.stream()))
            return
        if self.u8:         # raw (exact integer) sums like the stepwise uint8 path
            c.check(c.lib.ofc_kmeans_tc_sums_u8(_ptr(st.X), C.c_int64(st.n), st.d, st.k, _ptr(labels), _ptr(sums), _ptr(counts),
                                                _ptr(self.ws), C.c_size_t(self.ws_bytes), c.stream()))
            return
        c.check(c.lib.ofc_kmeans_tc_sums(_ptr(self.Xh), _ptr(self.Xl), C.c_int64(st.n), st.d, st.k, _ptr(labels), _ptr(sums),
                                         _ptr(counts), _ptr(self.ws), C.c_size_t(self.ws_bytes), c.stream()))


def _tc_worth_it(dtype: int, d: int, k: int) -> bool:
    """float32 rows: always past d = 32.  uint8 rows pay 8 bytes per element for the split copy, so the tensor cores
    are only used where the float64 CUDA-core E-step is the bottleneck (k * d large)."""
    return dtype == 1 or k * d >= 4096


def _tc_wanted(Xb, k) -> bool:
    """does the fit of ``Xb`` ([B, n, d]) with k clusters run its E/M steps on the tensor cores (TensorCoreSteps)?"""
    B, n, d = (int(s) for s in Xb.shape)
    return (_TEST_LIBRARY is None and Xb.is_cuda and Xb.dtype in (torch.float32, torch.uint8) and B == 1
            and d > 32 and d % 4 == 0 and 2 <= k <= 4096 and n < 2 ** 31
            and _tc_worth_it(_DT[Xb.dtype], d, k) and os.environ.get("OFC_KMEANS_TC", "1") != "0")


def _relocate_across_ranks(st: "LloydState", mean, labels, centres_old, sums, counts, raw_sums: bool, group, row_offset: int):
    """Empty-cluster relocation (_k_means_common.pyx:167-211) for row-sharded data, on the all-reduced sums / counts:
    every rank lists its farthest rows (ofc_kmeans_far_points: the single-GPU kernel's arithmetic and tie rule),
    the lists are all-gathered, and every rank applies the same moves -- each empty cluster, in index order, takes
    the globally farthest remaining row (ties: lowest global row index).  Same result as one GPU on the whole set."""
    import torch.distributed as dist
    c = st.ctx
    world = dist.get_world_size(group)
    B, k, d = st.B, st.k, st.d
    counts_h = counts.cpu().numpy()
    n_far = int((counts_h == 0).sum(axis=1).max())
    dev = st.X.device
    val = torch.full((B, n_far), -1.0, dtype=torch.float64, device=dev)
    idx = torch.full((B, n_far), -1, dtype=torch.int64, device=dev)
    if st.n > 0:
        c.check(c.lib.ofc_kmeans_far_points(_ptr(st.X), st.dtype, B, C.c_int64(st.n), d, k, _ptr(mean), _ptr(labels), _ptr(centres_old),
                                            n_far, _ptr(val), _ptr(idx), _ptr(st.row_scratch()), c.stream()))
    if st.n > 0:
        safe = idx.clamp(min=0)
        rows = torch.gather(st.X, 1, safe.unsqueeze(-1).expand(B, n_far, d)).to(torch.float64)
        if not raw_sums and mean is not None:
            rows = rows - mean.unsqueeze(1)
        lab = torch.gather(labels, 1, safe).to(torch.float64)
    else:                                                    # a rank without rows offers no candidate (idx stays -1)
        rows = torch.zeros((B, n_far, d), dtype=torch.float64, device=dev)
        lab = torch.zeros((B, n_far), dtype=torch.float64, device=dev)
    gidx = torch.where(idx >= 0, idx + row_offset, idx).to(torch.float64)
    pay = torch.cat([val.unsqueeze(-1), gidx.unsqueeze(-1), lab.unsqueeze(-1), rows], dim=-1).contiguous()   # [B, n_far, 3 + d]
    allpay = [torch.empty_like(pay) for _ in range(world)]
    dist.all_gather(allpay, pay, group=group)
    allpay = torch.cat(allpay, dim=1).cpu().numpy()                                                         # [B, world * n_far, 3 + d]
    sums_h, changed = sums.cpu().numpy(), False
    for b in range(B):
        cand = [r for r in allpay[b] if r[1] >= 0]
        cand.sort(key=lambda r: (-r[0], r[1]))
        empties = [j for j in range(k) if counts_h[b, j] == 0]
        if not empties or not cand or not (cand[0][0] > 0.0):
            continue                                         # np.max(distances) == 0: nothing to do
        for e, r in zip(empties, cand):
            old = int(r[2])
            sums_h[b, old] -= r[3:]
            sums_h[b, e] = r[3:]
            counts_h[b, e] = 1
            counts_h[b, old] -= 1
            changed = True
    if changed:
        sums.copy_(torch.from_numpy(sums_h))
        counts.copy_(torch.from_numpy(counts_h))


def _all_reduce(t, group):
    import torch.distributed as dist
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)


def column_mean_var(st: LloydState, group=None):
    """Column mean and variance of every problem ([B, d] float64 each), as numpy computes
    them for ``X.mean(axis=0)`` / ``np.var(X, axis=0)`` (_kmeans.py:285-293, 1487).
    uint8 data: exact integer sums -> exact rational variance."""
    B, d, dev = st.B, st.d, st.X.device
    s1 = torch.empty((B, 1, d), dtype=torch.float64, device=dev)
    cnt = torch.empty((B, 1), dtype=torch.int64, device=dev)
    st.sums_(None, None, s1, cnt, 1)
    red = torch.cat([s1.view(B, d), cnt.to(torch.float64)], dim=1)
    if group is not None:
        _all_reduce(red, group)
    n_tot = red[:, d:d + 1]
    mean = red[:, :d] / n_tot
    s2 = torch.empty((B, 1, d), dtype=torch.float64, device=dev)
    if st.dtype == 0:
        # exact: var = (sum x^2 - (sum x)^2 / n) / n with integer sums
        st.sums_(None, None, s2, None, 1, square=1)
        sq = s2.view(B, d).clone()
        if group is not None:
            _all_reduce(sq, group)
        # one read-back per fit (set-up, not the iteration loop); int / int is correctly rounded in Python
        host = torch.cat([red[:, :d], sq, n_tot], dim=1).cpu().numpy()
        var = np.empty((B, d))
        for b in range(B):
            N = int(host[b, 2 * d])
            var[b] = [(int(host[b, d + t]) * N - int(host[b, t]) ** 2) / (N * N) for t in range(d)]
        var = torch.from_numpy(var).to(dev)
    else:
        st.sums_(mean.contiguous(), None, s2, None, 1, square=1)
        sq = s2.view(B, d).clone()
        if group is not None:
            _all_reduce(sq, group)
        var = sq / n_tot
    return mean.contiguous(), var, n_tot.view(-1)


#: how many iterations the host may run ahead of the device's "everybody has stopped" signal
_POLL_LAG = 4
#: iterations enqueued one by one before the loop body is captured in a CUDA graph (even)
_EAGER_ITERATIONS = 8


def lloyd(X, init, max_iter: int = 300, tol: float = 1e-4, group=None, sample_weight=None, _host_relocation: bool = False):
    """Batched ``KMeans(n_clusters=k, init=init, n_init=1, max_iter=max_iter, tol=tol).fit(X, sample_weight=sample_weight)``.

    X ``[n,d]`` or ``[B,n,d]`` (uint8 / float32 / float64; torch on the compute device, or numpy);
    init ``[k,d]`` or ``[B,k,d]``.  With ``group`` every rank passes its own rows (same B, d, k)
    and receives the global centres / inertia and the labels of its rows.

    ``X [n,d]`` with ``init [R,k,d]``: R starts over the same rows, returned as ``[R, ...]``.  Every start gives the
    bits it gives alone (``lloyd(X, init[r])``): the batch reads X with a batch stride of 0 and the M-step sums
    of a start are folded in the order of a single problem.  The column statistics are computed once.  Where a
    single start runs on the tensor cores, the starts run one after another (a batch would take the CUDA-core
    M-step, whose float32 sums are ordered differently).  Not with ``group``.

    The loop keeps the host out of the data path: every iteration is a handful of kernel launches (E-step +
    M-step sums, empty-cluster relocation, ``ofc_kmeans_update`` = new centres + stopping rule on the device);
    the only thing the host reads is the "problems still running" counter, asynchronously and ``_POLL_LAG``
    iterations late -- the iterations enqueued past the stop are skipped by every kernel.  With ``group`` the
    kernels write into the buffers the two all-reduces move (float64 sums; int64 counts + label changes), and the
    relocation of empty clusters across ranks runs on the device as well: every rank lists its farthest rows
    (``ofc_kmeans_far_payload``, skipped on the device when no cluster is empty), the lists are all-gathered and every
    rank applies the same moves (``ofc_kmeans_relocate_merge``).  Should more clusters be empty at once than the
    list holds (16), the fit is redone with the host-merged relocation (``_relocate_across_ranks``).

    ``sample_weight`` (``[n]``, or ``[B, n]`` for a batch; numpy or torch; see :func:`_check_sample_weight`): the weighted
    fit of sklearn -- M-step sums of x w and float64 weight sums (a cluster is empty when its weight is 0), weighted
    relocation and inertia.  The column mean, the tolerance and the stopping rule stay unweighted, as in sklearn.  The
    weighted fit never takes the fused uint8 step.  ``None`` runs the unweighted kernels.  Not with ``group``.

    Returns ``(labels int32, centres float64, inertia float64, n_iter int64)`` as torch
    tensors on X's device, squeezed when X was ``[n,d]``.
    """
    if sample_weight is not None and group is not None:
        raise NotImplementedError("sample_weight with a row-sharded fit (group)")
    Xb, single = _as_batch(X, _target_device(X))
    ctx = _Ctx(Xb.device)
    w_host = _check_sample_weight(sample_weight, int(Xb.shape[1]), Xb.dtype, rows=int(Xb.shape[0]))
    init_arg = init
    init = torch.as_tensor(np.asarray(init) if not isinstance(init, torch.Tensor) else init)
    init = init.to(device=Xb.device, dtype=torch.float64)
    shared = single and init.dim() == 3                           # several starts over one X
    if shared:
        if group is not None:
            raise NotImplementedError("several starts (init [R, k, d]) of a row-sharded fit")
        if _tc_wanted(Xb, int(init.shape[1])):
            runs = [lloyd(Xb[0], init[r], max_iter, tol, sample_weight=w_host) for r in range(int(init.shape[0]))]
            return tuple(torch.stack(t) for t in zip(*runs))
    elif init.dim() == 2:
        init = init.unsqueeze(0).expand(Xb.shape[0], -1, -1)
    init = init.contiguous()
    B, n, d = (int(s) for s in Xb.shape)
    if shared:
        B = int(init.shape[0])
    k = int(init.shape[1])
    if init.dim() != 3 or init.shape[0] != B or init.shape[2] != d:
        raise ValueError(f"init shape {tuple(init.shape)} does not match X {tuple(Xb.shape)}")
    use_tc = not shared and _tc_wanted(Xb, k)
    weighted = w_host is not None
    w_dev = None
    if weighted:                     # float64 on the device: [n] read by every start of a shared batch, else [B, n]
        w_dev = torch.from_numpy(w_host.astype(np.float64)).to(Xb.device)
        if not shared:
            w_dev = w_dev.view(-1, n).expand(B, n).contiguous()
    st = LloydState(ctx, Xb, k, ws_k=1 if use_tc else None, shared_batch=B if shared else None, weights=w_dev)
    dev = Xb.device
    row_offset, n_total = 0, n
    if group is not None:
        # global index of this rank's first row (ranks hold consecutive row ranges): the tie rule of the relocation
        import torch.distributed as dist
        ns = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(dist.get_world_size(group))]
        dist.all_gather(ns, torch.tensor([n], dtype=torch.int64, device=dev), group=group)
        ns = [int(t.item()) for t in ns]
        row_offset, n_total = sum(ns[:dist.get_rank(group)]), sum(ns)
    if n_total < k:
        raise ValueError(f"n_samples={n_total} should be >= n_clusters={k}.")   # _kmeans.py:876-879
    # a shared batch: the statistics once, as a single fit computes them, then the same values for every start
    mean, var, _ = column_mean_var(LloydState(ctx, Xb, 1) if shared else st, group)
    tol_ = (var.mean(dim=1) * tol).expand(B).contiguous()        # stays on the device
    mean = mean.expand(B, d).contiguous()
    is_u8 = st.dtype == 0
    is_f32 = st.dtype == 1
    if is_f32:
        # sklearn keeps float32 data in float32: centre with the float32 mean
        mean = mean.to(torch.float32).to(torch.float64).contiguous()
    centres = (init - mean.unsqueeze(1)).contiguous()            # centred
    if is_f32:
        centres = centres.to(torch.float32).to(torch.float64).contiguous()
    # dense float32 corner (d > 32): E/M steps on the tensor-core path, same labels as the float32 kernels
    tc = TensorCoreSteps(st, mean[0].contiguous()) if use_tc else None
    # the fused step's exact integer accumulators do not hold real-valued x w: a weighted uint8 fit takes two kernels
    fused = tc is None and is_u8 and not weighted and st.step_supported()
    counts_or_w = st.wsum if weighted else st.counts            # what the relocation and the centre update run on

    active = st.active
    n_active = torch.zeros(max(max_iter, 1), dtype=torch.int32, device=dev)        # problems still running after iteration i
    is_cuda = dev.type == "cuda"
    seen = torch.empty(max(max_iter, 1), dtype=torch.int32, pin_memory=is_cuda)
    events = []
    flag_host = None
    n_far = min(k, 16)
    payload = allpay = overflow = None
    world = 1
    if group is not None:
        import torch.distributed as dist
        world = dist.get_world_size(group)
        if _host_relocation:
            flag_host = torch.empty(1, dtype=torch.uint8, pin_memory=is_cuda)
        else:
            payload = torch.empty((B, n_far, 3 + d), dtype=torch.float64, device=dev)
            allpay = torch.empty((world, B, n_far, 3 + d), dtype=torch.float64, device=dev)
            overflow = torch.zeros(1, dtype=torch.int32, device=dev)
    overflow_seen = torch.zeros(max(max_iter, 1), dtype=torch.int32, pin_memory=is_cuda) if overflow is not None else None
    # ranks on one node exchange through NVLink peer memory (peer.py): the E/M kernels write this rank's sums / counts /
    # label changes into its shared buffer (two slots, alternating per iteration) and ONE kernel pulls and adds every
    # rank's copy; the far-point lists of the relocation travel the same way.  None -> the NCCL collectives.
    px = None
    local = [(st.sums, st.counts, st.n_changed)] * 2
    n_f64, n_i64 = B * k * d, B * k + B
    if payload is not None and is_cuda and _TEST_LIBRARY is None:
        from .peer import PeerExchange
        px = PeerExchange.create(group, dev, (n_f64 + n_i64) * 8, payload.numel() * 8)
    if px is not None:
        local = []
        for s in (0, 1):
            r = px.region(px.slot_offset(s), (n_f64 + n_i64) * 8)
            ic = r[n_f64 * 8:].view(torch.int64)
            local.append((r[:n_f64 * 8].view(torch.float64).view(B, k, d), ic[:B * k].view(B, k), ic[B * k:]))
        payload = px.region(px.gather_offset(), payload.numel() * 8).view(torch.float64).view(B, n_far, 3 + d)
    it_counter = torch.zeros(1, dtype=torch.int32, device=dev)       # iteration number, kept on the device

    def iteration(cur):
        """one Lloyd iteration, enqueued on the current stream; nothing in it depends on host-side values, so on one GPU it
        can be captured in a CUDA graph (the iteration number is `it_counter`)"""
        lab, lab_old = st.labels[cur], st.labels[cur ^ 1]
        sums_w, counts_w, changed_w = local[cur]                 # where this rank's partial results go
        if tc is not None:
            tc.assign(centres, lab, prev=lab_old, n_changed=changed_w)
            tc.sums_(lab, sums_w, counts_w)
        elif fused:
            st.step(mean, centres, lab, lab_old, changed_w, sums_w, counts_w, active=active)
        else:
            st.assign(mean, centres, lab, prev=lab_old, n_changed=changed_w, active=active)
            # uint8: raw (exact integer) sums; floats: sums of the centred rows like sklearn
            if weighted:
                st.sums_weighted(None if is_u8 else mean, lab, sums_w, st.wsum, active=active)
            else:
                st.sums_(None if is_u8 else mean, lab, sums_w, counts_w, k, active=active)
        if group is not None:
            if B > 1:
                # stopped problems contribute nothing (their buffers hold already-reduced values)
                off = (active == 0)
                sums_w.masked_fill_(off.view(B, 1, 1), 0.0)
                counts_w.masked_fill_(off.view(B, 1), 0)
                changed_w.masked_fill_(off, 0)
            if px is not None:
                px.exchange(px.slot_offset(cur), 0, n_f64, n_i64, st.sums, st.icnt, None, ctx.stream())
            else:
                _all_reduce(st.sums, group)
                _all_reduce(st.icnt, group)
            if _host_relocation:
                flag_dev = ((st.counts == 0) & (active != 0).view(B, 1)).any().to(torch.uint8).view(1)
                flag_host.copy_(flag_dev, non_blocking=True)
                if is_cuda:
                    torch.cuda.current_stream(dev).synchronize()
                if int(flag_host[0]):
                    _relocate_across_ranks(st, mean, lab, centres, st.sums, st.counts, is_u8, group, row_offset)
            else:
                ctx.check(ctx.lib.ofc_kmeans_far_payload(_ptr(st.X), st.dtype, B, C.c_int64(n), d, k, _ptr(mean), _ptr(lab), _ptr(centres),
                                                         _ptr(st.counts), int(is_u8), n_far, C.c_int64(row_offset), _ptr(payload),
                                                         _ptr(st.row_scratch()), _ptr(active), ctx.stream()))
                if px is not None:
                    # only when some cluster is empty (the all-reduced counts say so on every rank alike)
                    px.exchange(px.gather_offset(), 1, payload.numel(), 0, allpay, None, st.counts.view(-1), ctx.stream())
                elif is_cuda:
                    dist.all_gather_into_tensor(allpay, payload, group=group)
                else:
                    dist.all_gather(list(allpay.unbind(0)), payload, group=group)
                ctx.check(ctx.lib.ofc_kmeans_relocate_merge(B, d, k, world, n_far, _ptr(allpay), _ptr(st.sums), _ptr(st.counts),
                                                            _ptr(overflow), _ptr(active), ctx.stream()))
        else:
            st.relocate(mean, lab, centres, st.sums, counts_or_w, is_u8, active=active)
        st.update_(st.sums, counts_or_w, mean if is_u8 else None, 0 if is_u8 else 1, 1 if is_f32 else 0, centres, st.n_changed,
                   tol_, 0, n_active, lab, lab_old, it_counter=it_counter)

    def stopped(upto):
        """have all problems stopped by iteration `upto` (as far as the host has seen)?  None = keep going"""
        if overflow is not None and int(overflow_seen[upto]):
            return True
        return int(seen[upto]) == 0

    lag = _POLL_LAG if is_cuda and not _host_relocation else 0
    # tensor-core fits with long iterations (>= ~0.3 ms of kernels): the tensor-core kernels do not look at the stop flag,
    # so every iteration enqueued past the stop costs its full time (measured r02k: 1 M x 128, k = 1024 on 2 GPUs, 81 ms
    # with six iterations of overshoot against 69 ms with four).  One iteration of look-ahead hides the host's poll there,
    # and launch overhead is noise next to the kernels, so no graph either.
    heavy = tc is not None and float(n) * k * d >= 1e9
    if heavy and lag:
        lag = 1
    use_graph = (is_cuda and _TEST_LIBRARY is None and max_iter >= 8 and not heavy and os.environ.get("OFC_KMEANS_GRAPH", "1") != "0"
                 and (group is None or px is not None))
    it = 0
    done = False
    n_eager = min(max_iter, _EAGER_ITERATIONS) if use_graph else max_iter
    # eager iterations: all of them without a graph; otherwise the first _EAGER_ITERATIONS (an even number: the graph
    # starts on label buffer 0).  They do the lazy allocations and shared-memory opt-ins a capture must not contain,
    # and short fits never pay for a capture: measured (r02i) a 5-iteration fit of 8 M x 4 rows takes 1.4 ms eagerly
    # and 2.4 ms when a graph is captured after two iterations
    while it < n_eager and not done:
        iteration(it & 1)
        seen[it:it + 1].copy_(n_active[it:it + 1], non_blocking=True)
        if overflow is not None:
            overflow_seen[it:it + 1].copy_(overflow, non_blocking=True)
        if is_cuda:
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(dev))
            events.append(ev)
        back = it - lag
        if back >= 0:
            if is_cuda:
                events[back].synchronize()
            done = stopped(back)
        it += 1
    if use_graph and not done and it < max_iter:
        # one GPU: two iterations (one per label buffer) captured once and replayed -- a fit is then a handful of graph
        # launches instead of ~10 kernel launches and ctypes calls per iteration
        torch.cuda.current_stream(dev).synchronize()
        if int(seen[it - 1]) != 0:
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                iteration(0)
                iteration(1)
            replays = []
            while it + 2 <= max_iter:
                graph.replay()
                seen.copy_(n_active, non_blocking=True)
                if overflow is not None:
                    overflow_seen[:1].copy_(overflow, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(dev))
                replays.append((ev, it + 1))
                it += 2
                if len(replays) > 2:
                    ev_b, upto = replays[-3]
                    ev_b.synchronize()
                    if int(seen[upto]) == 0 or (overflow is not None and int(overflow_seen[0])):
                        done = True
                        break
            if not done and it < max_iter:                     # odd max_iter: the last iteration
                torch.cuda.current_stream(dev).synchronize()
                if int(seen[it - 1]) != 0:
                    iteration(it & 1)
                    it += 1
    if overflow is not None:
        if is_cuda:
            torch.cuda.current_stream(dev).synchronize()
        if px is not None:
            px.check()
        if int(overflow.item()):
            # more clusters empty at once than the device-side candidate list holds: redo the fit with the host-merged
            # relocation (every rank takes this branch: the all-reduced counts are the same everywhere)
            return lloyd(X, init_arg, max_iter, tol, group, sample_weight, _host_relocation=True)
    final = st.labels[0]
    # strict stops already hold the labels of the final centres; the rest get one more E-step
    # (_kmeans.py:745-755).  Re-running it for everyone is idempotent for the strict ones and
    # yields the inertia of the final (centres, labels) in the same pass.
    if tc is not None:
        tc.assign(centres, final, inertia=st.inertia)
    else:
        st.assign(mean, centres, final, inertia=st.inertia)
    inertia = st.inertia.clone()
    if group is not None:
        _all_reduce(inertia, group)
    out_centres = centres + mean.unsqueeze(1)
    n_iter_t = st.n_iter.to(torch.int64)
    if single and not shared:
        return final[0], out_centres[0], inertia[0], n_iter_t[0]
    return final, out_centres, inertia, n_iter_t


def lloyd_cells(X, n_clusters: int, init=None, seed: int = 0, max_iter: int = 300, tol: float = 1e-4):
    """All Lloyd runs of a batch of small uint8 problems in ONE kernel launch (one CTA per problem): the
    reference's per-cell ``KMeans(n_clusters=k).fit`` loop over a frame's grid cells
    (KmeanGrids.py:376-392).  X uint8 ``[B, n, d]`` (d <= 8, k <= 64).  ``init`` ``[B,k,d]`` / ``[k,d]``
    gives the results of :func:`lloyd`; ``init=None`` seeds every problem with k-means++ from ``seed``.

    Returns ``(labels int32 [B,n], centres float64 [B,k,d], inertia [B], n_iter int32 [B], counts int64 [B,k])``
    on X's device; ``counts`` are the member counts of the final labels."""
    Xb, single = _as_batch(X, _target_device(X))
    if Xb.dtype != torch.uint8:
        raise TypeError("lloyd_cells takes uint8 rows (the reference's pixels)")
    ctx = _Ctx(Xb.device)
    B, n, d = (int(v) for v in Xb.shape)
    k = int(n_clusters)
    dev = Xb.device
    init_t = None
    if init is not None:
        init_t = torch.as_tensor(np.asarray(init) if not isinstance(init, torch.Tensor) else init)
        init_t = init_t.to(device=dev, dtype=torch.float64)
        if init_t.dim() == 2:
            init_t = init_t.unsqueeze(0).expand(B, -1, -1)
        init_t = init_t.contiguous()
        if tuple(init_t.shape) != (B, k, d):
            raise ValueError(f"init shape {tuple(init_t.shape)} does not match ({B}, {k}, {d})")
    labels = torch.empty((B, n), dtype=torch.int32, device=dev)
    centres = torch.empty((B, k, d), dtype=torch.float64, device=dev)
    inertia = torch.empty(B, dtype=torch.float64, device=dev)
    n_iter = torch.empty(B, dtype=torch.int32, device=dev)
    counts = torch.empty((B, k), dtype=torch.int64, device=dev)
    ws = torch.empty(B * n if init_t is None else 1, dtype=torch.float64, device=dev)
    ctx.check(ctx.lib.ofc_kmeans_cells(_ptr(Xb), B, C.c_int64(n), d, k, _ptr(init_t), C.c_uint64(int(seed) & (2 ** 64 - 1)),
                                       int(max_iter), C.c_double(float(tol)), _ptr(labels), _ptr(centres), _ptr(inertia),
                                       _ptr(n_iter), _ptr(counts), _ptr(ws), C.c_size_t(ws.numel() * 8), ctx.stream()))
    if single:
        return labels[0], centres[0], inertia[0], n_iter[0], counts[0]
    return labels, centres, inertia, n_iter, counts


def predict(X, centres):
    """``KMeans.predict``: E-step on the un-centred rows (_kmeans.py:1075-1107)."""
    Xb, single = _as_batch(X, _target_device(X))
    ctx = _Ctx(Xb.device)
    c = torch.as_tensor(np.asarray(centres) if not isinstance(centres, torch.Tensor) else centres)
    c = c.to(device=Xb.device, dtype=torch.float64)
    if c.dim() == 2:
        c = c.unsqueeze(0).expand(Xb.shape[0], -1, -1)
    c = c.contiguous()
    st = LloydState(ctx, Xb, int(c.shape[1]))
    st.assign(None, c, st.labels[0])
    return st.labels[0][0] if single else st.labels[0]


def transform(X, centres):
    """``KMeans.transform``: every row's Euclidean distance to every centre, ``euclidean_distances(X, centres)``
    (_kmeans.py ``_transform``), as ``[n, k]`` on X's compute device.  The distances are the direct difference in float64
    on the un-centred rows (``ofc_kmeans_distances``), not sklearn's norm form, so they do not cancel.  The output is
    float32 exactly when X and ``centres`` are both float32 (sklearn's ``check_pairwise_arrays``), float64 otherwise;
    X of another dtype is worked as float64, as sklearn's ``validate_data(dtype=[float64, float32])``."""
    Xb, single = _as_batch(X, _target_device(X))
    if not single:
        raise ValueError("Expected 2D array")
    n, d = int(Xb.shape[1]), int(Xb.shape[2])
    if n == 0:
        raise ValueError(f"Found array with 0 sample(s) (shape=(0, {d})) while a minimum of 1 is required.")
    c = centres if isinstance(centres, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(centres))
    out_f32 = Xb.dtype == torch.float32 and c.dtype == torch.float32
    c = c.to(device=Xb.device, dtype=torch.float64).contiguous()
    if c.dim() != 2 or int(c.shape[1]) != d:
        raise ValueError(f"centres shape {tuple(c.shape)} does not match X with {d} features")
    k = int(c.shape[0])
    out = torch.empty((n, k), dtype=torch.float32 if out_f32 else torch.float64, device=Xb.device)
    ctx = _Ctx(Xb.device)
    ctx.check(ctx.lib.ofc_kmeans_distances(_ptr(Xb), _DT[Xb.dtype], C.c_int64(n), d, k, _ptr(c), _ptr(out), int(out_f32),
                                           ctx.stream()))
    return out


def _estimator_transform(est, X):
    """``transform`` of KMeans and MiniBatchKMeans: the feature-count check, the centres sklearn's ``cluster_centers_``
    holds (float32 after a float32 fit), and numpy out for anything but a torch tensor in"""
    d = int(X.shape[1]) if np.ndim(X) == 2 else None
    if d is not None and d != est.n_features_in_:
        raise ValueError(f"X has {d} features, but {type(est).__name__} is expecting {est.n_features_in_} features as input.")
    centres = est._centres_t.to(torch.float32) if est._f32 else est._centres_t
    out = transform(X, centres)
    return out if isinstance(X, torch.Tensor) else out.cpu().numpy()


def kmeans_plusplus(X, n_clusters: int, random_state=None, sample_weight=None):
    """k-means++ seeding with sklearn's procedure and RNG call sequence
    (sklearn/cluster/_kmeans.py:181-268): first centre by ``random_state.choice``, then
    ``2 + int(log(k))`` candidates per step sampled in proportion to the squared distance to
    the closest chosen centre, keeping the candidate that lowers the potential most.
    Distances come from the E-step kernel (one candidate = a one-centre problem).
    X ``[n, d]``; returns ``(centres float64 [k,d] tensor, indices)``.  ``sample_weight`` ``[n]``: the first centre is
    drawn with ``p = w / w.sum()``, the potentials are ``closest @ w`` and the candidates are sampled from
    ``cumsum(w * closest)``, as sklearn does (a row of weight 0 is never a seed).

    The reference leaves ``random_state`` unset (KmeanGrids.py:300), so this seeding is not
    pinned by any reference output (SURVEY.md Q9)."""
    Xb, single = _as_batch(X, _target_device(X))
    if not single:
        raise ValueError("kmeans_plusplus takes one problem [n, d]")
    ctx = _Ctx(Xb.device)
    rs = random_state if isinstance(random_state, np.random.RandomState) else np.random.RandomState(random_state)
    n, d = int(Xb.shape[1]), int(Xb.shape[2])
    k = int(n_clusters)
    w_host = _check_sample_weight(sample_weight, n, Xb.dtype)
    w = None if w_host is None else torch.from_numpy(w_host.astype(np.float64)).to(Xb.device)
    st = LloydState(ctx, Xb, 1)
    trials = 2 + int(math.log(k))
    Xf = Xb[0]
    centres = torch.empty((k, d), dtype=torch.float64, device=Xb.device)
    indices = np.full(k, -1, dtype=np.int64)
    cid = int(rs.choice(n, p=np.full(n, 1.0 / n) if w is None else w_host / w_host.sum()))
    centres[0] = Xf[cid].to(torch.float64)
    indices[0] = cid
    closest = torch.empty((1, n), dtype=torch.float64, device=Xb.device)
    cand = torch.empty((1, n), dtype=torch.float64, device=Xb.device)
    st.assign(None, centres[0:1].unsqueeze(0).contiguous(), st.labels[0], min_dist=closest)
    pot = float((closest.sum() if w is None else (closest * w).sum()).item())
    for c in range(1, k):
        rand_vals = rs.uniform(size=trials) * pot
        cum = torch.cumsum(closest[0] if w is None else closest[0] * w, dim=0)
        ids = torch.searchsorted(cum, torch.from_numpy(rand_vals).to(Xb.device)).clamp_(max=n - 1).cpu().numpy()
        best = None
        for cidx in ids:
            st.assign(None, Xf[int(cidx)].to(torch.float64).view(1, 1, d).contiguous(), st.labels[0], min_dist=cand)
            dmin = torch.minimum(closest, cand)
            p = float((dmin.sum() if w is None else (dmin * w).sum()).item())
            if best is None or p < best[0]:
                best = (p, int(cidx), dmin)
        pot, cid, closest = best[0], best[1], best[2].contiguous()
        centres[c] = Xf[cid].to(torch.float64)
        indices[c] = cid
    return centres, indices


def kmeans_plusplus_starts(X, n_clusters: int, n_starts: int, random_state, sample_weight=None):
    """The k-means++ seeds of ``n_starts`` starts of one fit, the same as ``n_starts`` calls of
    :func:`kmeans_plusplus` one after another on one ``RandomState`` -- computed in lockstep on the device, without
    a host round trip until the seeds are done.  X ``[n, d]`` on the compute device; returns ``(centres float64
    [R, k, d] tensor, indices int64 [R, k])``.

    The host first makes every start's RNG calls in sklearn's order (one ``choice`` and k - 1 ``uniform(size=T)``
    per start: how many numbers they draw does not depend on the data).  Each of the k - 1 steps then computes the
    distances of all R*T candidates in ONE E-step call (a shared-row batch of one-centre problems), and every start
    runs the torch operations of :func:`kmeans_plusplus` on tensors of the same shapes, each in an allocation of its
    own (a reduction may order its sum by the data's alignment), so a start's seeds do not depend on R.
    ``sample_weight`` ``[n]``: the weighted seeding of :func:`kmeans_plusplus`, with the same operations."""
    Xb, single = _as_batch(X, _target_device(X))
    if not single:
        raise ValueError("kmeans_plusplus_starts takes one problem [n, d]")
    ctx = _Ctx(Xb.device)
    rs = random_state if isinstance(random_state, np.random.RandomState) else np.random.RandomState(random_state)
    n, d = int(Xb.shape[1]), int(Xb.shape[2])
    k, R = int(n_clusters), int(n_starts)
    trials = 2 + int(math.log(k))
    dev = Xb.device
    w_host = _check_sample_weight(sample_weight, n, Xb.dtype)
    w = None if w_host is None else torch.from_numpy(w_host.astype(np.float64)).to(dev)
    first = np.empty(R, np.int64)
    uni = np.empty((R, max(k - 1, 1), trials))
    for r in range(R):
        first[r] = rs.choice(n, p=np.full(n, 1.0 / n) if w is None else w_host / w_host.sum())
        for c in range(1, k):
            uni[r, c - 1] = rs.uniform(size=trials)
    uni = torch.from_numpy(uni).to(dev)
    Xf = Xb[0]
    idx = torch.empty((R, k), dtype=torch.int64, device=dev)
    idx[:, 0] = torch.from_numpy(first).to(dev)
    st = LloydState(ctx, Xb, 1, shared_batch=R)
    dist0 = torch.empty((R, n), dtype=torch.float64, device=dev)
    st.assign(None, Xf[idx[:, 0]].to(torch.float64).view(R, 1, d).contiguous(), st.labels[0], min_dist=dist0)
    closest = [dist0[r:r + 1].clone() for r in range(R)]
    pot = [cl.sum() if w is None else (cl * w).sum() for cl in closest]
    if k > 1:
        cst = LloydState(ctx, Xb, 1, shared_batch=R * trials)
        cand = torch.empty((R * trials, n), dtype=torch.float64, device=dev)
    for c in range(1, k):
        ids = []
        for r in range(R):
            rand_vals = uni[r, c - 1] * pot[r]
            cum = torch.cumsum(closest[r][0] if w is None else closest[r][0] * w, dim=0)
            ids.append(torch.searchsorted(cum, rand_vals).clamp_(max=n - 1))
        ids = torch.cat(ids)
        cst.assign(None, Xf[ids].to(torch.float64).view(R * trials, 1, d).contiguous(), cst.labels[0], min_dist=cand)
        for r in range(R):
            dmin = [torch.minimum(closest[r], cand[r * trials + t:r * trials + t + 1]) for t in range(trials)]
            p = torch.stack([dm.sum() if w is None else (dm * w).sum() for dm in dmin])
            best = torch.argmin(p).view(1)                     # the first of the smallest, as the strict `<` of the loop
            pot[r] = p[best][0]
            closest[r] = torch.stack(dmin).index_select(0, best)[0]
            idx[r, c] = ids[r * trials:(r + 1) * trials][best][0]
    return Xf[idx].to(torch.float64), idx.cpu().numpy()


def _is_same_clustering(labels1, labels2, k: int) -> bool:
    """sklearn's ``_is_same_clustering`` (_k_means_common.pyx:314-328): the map from ``labels1`` to ``labels2``, taken
    at the first row of every cluster of ``labels1``, is a function on all rows (not necessarily a bijection)."""
    n = int(labels1.shape[0])
    a = labels1.long()
    first = torch.full((k,), n, dtype=torch.int64, device=a.device)
    first.scatter_reduce_(0, a, torch.arange(n, device=a.device), reduce="amin")
    return bool(torch.equal(labels2[first[a]], labels2))


def best_start(labels, inertia, k: int) -> int:
    """sklearn's choice among the starts of one fit (_kmeans.py:1534-1543): start i replaces the best so far only if its
    inertia is strictly lower and its clustering is not the same (:func:`_is_same_clustering`)."""
    inert = inertia.cpu().numpy()
    best = 0
    for i in range(1, len(inert)):
        if inert[i] < inert[best] and not _is_same_clustering(labels[i], labels[best], k):
            best = i
    return best


def _resolve_n_init(n_init, init, default_n_init: int = 10) -> int:
    """sklearn's ``_check_params_vs_input`` (_kmeans.py:884-907): "auto" is 1 for k-means++ and an array,
    ``default_n_init`` for "random" (10 for KMeans, 3 for MiniBatchKMeans); an array with n_init != 1 warns and runs
    one start."""
    if isinstance(n_init, str):
        if n_init != "auto":
            raise ValueError(f"n_init must be 'auto' or an int >= 1, got {n_init!r}")
        r = default_n_init if isinstance(init, str) and init == "random" else 1
    else:
        if isinstance(n_init, bool) or not isinstance(n_init, (int, np.integer)) or n_init < 1:
            raise ValueError(f"n_init must be 'auto' or an int >= 1, got {n_init!r}")
        r = int(n_init)
    if not isinstance(init, str) and r != 1:
        import warnings
        warnings.warn("Explicit initial center position passed: performing only one init in KMeans instead of "
                      f"n_init={r}.", RuntimeWarning, stacklevel=3)
        r = 1
    return r


def random_starts(X, n_clusters: int, n_starts: int, random_state, sample_weight=None):
    """``init="random"`` (_kmeans.py:1030-1036): per start, ``choice(n, size=k, replace=False, p=w / w.sum())`` with
    ``w`` = ``sample_weight`` (ones when None) in the data's working dtype (float32 for float32 rows, else float64).
    Returns (centres float64 [R, k, d] tensor on X's device, indices int64 [R, k])."""
    Xb, _ = _as_batch(X, _target_device(X))
    rs = random_state if isinstance(random_state, np.random.RandomState) else np.random.RandomState(random_state)
    n = int(Xb.shape[1])
    w = _check_sample_weight(sample_weight, n, Xb.dtype)
    if w is None:
        w = np.ones(n, dtype=np.float32 if Xb.dtype == torch.float32 else np.float64)
    idx = np.stack([rs.choice(n, size=int(n_clusters), replace=False, p=w / w.sum()) for _ in range(int(n_starts))])
    return Xb[0][torch.from_numpy(idx).to(Xb.device)].to(torch.float64), idx.astype(np.int64)


class KMeans:
    """The subset of ``sklearn.cluster.KMeans`` the reference uses (KmeanGrids.py:299-304,
    color_kmeans.py:65-78): ``KMeans(n_clusters=k).fit(X)``, ``.predict(X)``,
    ``.cluster_centers_``, ``.labels_``, ``.inertia_``, ``.n_iter_``.  ``init`` may be
    ``'k-means++'`` (default, see :func:`kmeans_plusplus`), ``'random'`` or an array ``[k, d]``.

    ``n_init`` as scikit-learn 1.9: ``"auto"`` is one start for k-means++ and an array, 10 for ``"random"``.
    The starts draw their seeds one after another from one ``RandomState`` (so ``random_state=int`` reproduces
    sklearn), run as one batched Lloyd fit over a single copy of the rows, and the result is the start sklearn
    keeps: the first one, replaced by a later one only if that has a strictly lower inertia and a different
    clustering.

    ``fit(X, sample_weight=w)`` is sklearn's weighted fit (seeding, M-step, relocation and inertia weighted; see
    :func:`_check_sample_weight` for the accepted weights); :meth:`score` is its negative weighted inertia."""

    def __init__(self, n_clusters=8, *, init="k-means++", n_init="auto", max_iter=300, tol=1e-4, random_state=None):
        self.n_clusters, self.init, self.n_init = int(n_clusters), init, n_init
        self.max_iter, self.tol, self.random_state = int(max_iter), float(tol), random_state

    def fit(self, X, y=None, sample_weight=None):
        Xa = X if isinstance(X, torch.Tensor) else np.asarray(X)
        if Xa.ndim != 2:
            raise ValueError("Expected 2D array")
        if Xa.shape[0] < self.n_clusters:
            raise ValueError(f"n_samples={Xa.shape[0]} should be >= n_clusters={self.n_clusters}.")
        sw = _check_sample_weight(sample_weight, int(Xa.shape[0]), Xa.dtype)
        if isinstance(self.init, str) and self.init not in ("k-means++", "random"):
            raise ValueError(f"init={self.init!r}: 'k-means++', 'random' or an array")
        n_init = _resolve_n_init(self.n_init, self.init)
        if isinstance(self.init, str) and self.n_clusters > 1 and (n_init > 1 or self.init == "random"):
            rs = (self.random_state if isinstance(self.random_state, np.random.RandomState)
                  else np.random.RandomState(self.random_state))
            Xd, _ = _as_batch(Xa, _target_device(Xa))
            Xd = Xd[0]
            if self.init == "random":
                init, _ = random_starts(Xd, self.n_clusters, n_init, rs, sw)
            else:
                init, _ = kmeans_plusplus_starts(Xd, self.n_clusters, n_init, rs, sw)
            labels, centres, inertia, n_iter = lloyd(Xd, init, self.max_iter, self.tol, sample_weight=sw)
            b = best_start(labels, inertia, self.n_clusters)
            labels, centres, inertia, n_iter = labels[b], centres[b], inertia[b], n_iter[b]
        else:
            if isinstance(self.init, str):
                if self.n_clusters == 1:
                    init = (Xa[:1].to(torch.float64) if isinstance(Xa, torch.Tensor) else Xa[:1].astype(np.float64))
                else:
                    init, _ = kmeans_plusplus(Xa, self.n_clusters, self.random_state, sw)
            else:
                init = self.init
            labels, centres, inertia, n_iter = lloyd(Xa, init, self.max_iter, self.tol, sample_weight=sw)
        self._centres_t = centres
        # a float32 fit: sklearn's cluster_centers_ are float32, and transform measures against those
        self._f32 = Xa.dtype == (torch.float32 if isinstance(Xa, torch.Tensor) else np.float32)
        self.n_features_in_ = int(Xa.shape[1])
        self.cluster_centers_ = centres.cpu().numpy()
        if not isinstance(X, torch.Tensor) and np.asarray(X).dtype == np.float32:
            self.cluster_centers_ = self.cluster_centers_.astype(np.float32)
        self.labels_ = labels.cpu().numpy()
        self.inertia_ = float(inertia.item())
        self.n_iter_ = int(n_iter.item())
        return self

    def predict(self, X):
        return predict(X, self._centres_t).cpu().numpy()

    def fit_predict(self, X, y=None, sample_weight=None):
        return self.fit(X, sample_weight=sample_weight).labels_

    def score(self, X, y=None, sample_weight=None):
        """sklearn's ``KMeans.score`` (_kmeans.py:1159-1187): minus the (weighted) inertia of X against the fitted centres,
        on the un-centred rows as :meth:`predict` assigns them."""
        return score(X, self._centres_t, sample_weight)

    def transform(self, X):
        """sklearn's ``KMeans.transform``: the ``[n, k]`` distances of X's rows to ``cluster_centers_`` (see
        :func:`transform`).  numpy in gives numpy out; a torch tensor in gives a tensor on the compute device."""
        return _estimator_transform(self, X)

    def fit_transform(self, X, y=None, sample_weight=None):
        return self.fit(X, sample_weight=sample_weight).transform(X)


def score(X, centres, sample_weight=None) -> float:
    """sklearn's ``score`` of KMeans and MiniBatchKMeans (_kmeans.py:1159-1187): minus the (weighted) inertia of X
    ``[n, d]`` against ``centres`` ``[k, d]``, on the un-centred rows as :func:`predict` assigns them."""
    Xb, single = _as_batch(X, _target_device(X))
    if not single:
        raise ValueError("Expected 2D array")
    n = int(Xb.shape[1])
    w = _check_sample_weight(sample_weight, n, Xb.dtype)
    w = None if w is None else torch.from_numpy(w.astype(np.float64)).to(Xb.device)
    c = centres.to(device=Xb.device, dtype=torch.float64).unsqueeze(0).contiguous()
    st = LloydState(_Ctx(Xb.device), Xb, int(c.shape[1]), weights=w)
    st.assign(None, c, st.labels[0], inertia=st.inertia)
    return -float(st.inertia[0].item())


def kmeans_fit(X, init, max_iter: int = 300, tol: float = 1e-4, sample_weight=None):
    """SURVEY.md §8(b) parity entry point: numpy in / numpy out
    ``(labels int32[N], centers[k,D], inertia, n_iter)``; ``sample_weight`` as in :func:`lloyd`."""
    labels, centres, inertia, n_iter = lloyd(X, init, max_iter, tol, sample_weight=sample_weight)
    return labels.cpu().numpy(), centres.cpu().numpy(), float(inertia.item()), int(n_iter.item())
