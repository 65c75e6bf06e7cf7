"""MiniBatchKMeans on the GPU: the clustering behind the reference's colour quantisation script

    clt = MiniBatchKMeans(n_clusters = args["clusters"]); labels = clt.fit_predict(image)
    quant = clt.cluster_centers_.astype("uint8")[labels]            (color-quantization/quant.py:18-20)

following scikit-learn 1.9.0's ``MiniBatchKMeans.fit`` step for step (sklearn/cluster/_kmeans.py:2056-2227,
``_mini_batch_step`` :1566-1684, ``_mini_batch_convergence`` :1974-2037, ``_random_reassign`` :2039-2054,
``_minibatch_update_dense`` in _k_means_minibatch.pyx) including the order of its ``RandomState`` calls, so that
``MiniBatchKMeans(n_clusters=k, random_state=int)`` reproduces scikit-learn on uint8 rows (the script's LAB pixels):
same mini-batches, same seeds, same centres, same labels.

Where the work runs: the rows stay on the device; per step the mini-batch is gathered on the device, labelled by the
E-step kernel (``ofc_kmeans_assign``: ||c||^2 - 2 x.c, first strict minimum) and folded into the centres by
``ofc_minibatch_update`` in the reference's accumulation order.  The host keeps sklearn's bookkeeping -- the random
stream (numpy ``RandomState``, as sklearn), the smoothed-inertia early stopping and the low-count reassignment -- and
reads back k + 1 numbers per step.  torch is used for device memory only.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import kmeans as _km
from .kmeans import LloydState, _as_batch, _Ctx, _ptr, _target_device


class MiniBatchKMeans:
    """The subset of ``sklearn.cluster.MiniBatchKMeans`` the reference uses, and its streaming and weighted calls:
    constructor keywords, ``fit``, ``fit_predict``, ``partial_fit``, ``predict``, ``score``, ``cluster_centers_``,
    ``labels_``, ``inertia_``, ``n_steps_``, ``n_iter_``.  ``init`` is ``'k-means++'``, ``'random'`` or an array
    ``[k, d]``; ``n_init="auto"`` is one start for k-means++ and an array, 3 for ``'random'``.

    ``sample_weight`` (see :func:`kmeans._check_sample_weight`): ``fit`` seeds with the weights, draws its mini-batches
    in proportion to them and steps with unit weights, as sklearn; ``partial_fit`` steps with the caller's weights
    (``ofc_minibatch_update_weighted``).  ``partial_fit(X)`` runs one mini-batch step on all of X: the first call
    seeds, later calls continue the same centres, counts and random stream.  CUDA tensors in keep the rows, centres
    and labels on the device (``cluster_centers_`` and ``labels_`` are then tensors); numpy in gives numpy out."""

    def __init__(self, n_clusters=8, *, init="k-means++", max_iter=100, batch_size=1024, compute_labels=True,
                 random_state=None, tol=0.0, max_no_improvement=10, init_size=None, n_init="auto", reassignment_ratio=0.01):
        self.n_clusters, self.init, self.max_iter, self.batch_size = int(n_clusters), init, int(max_iter), int(batch_size)
        self.compute_labels, self.random_state, self.tol = bool(compute_labels), random_state, float(tol)
        self.max_no_improvement, self.init_size, self.n_init = max_no_improvement, init_size, n_init
        self.reassignment_ratio = float(reassignment_ratio)
        if self.reassignment_ratio < 0:
            raise ValueError(f"reassignment_ratio should be >= 0, got {self.reassignment_ratio} instead.")

    # -- helpers ---------------------------------------------------------------------------------------------
    def _labels_inertia(self, st: LloydState, centres: torch.Tensor, labels: torch.Tensor):
        st.assign(None, centres.view(1, self.n_clusters, -1), labels, inertia=st.inertia)
        return st.inertia

    @property
    def _counts(self):
        """the clusters' weight sums (sklearn's ``_counts``, in the rows' working dtype)"""
        c = self._counts_t.cpu().numpy()
        return c.astype(np.float32) if self._f32 else c

    def _check_params_vs_input(self, X: torch.Tensor):
        """_kmeans.py:1932-1962: the batch size, the init subset size and the rows' dtype and width"""
        n, k = int(X.shape[0]), self.n_clusters
        if n < k:
            raise ValueError(f"n_samples={n} should be >= n_clusters={k}.")
        if isinstance(self.init, str) and self.init not in ("k-means++", "random"):
            raise ValueError(f"init={self.init!r}: 'k-means++', 'random' or an array")
        self._batch_size = min(self.batch_size, n)
        init_size = self.init_size
        if init_size is None:
            init_size = 3 * self._batch_size
            if init_size < k:
                init_size = 3 * k
        elif init_size < k:
            init_size = 3 * k
        self._init_size = min(init_size, n)
        self._f32 = X.dtype == torch.float32
        self.n_features_in_ = int(X.shape[1])

    def _init_centroids(self, Xf: torch.Tensor, w, rs):
        """_init_centroids (:1000-1060): k-means++ or random seeds on a random subset of ``_init_size`` rows (with its
        weights), or the explicit array; float32 rows give float32-rounded centres"""
        n, k = int(Xf.shape[0]), self.n_clusters
        if isinstance(self.init, str):
            Xi, wi = Xf, w
            if self._init_size < n:
                init_idx = rs.randint(0, n, self._init_size)
                Xi = Xf.index_select(0, torch.from_numpy(init_idx).to(Xf.device)).contiguous()
                wi = None if w is None else w[init_idx]
            if self.init == "k-means++":
                centres, _ = _km.kmeans_plusplus(Xi, k, random_state=rs, sample_weight=wi)
            else:
                centres = _km.random_starts(Xi, k, 1, rs, wi)[0][0]
        else:
            centres = torch.as_tensor(np.asarray(self.init), dtype=torch.float64).to(Xf.device).clone()
        if self._f32:
            centres = centres.to(torch.float32).to(torch.float64)
        return centres.contiguous()

    def _random_reassign(self, counts_h) -> bool:
        """_random_reassign (:2039-2054), on the counts before the step"""
        self._n_since_last_reassign += self._batch_size
        if bool((counts_h == 0).any()) or self._n_since_last_reassign >= 10 * self.n_clusters:
            self._n_since_last_reassign = 0
            return True
        return False

    def _step(self, ctx, st, Xs, w_dev, centres, centres_new, rs, random_reassign, with_inertia):
        """_mini_batch_step (:1566-1684) on the rows of ``st``: labels (and the batch inertia) with the current centres,
        the centre update into ``centres_new`` (weighted when ``w_dev`` is given), then the low-count reassignment on
        the host.  Reads back the k counts (and the inertia); returns the batch inertia (0.0 without)."""
        k, lib = self.n_clusters, ctx.lib
        rows, d = int(Xs.shape[0]), int(Xs.shape[1])
        labels = st.labels[0]
        if with_inertia:
            inertia_t = self._labels_inertia(st, centres, labels)
        else:
            st.assign(None, centres.view(1, k, -1), labels)
        if w_dev is None:
            ctx.check(lib.ofc_minibatch_update(_ptr(Xs), st.dtype, rows, d, k, _ptr(labels), _ptr(centres), _ptr(centres_new),
                                               _ptr(self._counts_t), ctx.stream()))
        else:
            ctx.check(lib.ofc_minibatch_update_weighted(_ptr(Xs), st.dtype, rows, d, k, _ptr(labels), _ptr(w_dev), _ptr(centres),
                                                        _ptr(centres_new), _ptr(self._counts_t), ctx.stream()))
        host = (torch.cat([inertia_t.view(1), self._counts_t]) if with_inertia else self._counts_t).cpu().numpy()
        batch_inertia, counts_h = (float(host[0]), host[1:].copy()) if with_inertia else (0.0, host.copy())
        if random_reassign and self.reassignment_ratio > 0:
            to_reassign = counts_h < self.reassignment_ratio * counts_h.max()
            if to_reassign.sum() > 0.5 * rows:
                keep = np.argsort(counts_h)[int(0.5 * rows):]
                to_reassign[keep] = False
            n_re = int(to_reassign.sum())
            if n_re:
                new_rows = rs.choice(rows, replace=False, size=n_re)
                sel = Xs.index_select(0, torch.from_numpy(np.asarray(new_rows, dtype=np.int64)).to(Xs.device)).to(torch.float64)
                centres_new[torch.from_numpy(np.nonzero(to_reassign)[0]).to(Xs.device)] = sel
            counts_h[to_reassign] = np.min(counts_h[~to_reassign])
            self._counts_t.copy_(torch.from_numpy(counts_h))
        self._counts_h = counts_h
        return batch_inertia

    def fit(self, X, y=None, sample_weight=None):
        Xb, single = _as_batch(X, _target_device(X))
        if not single:
            raise ValueError("Expected 2D array")
        ctx = _Ctx(Xb.device)
        dev = Xb.device
        Xf = Xb[0]
        n, d = int(Xf.shape[0]), int(Xf.shape[1])
        k = self.n_clusters
        self._check_params_vs_input(Xf)
        bs = self._batch_size
        is_f32 = self._f32
        w = _km._check_sample_weight(sample_weight, n, Xf.dtype)
        n_init = _km._resolve_n_init(self.n_init, self.init, default_n_init=3)
        tol_ = 0.0
        if self.tol != 0:
            mean, var, _ = _km.column_mean_var(LloydState(ctx, Xb, 1))
            tol_ = float(var.mean().item()) * self.tol
        rs = self.random_state if isinstance(self.random_state, np.random.RandomState) else np.random.RandomState(self.random_state)

        # validation set for the init (:2110-2112); drawn even when a single init makes it unused
        valid_idx = rs.randint(0, n, self._init_size)
        best = None
        for _ in range(n_init):
            centres = self._init_centroids(Xf, w, rs)
            if n_init > 1:
                Xv = Xf.index_select(0, torch.from_numpy(valid_idx).to(dev)).contiguous().unsqueeze(0)
                wv = None if w is None else torch.from_numpy(w[valid_idx].astype(np.float64)).to(dev)
                stv = LloydState(ctx, Xv, k, weights=wv)
                inertia = float(self._labels_inertia(stv, centres, stv.labels[0]).item())
                if best is None or inertia < best[0]:
                    best = (inertia, centres)
            else:
                best = (0.0, centres)
        centres = best[1].contiguous()
        centres_new = torch.empty_like(centres)
        self._counts_t = torch.zeros(k, dtype=torch.float64, device=dev)     # X.dtype in sklearn; float32 values stay exact
        self._n_since_last_reassign = 0

        # the weighted sampling of the mini-batches (:2165-2170) is RandomState.choice(n, bs, p=w / w.sum()): a cumulative
        # table (the same every step) searched with `bs` uniform draws -- the table is built once, the draws are numpy's
        if w is None:
            p = np.ones(n, dtype=np.float64) / float(n)
            sum_of_weights = n
        else:
            sum_of_weights = np.sum(w)
            p = (w / sum_of_weights).astype(np.float64)
        cdf = p.cumsum()
        cdf /= cdf[-1]

        Xmb = torch.empty((1, bs, d), dtype=Xf.dtype, device=dev)
        st = LloydState(ctx, Xmb, k)
        ewa, ewa_min, no_improvement = None, None, 0
        self._counts_h = np.zeros(k)
        n_steps = (self.max_iter * n) // bs
        step = -1
        for step in range(n_steps):
            idx = cdf.searchsorted(rs.random_sample(bs), side="right")
            torch.index_select(Xf, 0, torch.from_numpy(np.asarray(idx, dtype=np.int64)).to(dev), out=Xmb[0])
            random_reassign = self._random_reassign(self._counts_h)
            batch_inertia = self._step(ctx, st, Xmb[0], None, centres, centres_new, rs, random_reassign, True)
            sq_diff = float(((centres_new - centres) ** 2).sum().item()) if tol_ > 0.0 else 0.0
            centres, centres_new = centres_new, centres
            # _mini_batch_convergence (:1974-2037)
            batch_inertia /= bs
            if step + 1 == 1:
                continue
            if ewa is None:
                ewa = batch_inertia
            else:
                alpha = min(bs * 2.0 / (n + 1), 1)
                ewa = ewa * (1 - alpha) + batch_inertia * alpha
            if tol_ > 0.0 and sq_diff <= tol_:
                break
            if ewa_min is None or ewa < ewa_min:
                no_improvement, ewa_min = 0, ewa
            else:
                no_improvement += 1
            if self.max_no_improvement is not None and no_improvement >= self.max_no_improvement:
                break
        self._centres_t = centres.clone()
        self.cluster_centers_ = centres.cpu().numpy()
        if is_f32:
            self.cluster_centers_ = self.cluster_centers_.astype(np.float32)
        self.n_steps_ = step + 1
        self.n_iter_ = int(np.ceil(((step + 1) * bs) / n))
        if self.compute_labels:
            wf = None if w is None else torch.from_numpy(w.astype(np.float64)).to(dev)
            stf = LloydState(ctx, Xb, k, weights=wf)
            inertia = self._labels_inertia(stf, centres, stf.labels[0])
            self._labels_t = stf.labels[0][0]
            self.labels_ = self._labels_t.cpu().numpy()
            self.inertia_ = float(inertia.item())
        else:
            self.inertia_ = float(ewa * sum_of_weights) if ewa is not None else 0.0
        return self

    def partial_fit(self, X, y=None, sample_weight=None):
        """sklearn's ``partial_fit`` (_kmeans.py:2227-2329): one mini-batch step on all rows of X with the caller's
        weights.  The first call (no centres yet) sizes the batch and init subset from this X, takes the random stream
        from ``random_state`` (kept across calls, and not reset by :meth:`fit`) and seeds once; every call then steps,
        and with ``compute_labels`` sets ``labels_`` / ``inertia_`` of X against the new centres."""
        as_tensor = isinstance(X, torch.Tensor)
        Xb, single = _as_batch(X, _target_device(X))
        if not single:
            raise ValueError("Expected 2D array")
        ctx = _Ctx(Xb.device)
        dev = Xb.device
        Xf = Xb[0]
        n, d = int(Xf.shape[0]), int(Xf.shape[1])
        k = self.n_clusters
        has_centres = hasattr(self, "_centres_t")
        if has_centres and d != self.n_features_in_:
            raise ValueError(f"X has {d} features, but MiniBatchKMeans is expecting {self.n_features_in_} features as input.")
        if not hasattr(self, "_random_state"):
            self._random_state = (self.random_state if isinstance(self.random_state, np.random.RandomState)
                                  else np.random.RandomState(self.random_state))
        rs = self._random_state
        w = _km._check_sample_weight(sample_weight, n, Xf.dtype)
        self.n_steps_ = getattr(self, "n_steps_", 0)
        if not has_centres:
            self._check_params_vs_input(Xf)
            self._centres_t = self._init_centroids(Xf, w, rs)
            self._counts_t = torch.zeros(k, dtype=torch.float64, device=dev)
            self._counts_h = np.zeros(k)
            self._n_since_last_reassign = 0
        w_dev = None if w is None else torch.from_numpy(w.astype(np.float64)).to(dev)
        st = LloydState(ctx, Xb, k, weights=w_dev)
        centres = self._centres_t.to(dev)
        centres_new = torch.empty_like(centres)
        self._step(ctx, st, Xf, w_dev, centres, centres_new, rs, self._random_reassign(self._counts_h), False)
        self._centres_t = centres_new
        if self.compute_labels:
            inertia = self._labels_inertia(st, centres_new, st.labels[1])
            self._labels_t = st.labels[1][0]
            self.labels_ = self._labels_t if as_tensor else self._labels_t.cpu().numpy()
            self.inertia_ = float(inertia.item())
        self.n_steps_ += 1
        if as_tensor:
            self.cluster_centers_ = centres_new.to(torch.float32) if self._f32 else centres_new
        else:
            self.cluster_centers_ = centres_new.cpu().numpy().astype(np.float32 if self._f32 else np.float64)
        return self

    def fit_predict(self, X, y=None, sample_weight=None):
        return self.fit(X, sample_weight=sample_weight).labels_

    def predict(self, X):
        return _km.predict(X, self._centres_t).cpu().numpy()

    def score(self, X, y=None, sample_weight=None):
        """minus the (weighted) inertia of X against the centres (sklearn's ``score``, shared with KMeans)"""
        return _km.score(X, self._centres_t, sample_weight)


def quantize(image_lab, n_clusters, random_state=None):
    """quant.py:15-20 on an image that is already in LAB (uint8 [H, W, 3], numpy or CUDA tensor): returns
    ``(labels [H*W], quantised image uint8 [H, W, 3])``; ``cluster_centers_.astype('uint8')[labels]`` is gathered on the
    device."""
    h, w = int(image_lab.shape[0]), int(image_lab.shape[1])
    flat = image_lab.reshape(h * w, 3)
    clt = MiniBatchKMeans(n_clusters=n_clusters, random_state=random_state)
    clt.fit(flat)
    cen_u8 = clt._centres_t.to(torch.uint8)                       # .astype("uint8"): truncation, values are in 0..255
    quant = cen_u8.index_select(0, clt._labels_t.long()).reshape(h, w, 3)
    if isinstance(image_lab, torch.Tensor):
        return clt._labels_t, quant
    return clt.labels_, quant.cpu().numpy()
