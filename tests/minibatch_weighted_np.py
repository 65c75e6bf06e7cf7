"""CPU restatement of scikit-learn 1.9.0 MiniBatchKMeans with its state (test infrastructure only; the product never
imports it): ``fit`` with sample weights, ``init="k-means++"`` / ``"random"`` / an array and ``n_init``, and
``partial_fit``, RandomState call for RandomState call, plus the centre update as a left fold.

The arithmetic is in the third-party wheel scikit-learn 1.9.0:
  sklearn/cluster/_kmeans.py:2056-2225            fit(): validation set, init on a random subset, weighted sampling
  sklearn/cluster/_kmeans.py:2227-2329            partial_fit(): the state kept across calls
  sklearn/cluster/_kmeans.py:1566-1684            _mini_batch_step (labels, update, low-count reassignment)
  sklearn/cluster/_k_means_minibatch.pyx:60-110   update_center_dense
The unit-weight ``fit`` of the reference's colour quantisation is restated in oracle/minibatch_np.py; this module
reproduces its results (tests/golden/minibatch_sklearn.npz) and is pinned by tests/golden/minibatch_sklearn_weighted.npz,
whose generator (tests/golden/make_minibatch_weighted_golden.py) checks it against sklearn.
"""
from __future__ import annotations

import numpy as np

from oracle import kmeans_np


def _kmeans_plusplus(X, k, rs, w):
    """sklearn/cluster/_kmeans.py:181-268 with sample weights ``w`` (float64 rows): first centre by
    ``choice(n, p=w / w.sum())``, potentials ``closest @ w``, candidates from ``cumsum(w * closest)``."""
    n = X.shape[0]
    trials = 2 + int(np.log(k))
    centers = np.empty((k, X.shape[1]), X.dtype)
    cid = rs.choice(n, p=w / w.sum())
    centers[0] = X[cid]
    closest = ((X - centers[0]) ** 2).sum(axis=1)
    pot = closest @ w
    for c in range(1, k):
        rand_vals = rs.uniform(size=trials) * pot
        ids = np.searchsorted(np.cumsum(w * closest), rand_vals)
        np.clip(ids, None, n - 1, out=ids)
        d2 = np.stack([((X - X[i]) ** 2).sum(axis=1) for i in ids])
        np.minimum(closest, d2, out=d2)
        pots = d2 @ w
        best = int(np.argmin(pots))
        pot, closest = pots[best], d2[best]
        centers[c] = X[ids[best]]
    return centers


def update_fold(X, labels, w, c_old, ws):
    """_minibatch_update_dense (_k_means_minibatch.pyx:60-110) as a left fold, the oracle of every kernel form of
    ofc_minibatch_update[_weighted]: per cluster, wsum = the members' weights folded from 0 in batch order (in the working
    type W: float32 for float32 rows, else float64); if wsum > 0, the centre is the fold of c_old * ws and the members'
    x * w, times 1 / (ws + wsum), and ws += wsum; else centre and weight sum stay.  ``w`` None: unit weights.
    Returns (new centres float64 [k, d], new weight sums float64 [k])."""
    W = np.float32 if X.dtype == np.float32 else np.float64
    Xw = np.asarray(X).astype(W)
    ww = np.ones(len(Xw), W) if w is None else np.asarray(w).astype(W)
    c_new, ws_new = np.array(c_old, np.float64), np.array(ws, np.float64)
    for j in range(c_new.shape[0]):
        m = np.nonzero(labels == j)[0]
        wsum = np.add.accumulate(np.r_[np.zeros(1, W), ww[m]])[-1]
        if wsum > 0:
            start = np.asarray(c_old[j]).astype(W) * W(ws[j])
            acc = np.add.accumulate(np.vstack([start[None], Xw[m] * ww[m][:, None]]), axis=0)[-1]
            ws_new[j] = W(ws[j]) + wsum
            c_new[j] = acc * (W(1) / W(ws_new[j]))
    return c_new, ws_new


class MiniBatch:
    """``sklearn.cluster.MiniBatchKMeans`` restated with its state: :meth:`fit` and :meth:`partial_fit` on dense uint8,
    float32 or float64 rows (worked in W = float32 for float32 rows, else float64), with sample weights,
    ``init="k-means++"`` / ``"random"`` / an array and ``n_init`` (``"auto"``: 1 for k-means++, 3 for random)."""

    def __init__(self, n_clusters, random_state=None, init="k-means++", n_init="auto", max_iter=100, batch_size=1024,
                 compute_labels=True, tol=0.0, max_no_improvement=10, init_size=None, reassignment_ratio=0.01):
        self.k, self.random_state, self.init, self.n_init = n_clusters, random_state, init, n_init
        self.max_iter, self.batch_size, self.compute_labels, self.tol = max_iter, batch_size, compute_labels, tol
        self.max_no_improvement, self.init_size, self.reassignment_ratio = max_no_improvement, init_size, reassignment_ratio

    def _prep(self, X, sample_weight):
        X = np.asarray(X)
        W = np.float32 if X.dtype == np.float32 else np.float64
        w = np.ones(len(X), W) if sample_weight is None else np.asarray(sample_weight).astype(W)
        return X.astype(W), w, W

    def _params(self, n):
        self._batch_size = min(self.batch_size, n)
        init_size = self.init_size
        if init_size is None:
            init_size = 3 * self._batch_size
            if init_size < self.k:
                init_size = 3 * self.k
        elif init_size < self.k:
            init_size = 3 * self.k
        self._init_size = min(init_size, n)
        if self.n_init == "auto":
            self._n_init = 3 if isinstance(self.init, str) and self.init == "random" else 1
        else:
            self._n_init = 1 if not isinstance(self.init, str) else self.n_init

    def _init_centroids(self, X, w, rs):
        n = X.shape[0]
        if not isinstance(self.init, str):
            return np.array(self.init, X.dtype)
        if self._init_size < n:
            idx = rs.randint(0, n, self._init_size)
            X, w = X[idx], w[idx]
        if self.init == "random":
            return X[rs.choice(X.shape[0], size=self.k, replace=False, p=w / w.sum())]
        c = _kmeans_plusplus(X.astype(np.float64), self.k, rs, w.astype(np.float64))
        return c.astype(X.dtype)

    def _labels_inertia(self, X, w, centers):
        labels = kmeans_np._e_step(X.astype(np.float64), centers.astype(np.float64))
        return labels, float((((X.astype(np.float64) - centers.astype(np.float64)[labels]) ** 2).sum(axis=1) * w).sum())

    def _random_reassign(self):
        self._n_since_last_reassign += self._batch_size
        if (self._counts == 0).any() or self._n_since_last_reassign >= 10 * self.k:
            self._n_since_last_reassign = 0
            return True
        return False

    def _step(self, X, w, centers, rs, reassign):
        labels, inertia = self._labels_inertia(X, w, centers)
        c_new, ws_new = update_fold(X, labels, w, centers, self._counts)
        counts = ws_new.astype(X.dtype)
        c_new = c_new.astype(X.dtype)
        if reassign and self.reassignment_ratio > 0:
            to_reassign = counts < self.reassignment_ratio * counts.max()
            if to_reassign.sum() > 0.5 * X.shape[0]:
                to_reassign[np.argsort(counts)[int(0.5 * X.shape[0]):]] = False
            if to_reassign.sum():
                c_new[to_reassign] = X[rs.choice(X.shape[0], replace=False, size=int(to_reassign.sum()))]
            counts[to_reassign] = np.min(counts[~to_reassign])
        self._counts = counts
        return c_new, inertia

    def fit(self, X, sample_weight=None):
        X, w, W = self._prep(X, sample_weight)
        n = X.shape[0]
        self._params(n)
        rs = self.random_state if isinstance(self.random_state, np.random.RandomState) else np.random.RandomState(self.random_state)
        tol = float(np.mean(np.var(X.astype(np.float64), axis=0)) * self.tol) if self.tol else 0.0
        valid = rs.randint(0, n, self._init_size)
        best = None
        for _ in range(self._n_init):
            c = self._init_centroids(X, w, rs)
            inertia = self._labels_inertia(X[valid], w[valid], c)[1]
            if best is None or inertia < best[0]:
                best = (inertia, c)
        centers = best[1]
        self._counts = np.zeros(self.k, W)
        self._n_since_last_reassign = 0
        ewa = ewa_min = None
        no_improvement = 0
        sum_w = np.sum(w)
        p = w / sum_w
        unit = np.ones(self._batch_size, W)
        bs = self._batch_size
        n_steps = (self.max_iter * n) // bs
        i = -1
        for i in range(n_steps):
            idx = rs.choice(n, bs, p=p, replace=True)
            c_new, inertia = self._step(X[idx], unit, centers, rs, self._random_reassign())
            sq = float(((c_new.astype(np.float64) - centers.astype(np.float64)) ** 2).sum()) if tol > 0 else 0.0
            centers = c_new
            batch_inertia = inertia / bs
            if i + 1 == 1:
                continue
            if ewa is None:
                ewa = batch_inertia
            else:
                alpha = min(bs * 2.0 / (n + 1), 1)
                ewa = ewa * (1 - alpha) + batch_inertia * alpha
            if tol > 0.0 and sq <= tol:
                break
            if ewa_min is None or ewa < ewa_min:
                no_improvement, ewa_min = 0, ewa
            else:
                no_improvement += 1
            if self.max_no_improvement is not None and no_improvement >= self.max_no_improvement:
                break
        self.cluster_centers_ = centers
        self.n_steps_ = i + 1
        if self.compute_labels:
            self.labels_, self.inertia_ = self._labels_inertia(X, w, centers)
        else:
            self.inertia_ = float(ewa * sum_w)
        return self

    def partial_fit(self, X, sample_weight=None):
        X, w, W = self._prep(X, sample_weight)
        has_centers = hasattr(self, "cluster_centers_")
        if not hasattr(self, "_random_state"):
            self._random_state = (self.random_state if isinstance(self.random_state, np.random.RandomState)
                                  else np.random.RandomState(self.random_state))
        rs = self._random_state
        self.n_steps_ = getattr(self, "n_steps_", 0)
        if not has_centers:
            self._params(X.shape[0])
            self.cluster_centers_ = self._init_centroids(X, w, rs)
            self._counts = np.zeros(self.k, W)
            self._n_since_last_reassign = 0
        self.cluster_centers_, _ = self._step(X, w, self.cluster_centers_, rs, self._random_reassign())
        if self.compute_labels:
            self.labels_, self.inertia_ = self._labels_inertia(X, w, self.cluster_centers_)
        self.n_steps_ += 1
        return self
