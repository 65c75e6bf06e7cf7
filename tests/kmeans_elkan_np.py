"""numpy restatement of scikit-learn 1.9.0's dense Elkan k-means (sklearn/cluster/_kmeans.py:462-624 and
_k_means_elkan.pyx), the reference the ofc_kmeans_elkan_* kernels are tested against.

Every distance is ``_euclidean_dense_dense`` (_k_means_common.pyx:16-43) in the working dtype: the features in groups of
four, each group summed as ((d0^2 + d1^2) + d2^2) + d3^2 and added to the running total, the remainder one feature at a
time, every operation rounded on its own (numpy's elementwise operations never fuse), the square root in the working
dtype.  The functions work on many rows at once, but every row goes through exactly the loop sklearn runs for it (rows
are independent), so labels and bounds are sklearn's bits given the same centres and centre half-distances
(tests/golden/make_elkan_golden.py pins this against sklearn's own functions).
"""
from __future__ import annotations

import numpy as np

from oracle.kmeans_np import _m_step, _work_dtype


def euclidean(A, b, squared=False):
    """``_euclidean_dense_dense`` of every row of ``A`` [m, d] and the vector ``b`` [d], in their (common) dtype."""
    A = np.atleast_2d(A)
    dt = A.dtype
    d = A.shape[1]
    r = np.zeros(A.shape[0], dt)
    g = d // 4
    for q in range(g):
        t = 4 * q
        df = [A[:, t + u] - b[t + u] for u in range(4)]
        r = r + (((df[0] * df[0] + df[1] * df[1]) + df[2] * df[2]) + df[3] * df[3])
    for t in range(4 * g, d):
        df = A[:, t] - b[t]
        r = r + df * df
    return r if squared else np.sqrt(r)


def elkan_init(Xc, centers, chd):
    """``init_bounds_dense``: (labels int32 [n], upper [n], lower [n, k]) of the centred rows ``Xc`` [n, d]."""
    n, k = Xc.shape[0], centers.shape[0]
    dt = Xc.dtype
    lower = np.zeros((n, k), dt)
    best = np.zeros(n, np.int32)
    m = euclidean(Xc, centers[0])
    lower[:, 0] = m
    for j in range(1, k):
        sel = np.nonzero(m > chd[best, j])[0]
        if sel.size == 0:
            continue
        dj = euclidean(Xc[sel], centers[j])
        lower[sel, j] = dj
        take = dj < m[sel]
        m[sel[take]] = dj[take]
        best[sel[take]] = j
    return best, m, lower


def elkan_step(Xc, centers, chd, dnc, labels, upper, lower):
    """The label half of ``_update_chunk_dense`` over all rows, on copies: returns (labels, upper, lower, n_distances)."""
    labels, upper, lower = labels.copy(), upper.copy(), lower.copy()
    k = centers.shape[0]
    rows = np.nonzero(~(dnc[labels] >= upper))[0]
    tight = np.zeros(rows.size, bool)
    lab = labels[rows]
    ub = upper[rows]
    n_dist = 0
    for j in range(k):
        cond = (lab != j) & (ub > lower[rows, j]) & (ub > chd[lab, j])
        first = np.nonzero(cond & ~tight)[0]
        if first.size:
            for c in np.unique(lab[first]):
                s = first[lab[first] == c]
                ub[s] = euclidean(Xc[rows[s]], centers[c])
                lower[rows[s], c] = ub[s]
            tight[first] = True
            n_dist += first.size
        again = np.nonzero(cond & ((ub > lower[rows, j]) | (ub > chd[lab, j])))[0]
        if again.size:
            dj = euclidean(Xc[rows[again]], centers[j])
            lower[rows[again], j] = dj
            n_dist += again.size
            take = dj < ub[again]
            lab[again[take]] = j
            ub[again[take]] = dj[take]
    labels[rows] = lab
    upper[rows] = ub
    return labels, upper, lower, n_dist


def center_shift(old, new):
    """``_center_shift``: the per-centre distance between old and new centres"""
    return np.array([euclidean(new[j:j + 1], old[j])[0] for j in range(old.shape[0])], old.dtype)


def update_bounds(labels, upper, lower, shift):
    """the bound update at the end of ``elkan_iter_chunked_dense`` (on copies)"""
    upper = upper + shift[labels]
    lower = lower - shift[None, :]
    lower[lower < 0] = 0
    return upper, lower


def half_distances_direct(centers):
    """chd and dnc with the pairwise distances as the direct difference (the device's form, up to its fma rounding)"""
    diff = centers[:, None, :].astype(np.float64) - centers[None, :, :].astype(np.float64)
    chd = (np.sqrt((diff * diff).sum(-1)).astype(centers.dtype)) / centers.dtype.type(2)
    return chd, np.partition(chd, kth=1, axis=0)[1]


def elkan_fit(X, init, max_iter: int = 300, tol: float = 1e-4, sample_weight=None, half_distances=half_distances_direct):
    """``KMeans(algorithm="elkan", init=init, n_init=1, max_iter, tol).fit(X, sample_weight)``:
    ``(labels int32 [n], centers [k, d], inertia, n_iter)``.  ``half_distances(centers) -> (chd, dnc)`` gives the
    centre geometry (sklearn: ``euclidean_distances(centers) / 2`` and its second smallest per column)."""
    X = np.asarray(X)
    dt = _work_dtype(X)
    X = X.astype(dt)
    sw = None if sample_weight is None else np.asarray(sample_weight).astype(dt)
    tol_ = float(np.mean(np.var(X, axis=0)) * tol)
    mean = X.mean(axis=0)
    Xc = X - mean
    centers = np.asarray(init).astype(dt) - mean
    chd, dnc = half_distances(centers)
    labels, upper, lower = elkan_init(Xc, centers, chd)
    labels_old = np.full(X.shape[0], -1, np.int32)
    strict = False
    n_iter = 0
    for i in range(max_iter):
        labels, upper, lower, _ = elkan_step(Xc, centers, chd, dnc, labels, upper, lower)
        new, _, _ = _m_step(Xc, labels, centers, sw)
        shift = center_shift(centers, new)
        upper, lower = update_bounds(labels, upper, lower, shift)
        centers = new
        chd, dnc = half_distances(centers)
        n_iter = i + 1
        if np.array_equal(labels, labels_old):
            strict = True
            break
        if float((shift ** 2).sum()) <= tol_:
            break
        labels_old = labels
    if not strict:
        labels, upper, lower, _ = elkan_step(Xc, centers, chd, dnc, labels, upper, lower)
    sq = euclidean(Xc - centers[labels], np.zeros(X.shape[1], dt), squared=True)
    inertia = float(sq.astype(np.float64).sum() if sw is None else (sq * sw).astype(np.float64).sum())
    return labels, centers + mean, inertia, n_iter
