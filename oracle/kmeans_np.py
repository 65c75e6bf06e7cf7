"""CPU oracle: numpy restatement of scikit-learn 1.9.0 KMeans (lloyd, dense).

TEST INFRASTRUCTURE ONLY (see oracle/farneback_np.py header for the rule).

The reference calls ``KMeans(n_clusters=k).fit(X)`` then ``.predict(X)``
(k-means-color-clustering/KmeanGrids.py:299-304, color_kmeans.py:65-78).  The
arithmetic is in the third-party wheel scikit-learn 1.9.0 (not vendored, not
pinned by the reference); its Cython sources are readable on this image:
  sklearn/cluster/_kmeans.py:1463-1546     fit(): dtype promotion, tol, centring
  sklearn/cluster/_kmeans.py:627-758       _kmeans_single_lloyd loop / stopping
  sklearn/cluster/_k_means_lloyd.pyx:160-213  E-step: ||c||^2 - 2 x.c, first strict min
  sklearn/cluster/_k_means_common.pyx:167-311 relocate empty, average, shift
This file restates that algorithm (SURVEY.md Appendix A.5).

Parity pin: tests/test_oracle_kmeans.py against live sklearn with
``KMeans(init=C0, n_init=1)`` (k>1 is unpinned in the reference itself because
it never fixes random_state) and against the reference's k=1 goldens G1/G2/G4
(tests/golden/).
"""
from __future__ import annotations

import numpy as np


def _work_dtype(X: np.ndarray):
    return np.float32 if X.dtype == np.float32 else np.float64


def _e_step(X, centers):
    """labels = first strict minimum of ||c||^2 - 2 x.c  (ties -> lowest index)."""
    # sklearn: row_norms(centers, squared=True) == np.einsum("ij,ij->i", ...) -- its summation order (two interleaved
    # partial sums, no fma) differs from .sum(axis=1) in the last bit, which decides labels of rows that sit exactly on
    # a bisector (uint8 lattice data)
    c2 = np.einsum("ij,ij->i", centers, centers)
    n = X.shape[0]
    labels = np.empty(n, np.int32)
    chunk = 1 << 16
    for s in range(0, n, chunk):
        d = c2[None, :] - 2.0 * (X[s:s + chunk] @ centers.T)
        labels[s:s + chunk] = np.argmin(d, axis=1)
    return labels


def _m_step(X, labels, centers_old, sw=None):
    """sklearn's M-step on the centred rows: weighted sums and weight sums, _relocate_empty_clusters_dense, then
    _average_centers.  ``sw`` None = unit weights (the same bits: x * 1 == x)."""
    k, D = centers_old.shape
    if sw is None:
        w = np.bincount(labels, minlength=k).astype(X.dtype)
    else:
        w = np.bincount(labels, weights=sw, minlength=k).astype(X.dtype)
    sums = np.zeros((k, D), X.dtype)
    for d in range(D):
        sums[:, d] = np.bincount(labels, weights=X[:, d] if sw is None else X[:, d] * sw, minlength=k)
    # relocate empty clusters to the farthest points (_k_means_common.pyx:167-211): the clusters of weight 0 are listed
    # ONCE, before any move -- a cluster that a move empties stays empty -- and the n_empty farthest rows (unweighted
    # distance to the old centre of their label; largest first, ties to the lowest row index, DESIGN.md section 3) move
    # in, carrying x w and w
    empty = np.where(w == 0)[0]
    if empty.size:
        dist = ((X - centers_old[labels]) ** 2).sum(axis=1)
        if dist.max() > 0:
            far = np.lexsort((np.arange(dist.size), -dist))[:empty.size]
            for fi, new_id in zip(far, empty):
                old_id = labels[fi]
                wf = X.dtype.type(1.0) if sw is None else sw[fi]
                xw = X[fi] if sw is None else X[fi] * wf
                sums[old_id] -= xw
                sums[new_id] = xw
                w[new_id] = wf
                w[old_id] -= wf
    # _average_centers (:274-295) works in place in index order: an empty cluster copies row argmax(w) as it is at
    # that moment -- still the heaviest cluster's SUM when the empty cluster's index is the lower one
    new = sums.copy()
    amax = int(np.argmax(w))
    for j in range(k):
        if w[j] > 0:
            new[j] = new[j] * (X.dtype.type(1.0) / w[j])
        else:
            new[j] = new[amax]
    shift = np.sqrt(((new - centers_old) ** 2).sum(axis=1))
    return new, w, shift


def kmeans_fit(X, init, max_iter: int = 300, tol: float = 1e-4, sample_weight=None):
    """KMeans(n_clusters=k, init=init, n_init=1, max_iter, tol).fit(X, sample_weight=sample_weight).

    Returns ``(labels int32[N], centers[k,D], inertia, n_iter)`` with the
    semantics of ``labels_``, ``cluster_centers_``, ``inertia_``, ``n_iter_``.
    The weights enter the M-step sums, the relocation and the inertia; the
    column mean, the tolerance and the E-step stay unweighted, as in sklearn.
    """
    X = np.asarray(X)
    dt = _work_dtype(X)
    X = X.astype(dt)                                      # uint8 -> float64
    sw = None if sample_weight is None else np.asarray(sample_weight).astype(dt)
    centers = np.asarray(init).astype(dt).copy()
    tol_ = float(np.mean(np.var(X, axis=0)) * tol)        # _tolerance()
    mean = X.mean(axis=0)
    Xc = X - mean
    centers -= mean
    labels_old = np.full(X.shape[0], -1, np.int32)
    strict = False
    n_iter = 0
    labels = labels_old
    for it in range(max_iter):
        labels = _e_step(Xc, centers)
        new, w, shift = _m_step(Xc, labels, centers, sw)
        centers = new
        n_iter = it + 1
        if np.array_equal(labels, labels_old):
            strict = True
            break
        if float((shift ** 2).sum()) <= tol_:
            break
        labels_old = labels
    if not strict:
        labels = _e_step(Xc, centers)
    diff = Xc - centers[labels]
    if sw is None:
        inertia = float((diff * diff).sum())
    else:
        inertia = float(((diff * diff).sum(axis=1) * sw).sum())
    return labels, (centers + mean), inertia, n_iter


def kmeans_predict(X, centers):
    """KMeans.predict: E-step on the un-centred data (_kmeans.py:1075-1107)."""
    X = np.asarray(X)
    dt = _work_dtype(X)
    return _e_step(X.astype(dt), np.asarray(centers).astype(dt))


def rint_mean_exact(sum_int: np.ndarray, n: int) -> np.ndarray:
    """np.rint(sum/n) in exact integer arithmetic (round-half-even).

    For k = 1 the fitted centre is the column mean; sklearn's centred fp64
    computation is within ~1e-14 of sum/n and exact when sum/n is a half
    integer, so np.rint of it equals this integer rule (SURVEY.md H6; checked
    against sklearn in tests/test_oracle_kmeans.py).
    """
    s = np.asarray(sum_int, dtype=np.int64)
    q, r = np.divmod(s, n)
    up = (2 * r > n) | ((2 * r == n) & (q % 2 == 1))
    return q + up.astype(np.int64)


# ---------------------------------------------------------------------------------------------------
# k-means++ seeding of the DEVICE-RESIDENT per-cell fits (ofc_kmeans_cells / ofc_grid_kmeans_cells with
# init = NULL).  The procedure is scikit-learn's (sklearn/cluster/_kmeans.py:181-268: first centre uniform,
# then 2 + int(log k) candidates per step drawn in proportion to the squared distance to the closest chosen
# centre, keep the candidate with the lowest potential); the RANDOM STREAM is the build's own counter-based
# one (splitmix64 of (seed, problem index)) because the reference leaves random_state unset (SURVEY.md Q9),
# so there is no sklearn output to pin it to: this restatement in numpy integers is the independent check
# of the CUDA kernels' seeding.  The sklearn-RNG-exact seeding is kmeans.kmeans_plusplus (host loop).
# ---------------------------------------------------------------------------------------------------
_M64 = (1 << 64) - 1


def _splitmix64(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & _M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def cells_seed_indices(X: np.ndarray, k: int, seed: int, problem: int) -> np.ndarray:
    """Row indices the device-resident seeding picks for problem number ``problem`` (uint8 rows [n, d])."""
    import math
    Xi = X.astype(np.int64)
    n = Xi.shape[0]
    state = [_splitmix64((seed ^ ((0xD1B54A32D192ED03 * (problem + 1)) & _M64)) & _M64)]

    def uniform():
        state[0] = _splitmix64(state[0])
        return float(state[0] >> 11) * (1.0 / 9007199254740992.0)

    def dist_to(i):
        return ((Xi - Xi[i]) ** 2).sum(axis=1)

    trials = 2 + int(math.log(k))
    first = min(int(uniform() * float(n)), n - 1)
    idx = [first]
    closest = dist_to(first)
    for _ in range(1, k):
        pot = int(closest.sum())
        cum = np.cumsum(closest).astype(np.float64)           # exact: < 2^53
        cands = []
        for _t in range(trials):
            r = uniform() * float(pot)
            cands.append(min(int(np.searchsorted(cum, r, side="right")), n - 1))      # first row with r < running sum
        pots = [int(np.minimum(closest, dist_to(c)).sum()) for c in cands]
        best = cands[int(np.argmin(pots))]                    # first lowest
        idx.append(best)
        closest = np.minimum(closest, dist_to(best))
    return np.array(idx, np.int64)


def cells_fit(X: np.ndarray, k: int, seed: int, problem: int, max_iter: int = 300, tol: float = 1e-4):
    """One device-resident per-cell fit: seeding above, then :func:`kmeans_fit`.  Returns
    ``(labels, centers, inertia, n_iter, seed_indices)``."""
    idx = cells_seed_indices(X, k, seed, problem)
    lab, cen, inertia, n_iter = kmeans_fit(X, X[idx].astype(np.float64), max_iter=max_iter, tol=tol)
    return lab, cen, inertia, n_iter, idx


def dominant_centre_hue(X: np.ndarray, labels: np.ndarray, centers: np.ndarray):
    """Largest cluster (first on equal shares) -> np.rint -> uint8 BGR -> cv2 BGR2HSV hue
    (reference KmeanGrids.py:304-336)."""
    from . import viz_np
    counts = np.bincount(labels, minlength=centers.shape[0])
    c = np.rint(centers[int(np.argmax(counts))])
    hue = viz_np.bgr2hsv_u8(c[:3].astype(np.uint8).reshape(1, 1, 3))[0, 0, 0]
    return c, int(hue)
