"""Generate tests/golden/kmeans_sklearn_elkan.npz: scikit-learn 1.9.0 ``KMeans(algorithm="elkan")`` results for the tests of
``KMeans(algorithm="elkan")`` and the ofc_kmeans_elkan_* kernels, and pin tests/kmeans_elkan_np.py against sklearn's own
functions on the way.

    python tests/golden/make_elkan_golden.py

Elkan merges its per-thread chunk sums under a lock in thread order, so the script runs with one OpenMP / BLAS thread (set
below, before numpy loads): more threads make sklearn's result depend on the schedule.  The rows are regenerated from each
case's name by ``elkan_case``, so the fixture stores only the results."""
from __future__ import annotations

import os

os.environ["OMP_NUM_THREADS"] = os.environ["OPENBLAS_NUM_THREADS"] = "1"

import sys  # noqa: E402

import numpy as np  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))

ELKAN_CASES = {   # name: (rows kind, n, d, k, init, n_init, random_state, weights, max_iter)
    "ties_u8_k7_s0": ("ties_u8", 4000, 3, 7, "k-means++", 1, 0, None, 300),
    "ties_u8_k7_s2": ("ties_u8", 4000, 3, 7, "k-means++", 1, 2, None, 300),
    "cell_u8_k8_pp10": ("cell_u8", 5852, 4, 8, "k-means++", 10, 3, None, 300),
    "blobs_u8_k8": ("blobs_u8", 6000, 4, 8, "k-means++", 1, 1, None, 300),
    "blobs_f32_k6_random3": ("blobs_f32", 3000, 8, 6, "random", 3, 2, None, 300),
    "blobs_f64_k5_pp2": ("blobs_f64", 2000, 16, 5, "k-means++", 2, 4, None, 300),
    "weights_int_u8_k5": ("blobs_u8", 2000, 4, 5, "k-means++", 1, 5, "int", 300),
    "weights_real_f64_k4": ("blobs_f64", 1500, 6, 4, "random", 2, 6, "real", 300),
    "weights_real_f32_k4": ("blobs_f32", 1500, 5, 4, "k-means++", 1, 7, "real", 300),
    "dup_init_f64_k4": ("blobs_f64", 1200, 3, 4, "dup", 1, 0, None, 300),
    "f32_d64_k8": ("blobs_f32", 2000, 64, 8, "k-means++", 1, 8, None, 300),
    "cell_u8_k8_maxiter1": ("cell_u8", 5852, 4, 8, "k-means++", 1, 9, None, 1),
    "cell_u8_k8_maxiter2": ("cell_u8", 5852, 4, 8, "k-means++", 1, 9, None, 2),
    "cell_u8_k1": ("cell_u8", 1000, 4, 1, "k-means++", 1, 0, None, 300),
}


def elkan_case(name):
    """(rows, sample_weight or None, init) of a case, regenerated from its name"""
    kind, n, d, k, init, n_init, rs, wk, max_iter = ELKAN_CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    if kind == "ties_u8":
        X = rng.integers(0, 6, (n, d), dtype=np.uint8)
    elif kind == "cell_u8":
        X = rng.integers(0, 256, (n, d), dtype=np.uint8)
    else:
        cen = rng.uniform(20, 230, (k + 3, d))
        Xf = cen[rng.integers(k + 3, size=n)] + rng.normal(0, 14, (n, d))
        X = (np.clip(np.rint(Xf), 0, 255).astype(np.uint8) if kind == "blobs_u8"
             else Xf.astype(np.float32 if kind == "blobs_f32" else np.float64))
    w = None
    if wk == "int":
        w = rng.integers(0, 4, n).astype(np.float64)
    elif wk == "real":
        w = rng.uniform(0.25, 3.0, n)
        w[::17] = 0.0
    if init == "dup":               # two equal initial centres: an empty cluster, and dnc = 0
        init = X[[0, 0, 5, 9]].astype(np.float64)
    return X, w, init


def pin_oracle():
    """tests/kmeans_elkan_np.py against sklearn's own Cython functions: distances, init_bounds_dense and the label half
    of elkan_iter_chunked_dense bit for bit (bounds included) given the same centre half-distances"""
    sys.path.insert(0, ROOT)
    from sklearn.cluster._k_means_common import _euclidean_dense_dense_wrapper
    from sklearn.cluster._k_means_elkan import elkan_iter_chunked_dense, init_bounds_dense
    from sklearn.metrics import euclidean_distances
    from tests import kmeans_elkan_np as E
    rng = np.random.default_rng(0)
    for dt in (np.float32, np.float64):
        for d in (1, 2, 3, 4, 5, 7, 8, 13, 64):
            A = (rng.normal(0, 50, (40, d))).astype(dt)
            b = A[3] + rng.normal(0, 1, d).astype(dt)
            for sq in (False, True):
                want = np.array([_euclidean_dense_dense_wrapper(a, b, sq) for a in A], dt)
                assert np.array_equal(E.euclidean(A, b, sq), want), (dt, d, sq)
    moved = 0
    for name, dt, k in (("ties", np.float64, 7), ("ties", np.float32, 7), ("normal", np.float64, 9), ("normal", np.float32, 9)):
        if name == "ties":
            X = rng.integers(0, 6, (3000, 3)).astype(dt)
        else:
            X = rng.normal(0, 30, (3000, 6)).astype(dt)
        Xc = X - X.mean(axis=0)
        C = Xc[rng.choice(3000, k, replace=False)].copy()
        C[1] = C[0]                                            # duplicate centres: chd = 0 between them
        chd = (euclidean_distances(C) / 2).astype(dt)
        dnc = np.partition(chd, kth=1, axis=0)[1]
        lab = np.full(3000, -1, np.int32)
        up = np.zeros(3000, dt)
        lo = np.zeros((3000, k), dt)
        init_bounds_dense(Xc, C, chd, lab, up, lo, 1)
        l0, u0, w0 = E.elkan_init(Xc, C, chd)
        assert np.array_equal(l0, lab) and np.array_equal(u0, up) and np.array_equal(w0, lo), (name, dt, "init")
        # move the centres a little so that rows change label, then one label-only iteration from the init bounds
        C2 = (C + rng.normal(0, 2.0, C.shape)).astype(dt)
        C2[1] = C2[0]
        chd2 = (euclidean_distances(C2) / 2).astype(dt)
        dnc2 = np.partition(chd2, kth=1, axis=0)[1]
        l1, u1, w1, _ = E.elkan_step(Xc, C2, chd2, dnc2, lab, up, lo)
        elkan_iter_chunked_dense(Xc, np.ones(3000, dt), C2, C2.copy(), np.zeros(k, dt), chd2, dnc2, up, lo, lab, np.zeros(k, dt), 1,
                                 update_centers=False)
        assert np.array_equal(l1, lab) and np.array_equal(u1, up) and np.array_equal(w1, lo), (name, dt, "step")
        moved += int((l1 != l0).sum())
    assert moved > 0


def sklearn_geometry(C):
    from sklearn.metrics import euclidean_distances
    chd = euclidean_distances(C) / 2
    return chd, np.partition(chd, kth=1, axis=0)[1]


def make_elkan_golden():
    import warnings
    from sklearn.cluster import KMeans
    sys.path.insert(0, ROOT)
    from tests import kmeans_elkan_np as E
    pin_oracle()
    out = {}
    for name, (_, n, d, k, init, n_init, rs, _, max_iter) in ELKAN_CASES.items():
        X, w, init_arr = elkan_case(name)
        init_p = init_arr if not isinstance(init_arr, str) else init
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", RuntimeWarning)
            km = KMeans(k, init=init_p, n_init=n_init, random_state=rs, max_iter=max_iter, algorithm="elkan").fit(X, sample_weight=w)
            ll = KMeans(k, init=init_p, n_init=n_init, random_state=rs, max_iter=max_iter, algorithm="lloyd").fit(X, sample_weight=w)
        out[name + "_labels"] = km.labels_.astype(np.int32)
        out[name + "_centers"] = km.cluster_centers_
        out[name + "_inertia"] = np.float64(km.inertia_)
        out[name + "_n_iter"] = np.int64(km.n_iter_)
        out[name + "_lloyd_labels"] = ll.labels_.astype(np.int32)
        if n_init == 1 and k > 1:
            # the oracle's whole fit from sklearn's seeds (one start: the same seeds as the estimator's)
            if isinstance(init_p, str):
                from sklearn.cluster import kmeans_plusplus
                Xw = X.astype(np.float64) if X.dtype == np.uint8 else X
                _, idx = kmeans_plusplus(Xw, k, random_state=np.random.RandomState(rs), sample_weight=w)
                seeds = X[idx].astype(np.float64)
            else:
                seeds = init_p
            lab, cen, inertia, n_iter = E.elkan_fit(X, seeds, max_iter=max_iter, sample_weight=w, half_distances=sklearn_geometry)
            assert np.array_equal(lab, km.labels_) and n_iter == km.n_iter_, name
            assert np.allclose(cen, km.cluster_centers_, rtol=0, atol=1e-4 if X.dtype == np.float32 else 1e-9), name
            assert abs(inertia - km.inertia_) <= (1e-5 if X.dtype == np.float32 else 1e-9) * abs(km.inertia_), name
        print(f"{name}: n_iter {km.n_iter_}, labels differing from lloyd: {int((km.labels_ != ll.labels_).sum())}")
    assert any((out[c + "_labels"] != out[c + "_lloyd_labels"]).any() for c in ("ties_u8_k7_s0", "ties_u8_k7_s2"))
    np.savez_compressed(os.path.join(HERE, "kmeans_sklearn_elkan.npz"), **out)


if __name__ == "__main__":
    make_elkan_golden()
