"""Generate tests/golden/kmeans_sklearn_ninit.npz: scikit-learn 1.9.0 ``KMeans(init, n_init, random_state)`` restated
start by start (every start's seeds, inertia and n_iter, the start sklearn keeps, and its labels / centres / inertia /
n_iter), for the tests of ``KMeans(n_init=R)`` and ``init="random"``.

    python tests/golden/make_ninit_golden.py

The rows are regenerated from each case's name by ``ninit_case``, so the fixture stores only the results."""
from __future__ import annotations

import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


NINIT_CASES = {   # name: (rows kind, n, d, k, init, n_init, random_state)
    "blobs_u8_k5_pp10": ("blobs_u8", 3000, 4, 5, "k-means++", 10, 0),
    "cell_u8_k8_pp10": ("cell_u8", 76 * 77, 4, 8, "k-means++", 10, 3),
    "u8_k8_random_auto": ("blobs_u8", 4000, 4, 8, "random", "auto", 1),
    "f32_k6_pp4": ("blobs_f32", 2000, 8, 6, "k-means++", 4, 2),
    "f64_k4_random3": ("blobs_f64", 1500, 3, 4, "random", 3, 4),
    "separated_k3_pp6": ("separated_u8", 900, 4, 3, "k-means++", 6, 5),
}


def ninit_case(name):
    """regenerate the rows of an n_init case from its name (the fixture stores the sklearn results)"""
    kind, n, d, k, init, n_init, rs = NINIT_CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    if kind == "cell_u8":
        return rng.integers(0, 256, (n, d), dtype=np.uint8)
    if kind == "separated_u8":             # three tight blobs far apart: every start finds the same clustering
        cen = np.array([[20, 20, 20, 20], [128, 128, 128, 128], [235, 235, 235, 235]], np.float64)
        return np.clip(np.rint(cen[np.arange(n) % 3] + rng.normal(0, 3, (n, d))), 0, 255).astype(np.uint8)
    cen = rng.uniform(20, 230, (k + 3, d))        # more blobs than clusters: the starts end in different optima
    X = cen[rng.integers(k + 3, size=n)] + rng.normal(0, 14, (n, d))
    if kind == "blobs_u8":
        return np.clip(np.rint(X), 0, 255).astype(np.uint8)
    return X.astype(np.float32 if kind == "blobs_f32" else np.float64)


def make_ninit_kmeans_golden():
    """KMeans(n_init=R, init=..., random_state=rs) of sklearn 1.9.0, restated start by start: every start's seeds from
    sklearn's own kmeans_plusplus / RandomState.choice on one RandomState, its Lloyd fit by KMeans(init=seeds,
    n_init=1), then sklearn's choice of the start (strictly lower inertia and a different clustering).  The
    restatement is checked against KMeans(n_init=R).fit here."""
    from sklearn.cluster import KMeans, kmeans_plusplus
    from sklearn.cluster._k_means_common import _is_same_clustering
    cases = {}
    for name, (_, n, d, k, init, n_init, seed) in NINIT_CASES.items():
        X = ninit_case(name)
        R = n_init if n_init != "auto" else (10 if init == "random" else 1)
        rs = np.random.RandomState(seed)
        Xw = X.astype(np.float64) if X.dtype == np.uint8 else X
        seeds, runs = [], []
        for _ in range(R):
            if init == "k-means++":
                _, idx = kmeans_plusplus(Xw, k, random_state=rs)
            else:
                w = np.ones(n, dtype=Xw.dtype)
                idx = rs.choice(n, size=k, replace=False, p=w / w.sum())
            seeds.append(idx)
            runs.append(KMeans(n_clusters=k, init=Xw[idx], n_init=1).fit(X))
        best = 0
        for i in range(1, R):
            if runs[i].inertia_ < runs[best].inertia_ and not _is_same_clustering(
                    runs[i].labels_.astype(np.int32), runs[best].labels_.astype(np.int32), k):
                best = i
        ref = KMeans(n_clusters=k, init=init, n_init=n_init, random_state=seed).fit(X)
        win = runs[best]
        assert (ref.labels_ == win.labels_).all() and ref.n_iter_ == win.n_iter_, name
        assert np.abs(ref.cluster_centers_ - win.cluster_centers_).max() < (1e-4 if X.dtype == np.float32 else 1e-9), name
        assert abs(ref.inertia_ - win.inertia_) <= 1e-9 * ref.inertia_, name
        if name.startswith("separated"):
            assert best == 0, name
        cases[name + "_seed_idx"] = np.array(seeds, np.int64)
        cases[name + "_start_inertia"] = np.array([r.inertia_ for r in runs], np.float64)
        cases[name + "_start_niter"] = np.array([r.n_iter_ for r in runs], np.int64)
        cases[name + "_best"] = np.int64(best)
        cases[name + "_labels"] = win.labels_.astype(np.int32)
        cases[name + "_centers"] = win.cluster_centers_
        cases[name + "_inertia"] = np.float64(win.inertia_)
        cases[name + "_niter"] = np.int64(win.n_iter_)
        print(name, "best start", best, "of", R, "inertias", np.round(cases[name + "_start_inertia"], 1).tolist())
    np.savez_compressed(f"{HERE}/kmeans_sklearn_ninit.npz", **cases)
    print("n_init kmeans goldens ok")


if __name__ == "__main__":
    make_ninit_kmeans_golden()
