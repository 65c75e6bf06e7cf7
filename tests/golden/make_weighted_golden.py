"""Generate tests/golden/kmeans_sklearn_weighted.npz: scikit-learn 1.9.0 ``KMeans(...).fit(X, sample_weight=w)`` restated
start by start (every start's seeds, inertia and n_iter, the start sklearn keeps, and its labels / centres / inertia /
n_iter), for the tests of the weighted fit.

    python tests/golden/make_weighted_golden.py

The rows and weights are regenerated from each case's name by ``weighted_case``, so the fixture stores only the results."""
from __future__ import annotations

import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


WEIGHTED_CASES = {   # name: (rows kind, n, d, k, init, n_init, random_state, weights kind)
    "u8_k5_pp1_intw": ("blobs_u8", 3000, 4, 5, "k-means++", 1, 0, "int"),
    "u8_k6_pp10_realw": ("blobs_u8", 3000, 4, 6, "k-means++", 10, 1, "real"),
    "u8_k8_random_auto": ("blobs_u8", 4000, 4, 8, "random", "auto", 2, "real"),
    "f32_k6_pp4": ("blobs_f32", 2000, 8, 6, "k-means++", 4, 3, "real"),
    "f64_k4_random3": ("blobs_f64", 1500, 3, 4, "random", 3, 4, "real"),
    "u8_k5_pp3_zerow": ("blobs_u8", 2000, 4, 5, "k-means++", 3, 5, "zeros"),
    "probe_zero_weight_cluster": ("probe", 5, 2, 3, "explicit", 1, 0, "probe"),
    "f32_d64_k8_pp1": ("blobs_f32", 3000, 64, 8, "k-means++", 1, 6, "real"),
}

#: the explicit init of the probe case: rows 0, 2 and 4 (row 4 has weight 0, so its cluster is empty by weight).  Row 3
#: is (10, 12), not (10, 11), so that it is the single farthest row: at (10, 11) it would tie with row 1, and sklearn's
#: argpartition and this library's relocation (lowest index on ties) would move different rows.
PROBE_INIT_ROWS = np.array([0, 2, 4])


def weighted_case(name):
    """regenerate the rows X and weights w of a case from its name (the fixture stores the sklearn results)"""
    kind, n, d, k, init, n_init, rs, wkind = WEIGHTED_CASES[name]
    if kind == "probe":
        return (np.array([[0, 0], [0, 1], [10, 10], [10, 12], [50, 50]], np.float64),
                np.array([1, 1, 1, 1, 0], np.float64))
    rng = np.random.default_rng(sum(map(ord, name)))
    cen = rng.uniform(20, 230, (k + 3, d))        # more blobs than clusters: the starts end in different optima
    X = cen[rng.integers(k + 3, size=n)] + rng.normal(0, 14, (n, d))
    if kind == "blobs_u8":
        X = np.clip(np.rint(X), 0, 255).astype(np.uint8)
    else:
        X = X.astype(np.float32 if kind == "blobs_f32" else np.float64)
    wdt = np.float32 if X.dtype == np.float32 else np.float64
    if wkind == "int":
        w = rng.integers(1, 6, n).astype(wdt)
    elif wkind == "zeros":                        # a third of the rows weigh nothing: never a seed
        w = rng.uniform(0.2, 4.0, n) * (rng.uniform(size=n) > 0.33)
    else:
        w = rng.uniform(0.05, 3.0, n)
    return X, w.astype(wdt)


def make_weighted_kmeans_golden():
    """KMeans(init, n_init, random_state).fit(X, sample_weight=w) of sklearn 1.9.0, restated start by start: every start's
    seeds from sklearn's own kmeans_plusplus(sample_weight=w) / RandomState.choice(p=w / w.sum()) on one RandomState, its
    Lloyd fit by KMeans(init=seeds, n_init=1).fit(X, sample_weight=w), then sklearn's choice of the start (strictly lower
    inertia and a different clustering).  The restatement is checked against KMeans(...).fit(X, sample_weight=w) here."""
    from sklearn.cluster import KMeans, kmeans_plusplus
    from sklearn.cluster._k_means_common import _is_same_clustering
    cases = {}
    for name, (_, n, d, k, init, n_init, seed, _w) in WEIGHTED_CASES.items():
        X, w = weighted_case(name)
        Xw = X.astype(np.float64) if X.dtype == np.uint8 else X
        if init == "explicit":
            fit = KMeans(n_clusters=k, init=Xw[PROBE_INIT_ROWS], n_init=1).fit(X, sample_weight=w)
            seeds, runs, best, ref = [PROBE_INIT_ROWS], [fit], 0, fit
            assert (fit.labels_ == [0, 0, 1, 2, 2]).all() and fit.n_iter_ == 2, name
            assert np.allclose(fit.cluster_centers_, [[0, 0.5], [10, 10], [10, 12]], atol=1e-12, rtol=0), name
        else:
            R = n_init if n_init != "auto" else (10 if init == "random" else 1)
            rs = np.random.RandomState(seed)
            seeds, runs = [], []
            for _ in range(R):
                if init == "k-means++":
                    _, idx = kmeans_plusplus(Xw, k, sample_weight=w, random_state=rs)
                else:
                    idx = rs.choice(n, size=k, replace=False, p=w / w.sum())
                seeds.append(idx)
                runs.append(KMeans(n_clusters=k, init=Xw[idx], n_init=1).fit(X, sample_weight=w))
            best = 0
            for i in range(1, R):
                if runs[i].inertia_ < runs[best].inertia_ and not _is_same_clustering(
                        runs[i].labels_.astype(np.int32), runs[best].labels_.astype(np.int32), k):
                    best = i
            ref = KMeans(n_clusters=k, init=init, n_init=n_init, random_state=seed).fit(X, sample_weight=w)
        win = runs[best]
        assert (ref.labels_ == win.labels_).all() and ref.n_iter_ == win.n_iter_, name
        assert np.abs(ref.cluster_centers_ - win.cluster_centers_).max() < (1e-4 if X.dtype == np.float32 else 1e-9), name
        assert abs(ref.inertia_ - win.inertia_) <= 1e-6 * ref.inertia_, name
        if name.endswith("zerow"):
            assert all((w[s] > 0).all() for s in seeds), name
        cases[name + "_seed_idx"] = np.array(seeds, np.int64)
        cases[name + "_start_inertia"] = np.array([r.inertia_ for r in runs], np.float64)
        cases[name + "_start_niter"] = np.array([r.n_iter_ for r in runs], np.int64)
        cases[name + "_best"] = np.int64(best)
        cases[name + "_labels"] = win.labels_.astype(np.int32)
        cases[name + "_centers"] = win.cluster_centers_
        cases[name + "_inertia"] = np.float64(win.inertia_)
        cases[name + "_niter"] = np.int64(win.n_iter_)
        print(name, "best start", best, "of", len(runs), "n_iter", win.n_iter_,
              "inertias", np.round(cases[name + "_start_inertia"], 1).tolist())
    np.savez_compressed(f"{HERE}/kmeans_sklearn_weighted.npz", **cases)
    print("weighted kmeans goldens ok")


if __name__ == "__main__":
    make_weighted_kmeans_golden()
