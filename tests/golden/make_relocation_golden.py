"""Generate tests/golden/kmeans_sklearn_relocation.npz: scikit-learn 1.9.0 ``KMeans(init=C0, n_init=1, max_iter=m)
.fit(X, sample_weight=w)`` on fits where clusters go empty, for the tests of the empty-cluster relocation and of the
centre an empty cluster takes.

    python tests/golden/make_relocation_golden.py

sklearn's rules (_k_means_common.pyx:167-211, :274-295), which the library reproduces:
  * the clusters of weight 0 are listed ONCE; the n_empty farthest rows (unweighted squared distance to the old centre of
    their label) move into them, carrying x w and w.  A cluster that a move empties -- its only member, or its only member
    of positive weight, was the moved row -- stays empty for the iteration, whatever its index;
  * _average_centers divides the sums in place, in cluster index order: an empty cluster copies the row of the heaviest
    cluster as it is at that moment -- the heaviest cluster's (centred) SUM when the empty cluster's index is lower,
    its mean otherwise.

Every case is regenerated from its name (``PROBES``, ``relocation_case``), so the fixture stores only sklearn's results:
labels, centres, inertia and n_iter for max_iter = 1, 2 and 300 (converged).  Each is checked here against live sklearn
and against the oracle (oracle/kmeans_np.py)."""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_ITERS = (1, 2, 300)


# ---- the three probes -----------------------------------------------------------------------------------------------
# cascade: row 3 (x = 60) is the only member of cluster 2 and the farthest row; cluster 0 is empty.  Moving it empties
#   cluster 2, which sklearn leaves empty (it copies the heaviest cluster's mean); re-reading "count == 0" would fill it.
# in_place: the same rows with clusters 1 and 2 swapped: the emptied cluster 1 sits below the heaviest cluster 2, so it
#   takes cluster 2's centred sum (x = -28 after the mean is added back).
# zero_weight_move: the farthest row weighs 0, so the cluster it moves into stays empty by weight and takes the heaviest
#   cluster's centred sum (x = -8.2).
_X4 = np.array([[0, 0], [1, 0], [3, 0], [60, 0]], np.float64)
PROBES = {   # name: (X, init, sample_weight)
    "cascade": (_X4, np.array([[-1000, 0], [1, 0], [100, 0]], np.float64), None),
    "in_place": (_X4, np.array([[-1000, 0], [100, 0], [1, 0]], np.float64), None),
    "zero_weight_move": (np.array([[0, 0], [1, 0], [3, 0], [60, 0], [2, 0]], np.float64),
                         np.array([[-1000, 0], [2, 0], [1, 0]], np.float64), np.array([1, 1, 1, 0, 1], np.float64)),
}


def probe_form(name, form):
    """a probe as ``form``: "f64" (as stated), "f32", "u8" (4 columns: x, 0, 0, 255 -- the pixel shape; the init's x
    moved inside the byte range where it was not), "w" (cascade / in_place with weights: the far row and two rows of weight
    0 in its cluster, the rest real-valued).  Returns (X, init, sample_weight or None)."""
    X, init, w = PROBES[name]
    if form == "f64":
        return X, init, w
    if form == "f32":
        return X.astype(np.float32), init, None if w is None else w.astype(np.float32)
    if form == "u8":
        Xu = np.zeros((X.shape[0], 4), np.uint8)
        Xu[:, 0] = X[:, 0]
        Xu[:, 3] = 255
        iu = np.zeros((init.shape[0], 4))
        iu[:, 0] = np.where(init[:, 0] < 0, 250, init[:, 0])      # still nobody's nearest centre
        iu[:, 3] = 255
        return Xu, iu, w
    assert form == "w" and w is None
    Xw = np.concatenate([X, [[70, 0], [80, 0]]])                  # nearer the far row's centre (x = 100) than it is
    return Xw, init, np.array([1.5, 0.25, 2.0, 3.0, 0.0, 0.0])


PROBE_FORMS = [(p, f) for p in PROBES for f in ("f64", "f32", "u8")] + [("cascade", "w"), ("in_place", "w")]


# ---- the scalable case ----------------------------------------------------------------------------------------------
def relocation_case(n, d, dtype, k, weighted=False, below=False, seed=0):
    """Rows X [n, d], init [k, d] and weights (None unless ``weighted``) of a fit in which, at the first iteration,
    cluster 0 is empty and an outlier is the only member (``weighted``: the only member of positive weight, with two rows
    of weight 0 beside it) of another cluster -- so moving it empties that cluster:
      * k - 2 tight (sd 2), well-separated blobs of distinct sizes, each with its own centre as initial centre;
      * the outlier's cluster is k - 1 (above every blob: it copies the heaviest blob's mean) or, ``below``, 1 with the
        heaviest blob last (it copies the heaviest blob's centred sum, which lies far outside the data);
      * columns 2.. are padding, equal in every row and centre: no distance or tie changes, but d > 32 routes the same
        fit through the wide E-step kernels;
      * the outlier's squared distance to its centre (900) is well above any blob row's, so the farthest row is unique.
    The values are integers in [0, 255] for every dtype (so uint8 is the same case), blob noise excepted."""
    assert k >= 3 and d >= 2
    rng = np.random.default_rng(1000 * seed + 7 * k + d)
    nb = k - 2
    side = int(np.ceil(np.sqrt(nb)))
    grid = np.linspace(60, 230, max(side, 2))
    bc = np.array([[grid[i % side], grid[i // side]] for i in range(nb)])        # blob centres, >= 56 apart
    size_w = np.arange(1, nb + 1, dtype=np.float64) + 0.5                         # distinct sizes: the last is heaviest
    n_extra = 3 if weighted else 1
    counts = np.floor((n - n_extra) * size_w / size_w.sum()).astype(int)
    counts[-1] += n - n_extra - counts.sum()
    lab = np.repeat(np.arange(nb), counts)
    rows2 = bc[lab] + rng.normal(0, 2.0, (lab.size, 2))
    if dtype == np.uint8:
        rows2 = np.rint(rows2)
    extra = [[3.0, 3.0]] + ([[14.0, 3.0], [22.0, 3.0]] if weighted else [])       # the outlier, then its weight-0 rows
    rows2 = np.concatenate([rows2, extra])
    perm = rng.permutation(n)                                                     # the outlier lands anywhere
    rows2 = rows2[perm]
    X = np.full((n, d), 17.0)
    X[:, :2] = rows2
    X = X.astype(dtype)
    init = np.full((k, d), 17.0)
    init[0, :2] = (-400.0, -400.0)                                                 # empty from the start
    o = 1 if below else k - 1
    blob_idx = [j for j in range(1, k) if j != o]
    init[o, :2] = (33.0, 3.0)                                                      # the outlier is 30 away
    init[blob_idx, :2] = bc
    w = None
    if weighted:
        wdt = np.float32 if dtype == np.float32 else np.float64
        w = rng.uniform(0.25, 3.0, n)
        src = np.argsort(perm)                                                     # row of original index i
        w[src[n - n_extra:]] = [2.0, 0.0, 0.0][:n_extra]
        w = w.astype(wdt)
    return X, init, w


GEN_CASES = {   # name: relocation_case arguments
    "u8_d4_k8": (3000, 4, np.uint8, 8, False, False),
    "u8_d4_k8_below": (50000, 4, np.uint8, 8, False, True),
    "u8_d4_k16_w": (8000, 4, np.uint8, 16, True, False),
    "u8_d4_k3_w_below": (2000, 4, np.uint8, 3, True, True),
    "f64_d42_k6_below": (3000, 42, np.float64, 6, False, True),
    "f64_d130_k5_w": (2500, 130, np.float64, 5, True, False),
    "f32_d42_k6_w_below": (3000, 42, np.float32, 6, True, True),
    "f32_d390_k4": (1500, 390, np.float32, 4, False, False),
}


def gen_case(name):
    n, d, dt, k, weighted, below = GEN_CASES[name]
    return relocation_case(n, d, dt, k, weighted, below)


def golden_fit(z, key, max_iter):
    """sklearn's (labels, centres, inertia, n_iter) of case ``key`` ("probe_<name>_<form>" or "gen_<name>")"""
    t = f"{key}_m{max_iter}"
    return z[t + "_labels"], z[t + "_centers"], float(z[t + "_inertia"]), int(z[t + "_niter"])


def check_fit(what, got, ref, X):
    """the bars of the relocation tests on a fit of rows X: labels and n_iter exact; centres within 1e-9 (float32: 1e-4);
    a sum-valued centre (an empty cluster's copy of the heaviest cluster's centred sum: some value outside the rows'
    range) within 1e-12 (float32: 1e-5 -- sklearn sums float32 rows in float32) of its largest entry, times n / 1e5 past
    1e5 rows -- the reference's own sum of n centred rows carries about n eps of rounding, in every column; inertia
    within 1e-9 relative (float32: 1e-5).  The mismatch counts are printed before anything is asserted."""
    lab, cen, inertia, n_iter = (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v) for v in got)
    rl, rc, ri, rn = ref
    f32 = X.dtype == np.float32
    Xd = np.asarray(X, np.float64)
    sum_row = ((rc < Xd.min(axis=0) - 1.0) | (rc > Xd.max(axis=0) + 1.0)).any(axis=1, keepdims=True)
    sum_rel = (1e-5 if f32 else 1e-12) * max(1.0, X.shape[0] / 1e5)
    tol = np.where(sum_row, sum_rel * np.abs(rc).max(axis=1, keepdims=True), 1e-4 if f32 else 1e-9)
    n_lab, n_cen = int((lab != rl).sum()), int((np.abs(cen - rc) > tol).sum())
    rel = abs(float(inertia) - ri) / max(ri, 1e-300)
    print(f"{what}: {n_lab} labels differ, {n_cen} centre values off, n_iter {int(n_iter)} vs {rn}, inertia rel err {rel:.2e}")
    assert n_lab == 0 and int(n_iter) == rn, what
    assert n_cen == 0, (what, float(np.abs(cen - rc).max()))
    assert rel <= (1e-5 if f32 else 1e-9), what


def _fit(X, init, w, max_iter):
    from sklearn.cluster import KMeans
    return KMeans(n_clusters=init.shape[0], init=init, n_init=1, max_iter=max_iter).fit(X, sample_weight=w)


def make_relocation_golden():
    import warnings
    warnings.filterwarnings("ignore")                       # max_iter = 1, 2 stop before convergence on purpose
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import kmeans_np as K
    out = {}
    cases = [(f"probe_{p}_{f}",) + probe_form(p, f) for p, f in PROBE_FORMS]
    cases += [(f"gen_{name}",) + gen_case(name) for name in GEN_CASES]
    for key, X, init, w in cases:
        for m in MAX_ITERS:
            fit = _fit(X, init, w, m)
            ref = (fit.labels_, fit.cluster_centers_.astype(np.float64), float(fit.inertia_), int(fit.n_iter_))
            check_fit(f"oracle {key} max_iter={m}", K.kmeans_fit(X, init, max_iter=m, sample_weight=w), ref, X)
            tag = f"{key}_m{m}"
            out[tag + "_labels"] = fit.labels_.astype(np.int32)
            out[tag + "_centers"] = fit.cluster_centers_.astype(np.float64)
            out[tag + "_inertia"] = np.float64(fit.inertia_)
            out[tag + "_niter"] = np.int64(fit.n_iter_)
        print(key, "n_iter", int(out[f"{key}_m300_niter"]), "empty at the end:",
              int((np.bincount(out[f"{key}_m300_labels"], minlength=init.shape[0]) == 0).sum()))
    np.savez_compressed(f"{HERE}/kmeans_sklearn_relocation.npz", **out)
    print("relocation goldens ok")


if __name__ == "__main__":
    make_relocation_golden()
