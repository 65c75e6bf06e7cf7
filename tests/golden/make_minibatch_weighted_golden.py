"""Generate tests/golden/minibatch_sklearn_weighted.npz: scikit-learn 1.9.0 ``MiniBatchKMeans`` with sample weights,
``init="random"``, several starts, float32 rows and ``partial_fit`` sequences, for the tests of minibatch.py.

    python tests/golden/make_minibatch_weighted_golden.py

The rows and weights are regenerated from each case's name by ``fit_case`` / ``partial_case``, so the fixture stores only
the results: for a fit case ``cluster_centers_``, ``_counts``, ``labels_``, ``inertia_`` and ``n_steps_``; for a
partial_fit sequence the same after every call.  Before writing, the script checks the numpy restatement
(tests/minibatch_weighted_np.py) against sklearn on every case."""
from __future__ import annotations

import os
import sys

if __name__ == "__main__":
    # one thread, set before numpy and sklearn load: sklearn sums the inertia in per-thread chunks, so only a fixed
    # thread count regenerates the same bits
    os.environ["OMP_NUM_THREADS"] = os.environ["OPENBLAS_NUM_THREADS"] = "1"

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

FIT_CASES = {   # name: (rows kind, n, d, k, weights kind, estimator keywords)
    "u8_unique_counts": ("lab_u8", 20000, 3, 8, "counts", dict(random_state=0)),
    "u8_realw": ("lab_u8", 9000, 3, 6, "real", dict(random_state=1)),
    "u8_zerow": ("lab_u8", 8000, 3, 5, "zeros", dict(random_state=2)),
    "u8_random_auto": ("lab_u8", 6000, 3, 8, "real", dict(random_state=3, init="random")),
    "u8_pp3_realw": ("lab_u8", 6000, 3, 7, "real", dict(random_state=4, n_init=3)),
    "f32_realw": ("blobs_f32", 5000, 5, 6, "real", dict(random_state=5)),
    "u8_nolabels": ("lab_u8", 7000, 3, 6, "real", dict(random_state=6, compute_labels=False)),
    "f64_tol": ("blobs_f64", 6000, 4, 5, "int", dict(random_state=7, tol=1e-3)),
}

# name: (rows kind, d, k, [(rows, weights kind), ...] per call, estimator keywords, "fit" calls as ("fit", n, wkind))
PARTIAL_CASES = {
    "u8_sizes": ("lab_u8", 3, 8, [(3000, None), (700, None), (60000, None), (1024, None)], dict(random_state=0)),
    "u8_intw": ("lab_u8", 3, 6, [(2000, "int"), (1500, "int"), (2500, "int")], dict(random_state=1)),
    "u8_realw": ("lab_u8", 3, 6, [(2000, "real"), (1500, "real"), (2500, "real")], dict(random_state=2)),
    "f32_batches": ("blobs_f32", 4, 5, [(1500, None), (1200, "real"), (1800, None)], dict(random_state=3)),
    "u8_reassign": ("lab_u8", 3, 8, [(1500, None), (1500, None), (1500, None), (1500, None)],
                    dict(random_state=4, reassignment_ratio=0.6)),
    "u8_zero_weight_cluster": ("lab_u8", 3, 4, [(1200, "zero_blob"), (1200, "zero_blob"), (1200, None)], dict(random_state=5)),
    "fit_then_partial": ("lab_u8", 3, 6, [("fit", 5000, None), (2000, None), (2000, "real")], dict(random_state=6)),
    "rs_instance": ("lab_u8", 3, 5, [(2000, None), (2000, "int"), (2000, None)], dict(random_state="instance:7")),
    "partial_fit_partial": ("lab_u8", 3, 5, [(2000, None), ("fit", 4000, "real"), (1800, None), (1800, "int")],
                            dict(random_state=8)),
}


def _rows(kind, n, d, rng):
    if kind == "lab_u8":                          # LAB-like pixels: colour blobs on a smooth background
        cen = rng.uniform(30, 220, (10, d))
        X = cen[rng.integers(10, size=n)] + rng.normal(0, 9, (n, d))
        return np.clip(np.rint(X), 0, 255).astype(np.uint8)
    cen = rng.uniform(20, 230, (9, d))
    X = cen[rng.integers(9, size=n)] + rng.normal(0, 14, (n, d))
    return X.astype(np.float32 if kind == "blobs_f32" else np.float64)


def _weights(wkind, X, rng):
    n = X.shape[0]
    wdt = np.float32 if X.dtype == np.float32 else np.float64
    if wkind is None:
        return None
    if wkind == "int":
        w = rng.integers(1, 6, n)
    elif wkind == "real":
        w = rng.uniform(0.05, 3.0, n)
    elif wkind == "zeros":                        # a third of the rows weigh nothing
        w = rng.uniform(0.2, 4.0, n) * (rng.uniform(size=n) > 0.33)
    else:                                         # "zero_blob": the rows near the first row's colour weigh nothing
        w = np.where(np.abs(X.astype(np.float64) - X[0].astype(np.float64)).max(axis=1) < 25, 0.0, 1.0)
    return w.astype(wdt)


def fit_case(name):
    """(X, w, k, keywords) of a fit case, regenerated from its name"""
    kind, n, d, k, wkind, kw = FIT_CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    X = _rows(kind, n, d, rng)
    if wkind == "counts":                         # the unique colours of the pixels, weighted by their counts
        X, w = np.unique(X, axis=0, return_counts=True)
        return X, w.astype(np.float64), k, dict(kw)
    return X, _weights(wkind, X, rng), k, dict(kw)


def _random_state(v):
    return np.random.RandomState(int(v.split(":")[1])) if isinstance(v, str) else v


def partial_case(name):
    """(k, keywords, [(call, X, w), ...]) of a partial_fit sequence, regenerated from its name; call is "partial_fit" or
    "fit"; a "instance:s" random_state is a fresh RandomState(s)"""
    kind, d, k, calls, kw = PARTIAL_CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    seq = []
    for c in calls:
        call, n, wkind = ("fit",) + c[1:] if c[0] == "fit" else ("partial_fit",) + c
        X = _rows(kind, n, d, rng)
        seq.append((call, X, _weights(wkind, X, rng)))
    kw = dict(kw)
    kw["random_state"] = _random_state(kw["random_state"])
    return k, kw, seq


def _result(m, prefix, out, labels=True):
    out[prefix + "_centers"] = np.array(m.cluster_centers_, np.float64)      # a copy: partial_fit updates in place
    out[prefix + "_counts"] = np.array(m._counts, np.float64)
    out[prefix + "_inertia"] = np.float64(m.inertia_)
    out[prefix + "_nsteps"] = np.int64(m.n_steps_)
    if labels:
        out[prefix + "_labels"] = np.asarray(m.labels_, np.int32)


def _close(a, b, f32):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() <= (1e-3 if f32 else 1e-9) * max(1.0, np.abs(b).max())


def _check(o, prefix, out, labels, f32):
    assert int(o.n_steps_) == int(out[prefix + "_nsteps"]), prefix
    if labels:
        assert (o.labels_ == out[prefix + "_labels"]).all(), prefix
    assert _close(o.cluster_centers_, out[prefix + "_centers"], f32), prefix
    assert _close(o._counts, out[prefix + "_counts"], f32), prefix
    assert abs(o.inertia_ - out[prefix + "_inertia"]) <= (1e-5 if f32 else 1e-9) * max(1.0, abs(out[prefix + "_inertia"])), prefix


def make_minibatch_weighted_golden():
    import sklearn
    from sklearn.cluster import MiniBatchKMeans
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from tests import minibatch_weighted_np as MB
    assert sklearn.__version__ == "1.9.0", sklearn.__version__
    out = {}
    for name in FIT_CASES:
        X, w, k, kw = fit_case(name)
        m = MiniBatchKMeans(n_clusters=k, **kw).fit(X, sample_weight=w)
        _result(m, name, out, kw.get("compute_labels", True))
        X, w, k, kw = fit_case(name)
        o = MB.MiniBatch(k, **kw).fit(X, sample_weight=w)
        _check(o, name, out, kw.get("compute_labels", True), X.dtype == np.float32)
    for name in PARTIAL_CASES:
        for impl in ("sklearn", "oracle"):
            k, kw, seq = partial_case(name)
            m = MiniBatchKMeans(n_clusters=k, **kw) if impl == "sklearn" else MB.MiniBatch(k, **kw)
            for i, (call, X, w) in enumerate(seq):
                getattr(m, call)(X, sample_weight=w)
                if impl == "sklearn":
                    _result(m, f"{name}_{i}", out)
                else:
                    _check(m, f"{name}_{i}", out, True, X.dtype == np.float32)
    np.savez_compressed(os.path.join(HERE, "minibatch_sklearn_weighted.npz"), **out)
    print("weighted minibatch goldens ok:", len(FIT_CASES), "fit cases,", len(PARTIAL_CASES), "partial_fit sequences")


if __name__ == "__main__":
    make_minibatch_weighted_golden()
