"""Generate tests/golden/kmeans_sklearn_transform.npz: scikit-learn 1.9.0 ``KMeans`` / ``MiniBatchKMeans``
``cluster_centers_``, ``transform(Y)`` and ``fit_transform(X, sample_weight=w)``, for the tests of the transform.

    python tests/golden/make_transform_golden.py

The rows X, the rows Y and the weights are regenerated from each case's name by ``transform_case``, so the fixture
stores only the results.  Y is fresh rows of the case followed by the first fitted centres in Y's dtype (rows at distance 0
where that dtype holds a centre exactly).  ``fit_transform`` is stored for the rows ``FT_ROWS`` only, to keep the file
small."""
from __future__ import annotations

import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

TRANSFORM_CASES = {   # name: (estimator, X dtype, Y dtype, n, d, k, offset, weighted, random_state)
    "km_u8_d3_k8": ("KMeans", "uint8", "uint8", 600, 3, 8, 0.0, False, 0),
    "km_i64_d4_k5": ("KMeans", "int64", "int64", 500, 4, 5, 0.0, False, 1),
    "km_f32_d16_k16": ("KMeans", "float32", "float32", 800, 16, 16, 0.0, False, 2),
    "km_f64_d2_k4_off1e4": ("KMeans", "float64", "float64", 400, 2, 4, 1e4, False, 3),
    "km_f32_d64_k12_off1e3": ("KMeans", "float32", "float32", 600, 64, 12, 1e3, False, 4),
    "km_f64_d600_k6": ("KMeans", "float64", "float64", 150, 600, 6, 0.0, False, 5),
    "km_f32_d24_k256": ("KMeans", "float32", "float32", 600, 24, 256, 0.0, False, 6),
    "km_f32_fit_f64_rows": ("KMeans", "float32", "float64", 500, 6, 7, 0.0, False, 7),
    "km_f64_fit_f32_rows": ("KMeans", "float64", "float32", 500, 6, 7, 0.0, False, 8),
    "km_f64_d5_k6_weighted": ("KMeans", "float64", "float64", 600, 5, 6, 0.0, True, 9),
    "km_u8_d4_k8_weighted": ("KMeans", "uint8", "uint8", 600, 4, 8, 0.0, True, 10),
    "mb_u8_d3_k8": ("MiniBatchKMeans", "uint8", "uint8", 900, 3, 8, 0.0, False, 11),
    "mb_f32_d8_k6_weighted": ("MiniBatchKMeans", "float32", "float32", 700, 8, 6, 0.0, True, 12),
    "mb_f64_d5_k4_off1e3": ("MiniBatchKMeans", "float64", "float64", 600, 5, 4, 1e3, False, 13),
}

#: the rows of X whose fit_transform is stored
FT_ROWS = np.arange(0, 24) * 9
#: fresh rows in Y (the fitted centres follow them)
Y_ROWS = 24
#: fitted centres appended to Y
Y_CENTRES = 8


def transform_case(name):
    """regenerate (X, Y rows before the centres, weights or None) of a case from its name"""
    _, xdt, ydt, n, d, k, off, weighted, _ = TRANSFORM_CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    cen = rng.uniform(20, 230, (k, d))            # one well separated blob per cluster: a stable optimum
    lab = rng.integers(k, size=n + Y_ROWS)
    lab[:k] = np.arange(k)
    rows = cen[lab] + rng.normal(0, 6, (n + Y_ROWS, d)) + off

    def cast(a, dt):
        if dt == "uint8":
            return np.clip(np.rint(a), 0, 255).astype(np.uint8)
        if dt == "int64":
            return np.rint(a).astype(np.int64)
        return a.astype(dt)

    w = rng.uniform(0.2, 3.0, n) if weighted else None
    if w is not None and xdt == "float32":
        w = w.astype(np.float32)
    return cast(rows[:n], xdt), cast(rows[n:], ydt), w


def estimator(name):
    from sklearn.cluster import KMeans, MiniBatchKMeans
    est, _, _, _, _, k, _, _, rs = TRANSFORM_CASES[name]
    return (KMeans if est == "KMeans" else MiniBatchKMeans)(n_clusters=k, random_state=rs)


def with_centres(Y, centres):
    """Y's fresh rows followed by the first ``Y_CENTRES`` centres in Y's dtype"""
    return np.concatenate([Y, centres[:Y_CENTRES].astype(Y.dtype)])


def main():
    import sklearn
    assert sklearn.__version__ == "1.9.0", sklearn.__version__
    out = {}
    for name in TRANSFORM_CASES:
        X, Y, w = transform_case(name)
        est = estimator(name)
        ft = est.fit_transform(X, sample_weight=w)
        Yc = with_centres(Y, est.cluster_centers_)
        out[name + "_centers"] = est.cluster_centers_
        out[name + "_transform"] = est.transform(Yc)
        out[name + "_fit_transform"] = ft[FT_ROWS[FT_ROWS < X.shape[0]]]
    path = os.path.join(HERE, "kmeans_sklearn_transform.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
