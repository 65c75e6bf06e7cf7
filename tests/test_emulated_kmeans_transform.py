"""KMeans.transform / fit_transform and MiniBatchKMeans.transform / fit_transform on CPU: the .cu sources under the
emulation (tests/emu), at small shapes.  The distances must meet the bars of tests/transform_bars.py against the exact
distance and against scikit-learn 1.9.0 (tests/golden, make_transform_golden.py) on both kernel forms, an element must
not depend on the form or the rows around it, and the estimators must follow sklearn's types.  The `-m gpu` twins are in
tests/test_gpu_kmeans_transform.py."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN
from tests.transform_bars import check_exact, check_sklearn

E = pytest.importorskip("tests.emu.emu_lib")
from opticalflowclustering_b200 import kmeans as km    # noqa: E402
from opticalflowclustering_b200 import minibatch as mb  # noqa: E402

sys.path.insert(0, GOLDEN)
import make_transform_golden as TG                      # noqa: E402


@pytest.fixture(scope="module")
def L():
    E.build()
    km._use_test_library(E.lib())
    yield E.lib()
    km._use_test_library(None)


def _estimator(name):
    est, _, _, _, _, k, _, _, rs = TG.TRANSFORM_CASES[name]
    return (km.KMeans if est == "KMeans" else mb.MiniBatchKMeans)(n_clusters=k, random_state=rs)


def _rows(dt, n, d, seed, off=0.0):
    rng = np.random.default_rng(seed)
    X = rng.normal(0, 40, (n, d)) + 120 + off
    return np.clip(np.rint(X), 0, 255).astype(np.uint8) if dt == np.uint8 else X.astype(dt)


@pytest.mark.parametrize("name", list(TG.TRANSFORM_CASES))
def test_transform_goldens(L, name):
    """sklearn's transform of its own centres, and the estimator's fit_transform against sklearn's"""
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_transform.npz"))
    X, Y, w = TG.transform_case(name)
    sk_c = z[name + "_centers"]
    Yc = TG.with_centres(Y, sk_c)
    got = km.transform(Yc, torch.from_numpy(sk_c)).numpy()
    check_sklearn(got, Yc, sk_c, z[name + "_transform"])
    check_exact(got, Yc, sk_c)
    est = _estimator(name)
    ft = est.fit_transform(X, sample_weight=w)
    assert isinstance(ft, np.ndarray) and ft.shape == (X.shape[0], sk_c.shape[0])
    rows = TG.FT_ROWS[TG.FT_ROWS < X.shape[0]]
    c_gap = np.sqrt(((est.cluster_centers_.astype(np.float64) - sk_c.astype(np.float64)) ** 2).sum(1))
    check_sklearn(ft[rows], X[rows], sk_c, z[name + "_fit_transform"], extra=c_gap[None])
    assert est.cluster_centers_.dtype == sk_c.dtype


# the small form (d <= 16, k <= 64) and the dense one (anything else), with data offset from the origin
@pytest.mark.parametrize("dt,n,d,k,off", [(np.uint8, 300, 3, 8, 0.0), (np.uint8, 200, 4, 64, 0.0), (np.float32, 150, 16, 16, 1e3),
                                         (np.float64, 130, 32, 20, 1e4), (np.float64, 140, 5, 70, 0.0),
                                         (np.float32, 100, 40, 130, 1e3), (np.uint8, 70, 33, 9, 0.0), (np.float64, 40, 600, 5, 0.0)])
@pytest.mark.parametrize("c_f32", [False, True])
def test_exact_distance_bar_on_each_form(L, dt, n, d, k, off, c_f32):
    X = _rows(dt, n, d, n + d, off)
    Cc = _rows(np.float64, k, d, k, off)
    Cc[1] = X[3]                                             # a row equal to a centre: exactly 0
    if c_f32:
        Cc = Cc.astype(np.float32)
        if dt == np.float64:
            X[3] = Cc[1]
    out = km.transform(X, torch.from_numpy(Cc))
    assert out.dtype == (torch.float32 if (dt == np.float32 and c_f32) else torch.float64)
    check_exact(out.numpy(), X, Cc)
    assert float(out[3, 1]) == 0.0


def test_element_does_not_depend_on_form_or_neighbours(L):
    X = _rows(np.float64, 150, 6, 1, 1e3)
    Cc = _rows(np.float64, 80, 6, 2, 1e3)
    full = km.transform(X, Cc)                              # k = 80: the dense form
    assert torch.equal(full[:, :8], km.transform(X, Cc[:8]))  # k = 8: the small form
    assert torch.equal(km.transform(X[37:101], Cc), full[37:101])
    Xf = X.astype(np.float32)
    cf = Cc.astype(np.float32)
    assert torch.equal(km.transform(Xf, cf)[:, :8], km.transform(Xf, cf[:8]))
    assert torch.equal(km.transform(Xf[5:9], cf), km.transform(Xf, cf)[5:9])


def test_float32_output_needs_float32_rows(L):
    X = np.zeros((4, 3), np.float64)
    Cc = np.zeros((2, 3), np.float64)
    out = np.zeros((4, 2), np.float32)
    p = lambda a: C.c_void_p(a.ctypes.data)                 # noqa: E731
    for dt, x in ((0, X.astype(np.uint8)), (2, X)):
        assert L.ofc_kmeans_distances(p(x), dt, C.c_int64(4), 3, 2, p(Cc), p(out), 1, C.c_void_p(0)) == -1
    assert L.ofc_kmeans_distances(p(X.astype(np.float32)), 1, C.c_int64(4), 3, 2, p(Cc), p(out), 1, C.c_void_p(0)) == 0
    assert L.ofc_kmeans_distances(p(X), 3, C.c_int64(4), 3, 2, p(Cc), p(out), 0, C.c_void_p(0)) == -1
    with pytest.raises(ValueError):
        km.transform(np.zeros((0, 3)), Cc)


@pytest.mark.parametrize("cls", [km.KMeans, mb.MiniBatchKMeans])
def test_estimator_types_and_fit_transform(L, cls):
    X = _rows(np.float32, 400, 5, 3)
    w = np.random.default_rng(0).uniform(0.5, 2.0, 400)
    ft = cls(n_clusters=4, random_state=0).fit_transform(X, sample_weight=w)
    est = cls(n_clusters=4, random_state=0).fit(X, sample_weight=w)
    assert np.array_equal(ft, est.transform(X)) and ft.dtype == np.float32
    assert est.transform(X.astype(np.float64)).dtype == np.float64          # sklearn's check_pairwise_arrays rule
    assert est.transform(X.astype(np.uint8)).dtype == np.float64
    assert est.transform(X.astype(np.int64)).dtype == np.float64
    t = est.transform(torch.from_numpy(X))
    assert isinstance(t, torch.Tensor) and t.dtype == torch.float32 and torch.equal(t, torch.from_numpy(ft))
    # a float32 fit measures against float32 centres, also when the rows are float64
    c32 = est.cluster_centers_.astype(np.float32).astype(np.float64)
    assert torch.equal(torch.from_numpy(est.transform(X.astype(np.float64))), km.transform(X.astype(np.float64), c32))
    e64 = cls(n_clusters=4, random_state=0).fit(X.astype(np.float64))
    assert e64.transform(X).dtype == np.float64
    with pytest.raises(ValueError, match=f"X has 6 features, but {cls.__name__} is expecting 5 features as input."):
        est.transform(np.zeros((3, 6), np.float32))
    # a torch float32 fit is a float32 fit too
    et = cls(n_clusters=4, random_state=0).fit(torch.from_numpy(X))
    assert et.transform(X.astype(np.float64)).dtype == np.float64
    assert np.array_equal(et.transform(X.astype(np.float64)),
                          km.transform(X.astype(np.float64), et._centres_t.to(torch.float32).to(torch.float64)).numpy())
