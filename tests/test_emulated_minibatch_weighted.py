"""MiniBatchKMeans with sample weights, init="random" and partial_fit on CPU: the .cu sources under the emulation
(tests/emu), driven through minibatch.py.  The estimator must reproduce sklearn 1.9.0 (tests/golden,
make_minibatch_weighted_golden.py), and the centre update must give the bits of the left fold
(tests/minibatch_weighted_np.py update_fold) on every dtype, weight kind and path of its streaming kernel.  The
`-m gpu` twins are in tests/test_gpu_minibatch.py."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from tests.conftest import GOLDEN

E = pytest.importorskip("tests.emu.emu_lib")
from opticalflowclustering_b200 import kmeans as km            # noqa: E402
from opticalflowclustering_b200.minibatch import MiniBatchKMeans  # noqa: E402
from tests import minibatch_weighted_np as MB                  # noqa: E402

sys.path.insert(0, GOLDEN)
import make_minibatch_weighted_golden as MG                    # noqa: E402

DT = {np.uint8: 0, np.float32: 1, np.float64: 2}


@pytest.fixture(scope="module")
def L():
    E.build()
    km._use_test_library(E.lib())
    yield E.lib()
    km._use_test_library(None)


@pytest.fixture(scope="module")
def Z():
    return np.load(os.path.join(GOLDEN, "minibatch_sklearn_weighted.npz"))


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


def update(lib, X, labels, w, c_old, ws):
    """one centre update (ofc_minibatch_update, or _weighted with w); returns (centres, weight sums)"""
    k, d = c_old.shape
    c_new, ws_new = np.zeros_like(c_old), ws.copy()
    head = (_p(X), DT[X.dtype.type], X.shape[0], d, k, _p(labels))
    tail = (_p(c_old), _p(c_new), _p(ws_new), C.c_void_p(0))
    rc = lib.ofc_minibatch_update(*head, *tail) if w is None else lib.ofc_minibatch_update_weighted(*head, _p(w), *tail)
    assert rc == 0, lib.ofc_last_error()
    return c_new, ws_new


def fold_inputs(n, d, k, dt, wkind, seed):
    """rows, labels, weights, centres and weight sums with crossing-heavy starts: cluster 0 has weight sum 0, cluster 1
    starts just below a power of two (c_old * ws = 1024 - 1e-3), the others at large weight sums"""
    rng = np.random.default_rng(seed)
    W = np.float32 if dt == np.float32 else np.float64
    X = rng.integers(0, 256, (n, d)).astype(dt)
    if dt != np.uint8 and wkind == "real":
        X = (X + rng.uniform(0, 1, X.shape)).astype(dt)
    labels = rng.integers(0, k, n).astype(np.int32)
    w = None
    if wkind == "int":
        w = rng.integers(0, 4, n).astype(np.float64)
    elif wkind in ("real", "mixed"):
        w = rng.uniform(0, 3, n).astype(W).astype(np.float64)
        if wkind == "mixed":                        # integer weights in every other chunk of 512 rows: both paths
            even = (np.arange(n) // 512) % 2 == 0
            w[even] = np.rint(w[even])
        w[::7] = 0.0                                # members of weight 0
    c_old = rng.uniform(0, 255, (k, d)).astype(W).astype(np.float64)
    ws = rng.integers(1, 10 ** 6, k).astype(W).astype(np.float64)
    ws[0] = 0.0
    if k > 1:
        c_old[1], ws[1] = float(W((1024 - 1e-3) / 3)), 3.0
    return X, labels, w, c_old, ws


@pytest.mark.parametrize("dt", [np.uint8, np.float32, np.float64])
@pytest.mark.parametrize("wkind", [None, "int", "real", "mixed"])
@pytest.mark.parametrize("n,d,k", [(1, 1, 1), (2300, 3, 5), (700, 9, 3), (1500, 5, 12)])
def test_update_equals_the_left_fold(L, dt, wkind, n, d, k):
    """d > 4 takes several feature passes; "mixed" alternates the exact-integer and sequential paths chunk by chunk"""
    X, labels, w, c_old, ws = fold_inputs(n, d, k, dt, wkind, n + d)
    got = update(L, X, labels, w, c_old, ws)
    want = MB.update_fold(X, labels, w, c_old, ws)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_unit_weights_equal_the_unweighted_update(L):
    for dt in (np.uint8, np.float32, np.float64):
        X, labels, _, c_old, ws = fold_inputs(1800, 3, 6, dt, None, 3)
        assert all(np.array_equal(a, b) for a, b in zip(update(L, X, labels, np.ones(1800), c_old, ws),
                                                        update(L, X, labels, None, c_old, ws)))


def test_integer_path_crossings(L):
    """uint8 rows and integer weights (the exact-integer path) with a start just below many powers of two"""
    rng = np.random.default_rng(5)
    X = rng.integers(0, 256, (3000, 2)).astype(np.uint8)
    labels = np.zeros(3000, np.int32)
    w = rng.integers(0, 5, 3000).astype(np.float64)
    for start in (0.999, 255.5, 2.0 ** 20 - 0.25, 2.0 ** 40 - 0.5):
        c_old, ws = np.array([[start / 7, start / 7]]), np.array([7.0])
        want = MB.update_fold(X, labels, w, c_old, ws)
        assert all(np.array_equal(a, b) for a, b in zip(update(L, X, labels, w, c_old, ws), want)), start


def _check(m, z, prefix, f32, labels=True):
    assert int(m.n_steps_) == int(z[prefix + "_nsteps"]), prefix
    if labels:
        assert (np.asarray(m.labels_) == z[prefix + "_labels"]).all(), prefix
    tol, itol = (1e-3, 1e-5) if f32 else (1e-9, 1e-9)
    ref = z[prefix + "_centers"]
    assert np.abs(np.asarray(m.cluster_centers_, np.float64) - ref).max() <= tol * max(1.0, np.abs(ref).max()), prefix
    assert np.abs(m._counts - z[prefix + "_counts"]).max() <= tol * max(1.0, z[prefix + "_counts"].max()), prefix
    assert abs(m.inertia_ - z[prefix + "_inertia"]) <= itol * max(1.0, abs(z[prefix + "_inertia"])), prefix


@pytest.mark.parametrize("name", list(MG.FIT_CASES))
def test_weighted_fit_reproduces_sklearn(L, Z, name):
    X, w, k, kw = MG.fit_case(name)
    m = MiniBatchKMeans(n_clusters=k, **kw).fit(X, sample_weight=w)
    _check(m, Z, name, X.dtype == np.float32, kw.get("compute_labels", True))


@pytest.mark.parametrize("name", list(MG.PARTIAL_CASES))
def test_partial_fit_sequence_reproduces_sklearn(L, Z, name):
    k, kw, seq = MG.partial_case(name)
    m = MiniBatchKMeans(n_clusters=k, **kw)
    for i, (call, X, w) in enumerate(seq):
        getattr(m, call)(X, sample_weight=w)
        _check(m, Z, f"{name}_{i}", X.dtype == np.float32)


def test_oracle_reproduces_the_golden(Z):
    for name in MG.FIT_CASES:
        X, w, k, kw = MG.fit_case(name)
        o = MB.MiniBatch(k, **kw).fit(X, sample_weight=w)
        _check(o, Z, name, X.dtype == np.float32, kw.get("compute_labels", True))
    for name in MG.PARTIAL_CASES:
        k, kw, seq = MG.partial_case(name)
        o = MB.MiniBatch(k, **kw)
        for i, (call, X, w) in enumerate(seq):
            getattr(o, call)(X, sample_weight=w)
            _check(o, Z, f"{name}_{i}", X.dtype == np.float32)


def test_fit_with_a_batch_over_51200_rows(L):
    X, _, _ = _lab(70000, 3)
    m = MiniBatchKMeans(n_clusters=4, batch_size=60000, max_iter=2, random_state=0).fit(X)
    o = MB.MiniBatch(4, random_state=0, batch_size=60000, max_iter=2).fit(X)
    assert m.n_steps_ == o.n_steps_ and (m.labels_ == o.labels_).all()
    assert np.abs(m.cluster_centers_ - o.cluster_centers_).max() <= 1e-9


def _lab(n, seed):
    rng = np.random.default_rng(seed)
    cen = rng.uniform(30, 220, (6, 3))
    return np.clip(np.rint(cen[rng.integers(6, size=n)] + rng.normal(0, 9, (n, 3))), 0, 255).astype(np.uint8), rng, cen


def test_score_is_minus_the_weighted_inertia(L):
    X, rng, _ = _lab(3000, 2)
    w = rng.uniform(0, 2, 3000)
    m = MiniBatchKMeans(n_clusters=4, random_state=0).fit(X, sample_weight=w)
    c = m.cluster_centers_
    dist = ((X.astype(np.float64)[:, None, :] - c[None]) ** 2).sum(-1).min(axis=1)
    assert abs(m.score(X, sample_weight=w) - -(dist * w).sum()) <= 1e-12 * (dist * w).sum()
    assert m.score(X) == km.KMeans.score(m, X)


def test_validation(L):
    X, _, _ = _lab(500, 1)
    for bad in (np.ones(499), np.ones((500, 1)), -np.ones(500), np.r_[np.nan, np.ones(499)], np.zeros(500)):
        with pytest.raises(ValueError):
            MiniBatchKMeans(n_clusters=3, random_state=0).fit(X, sample_weight=bad)
        with pytest.raises(ValueError):
            MiniBatchKMeans(n_clusters=3, random_state=0).partial_fit(X, sample_weight=bad)
    m = MiniBatchKMeans(n_clusters=3, random_state=0).partial_fit(X)
    with pytest.raises(ValueError):
        m.partial_fit(np.zeros((100, 4), np.uint8))
    with pytest.raises(ValueError):
        MiniBatchKMeans(n_clusters=3, init="kmeans").fit(X)
