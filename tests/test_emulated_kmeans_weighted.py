"""KMeans.fit(X, sample_weight=w) on CPU: the .cu sources under the emulation (tests/emu), driven through kmeans.py.
The weighted fit must reproduce sklearn 1.9.0 (tests/golden, make_weighted_golden.py), weights of all ones must give
exactly the bits of the unweighted fit on every kernel path, a shared-row batch of weighted starts must give each
start's single weighted fit, and the lockstep weighted seeding the seeds of sequential weighted kmeans_plusplus calls.
The `-m gpu` twins are in tests/test_gpu_kmeans_weighted.py."""
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN

E = pytest.importorskip("tests.emu.emu_lib")
from opticalflowclustering_b200 import kmeans as km    # noqa: E402

sys.path.insert(0, GOLDEN)
import make_weighted_golden as WG                        # noqa: E402


@pytest.fixture(scope="module")
def L():
    E.build()
    km._use_test_library(E.lib())
    yield E.lib()
    km._use_test_library(None)


def _rows(dt, n, d, k, seed):
    rng = np.random.default_rng(seed)
    cen = rng.uniform(20, 230, (k + 2, d))
    X = cen[rng.integers(k + 2, size=n)] + rng.normal(0, 15, (n, d))
    return np.clip(np.rint(X), 0, 255).astype(dt) if dt == np.uint8 else X.astype(dt)


def _starts(X, k, R, seed):
    rng = np.random.default_rng(seed)
    init = np.stack([X[rng.choice(X.shape[0], k, replace=False)] for _ in range(R)]).astype(np.float64)
    init[:, 1] = init[:, 0]          # two equal initial centres: an empty cluster, relocated in the first iteration
    return init


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("name", list(WG.WEIGHTED_CASES))
def test_weighted_fit_reproduces_sklearn(L, name):
    """every start's seeds, inertia and n_iter, the kept start, and its labels / n_iter exactly; centres and inertia to
    1e-9 (uint8, float64) or the float32 bars"""
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_weighted.npz"))
    _, n, d, k, init, n_init, seed, _w = WG.WEIGHTED_CASES[name]
    X, w = WG.weighted_case(name)
    Xt = torch.from_numpy(X)
    f32 = X.dtype == np.float32
    if init == "explicit":
        clt = km.KMeans(n_clusters=k, init=X[WG.PROBE_INIT_ROWS].astype(np.float64)).fit(X, sample_weight=w)
    else:
        R = z[name + "_seed_idx"].shape[0]
        if init == "random":
            cen, idx = km.random_starts(Xt, k, R, np.random.RandomState(seed), w)
        else:
            cen, idx = km.kmeans_plusplus_starts(Xt, k, R, np.random.RandomState(seed), w)
        assert (idx == z[name + "_seed_idx"]).all()
        labels, _, inertia, n_iter = km.lloyd(Xt, cen, sample_weight=w)
        assert (n_iter.numpy() == z[name + "_start_niter"]).all()
        rel = 1e-5 if f32 else 1e-9
        assert np.all(np.abs(inertia.numpy() - z[name + "_start_inertia"]) <= rel * z[name + "_start_inertia"])
        assert km.best_start(labels, inertia, k) == int(z[name + "_best"])
        clt = km.KMeans(n_clusters=k, init=init, n_init=n_init, random_state=seed).fit(X, sample_weight=w)
    ref_c, ref_i = z[name + "_centers"], float(z[name + "_inertia"])
    assert (clt.labels_ == z[name + "_labels"]).all() and clt.n_iter_ == int(z[name + "_niter"])
    if f32:
        assert clt.cluster_centers_.dtype == np.float32
        assert np.abs(clt.cluster_centers_ - ref_c).max() < 1e-3 and abs(clt.inertia_ - ref_i) <= 1e-5 * ref_i
    else:
        assert np.abs(clt.cluster_centers_ - ref_c).max() <= 1e-9
        assert abs(clt.inertia_ - ref_i) <= 1e-9 * max(ref_i, 1.0)


# uint8 through the d = 4 fused step and the generic fused step when unweighted (the weighted fit takes two kernels)
# and through the two-kernel path at d = 40; float32 and float64 through the small and medium E-steps.  Every start
# has two equal initial centres, so a cluster is relocated.
@pytest.mark.parametrize("dt,n,d,k", [(np.uint8, 1003, 4, 8), (np.uint8, 803, 7, 4), (np.uint8, 400, 40, 6),
                                      (np.float32, 700, 5, 4), (np.float32, 300, 40, 5), (np.float64, 600, 3, 4)])
def test_unit_weights_give_the_unweighted_bits(L, dt, n, d, k):
    X = _rows(dt, n, d, k, n + d)
    init = _starts(X, k, 2, k)
    ones = np.ones(n)
    for r in range(2):
        assert _same(km.lloyd(X, init[r], sample_weight=ones), km.lloyd(X, init[r])), r
    assert _same(km.lloyd(X, init, sample_weight=ones), km.lloyd(X, init))          # a shared-row batch
    if dt == np.uint8:
        # against the two-kernel unweighted path too (the fused step is bit-identical to it)
        os.environ["OFC_KMEANS_FUSED"] = "0"
        try:
            two = km.lloyd(X, init[0])
        finally:
            del os.environ["OFC_KMEANS_FUSED"]
        assert _same(km.lloyd(X, init[0], sample_weight=torch.ones(n, dtype=torch.float64)), two)
    clt = km.KMeans(n_clusters=k, n_init=3, random_state=1).fit(X, sample_weight=ones)
    ref = km.KMeans(n_clusters=k, n_init=3, random_state=1).fit(X)
    assert (clt.labels_ == ref.labels_).all() and (clt.cluster_centers_ == ref.cluster_centers_).all()
    assert clt.inertia_ == ref.inertia_ and clt.n_iter_ == ref.n_iter_


@pytest.mark.parametrize("dt,d", [(np.uint8, 4), (np.float32, 6), (np.float64, 3)])
def test_weighted_shared_row_batch_equals_single_starts(L, dt, d):
    X = _rows(dt, 900, d, 5, d)
    w = np.random.default_rng(d).uniform(0.0, 3.0, 900)
    init = _starts(X, 5, 4, 2)
    got = km.lloyd(X, init, sample_weight=w)
    for r in range(4):
        assert _same([t[r] for t in got], km.lloyd(X, init[r], sample_weight=w)), r


def test_weighted_lockstep_seeds_equal_sequential_kmeans_plusplus(L):
    X = _rows(np.uint8, 2000, 4, 6, 4)
    w = np.random.default_rng(0).uniform(0.0, 2.0, 2000) * (np.arange(2000) % 3 != 0)
    c, idx = km.kmeans_plusplus_starts(X, 6, 3, np.random.RandomState(11), w)
    rs = np.random.RandomState(11)
    for r in range(3):
        c1, i1 = km.kmeans_plusplus(X, 6, rs, sample_weight=w)
        assert (i1 == idx[r]).all() and torch.equal(c1, c[r]), r
        assert (w[i1] > 0).all()                                 # a row of weight 0 is never a seed


def test_zero_weight_members_count_as_empty(L):
    """the probe of sklearn's weighted relocation: the cluster of row 4 (weight 0) is empty by weight and takes row 3"""
    X = np.array([[0, 0], [0, 1], [10, 10], [10, 12], [50, 50]], np.float64)
    w = np.array([1, 1, 1, 1, 0], np.float64)
    labels, centres, inertia, n_iter = km.lloyd(X, X[[0, 2, 4]], sample_weight=w)
    assert labels.tolist() == [0, 0, 1, 2, 2] and int(n_iter) == 2
    assert np.array_equal(centres.numpy(), [[0, 0.5], [10, 10], [10, 12]]) and float(inertia) == 0.5


def test_sample_weight_validation(L):
    X = _rows(np.uint8, 50, 4, 3, 1)
    clt = km.KMeans(n_clusters=3, random_state=0)
    for bad in (np.ones(49), np.ones((50, 1)), -np.ones(50), np.r_[np.nan, np.ones(49)], np.r_[np.inf, np.ones(49)],
                np.zeros(50)):
        with pytest.raises(ValueError):
            clt.fit(X, sample_weight=bad)
    with pytest.raises(NotImplementedError):
        km.lloyd(X, X[:3].astype(np.float64), sample_weight=np.ones(50), group=object())
    assert km._check_sample_weight(2, 4, torch.float32).dtype == np.float32       # a number: that weight for every row
    assert (km._check_sample_weight(2, 4, torch.uint8) == 2.0).all()


@pytest.mark.parametrize("dt", [np.uint8, np.float32, np.float64])
def test_score_is_minus_the_weighted_inertia(L, dt):
    X = _rows(dt, 800, 5, 4, 7)
    w = np.random.default_rng(1).uniform(0.0, 2.0, 800)
    clt = km.KMeans(n_clusters=4, random_state=0).fit(X, sample_weight=w)
    Y = _rows(dt, 300, 5, 4, 8)
    wy = np.random.default_rng(2).uniform(0.0, 2.0, 300).astype(np.float32 if dt == np.float32 else np.float64)
    c = clt.cluster_centers_.astype(np.float64)
    dist = ((Y.astype(np.float64)[:, None, :] - c[None]) ** 2).sum(-1)
    want = -(dist.min(axis=1) * wy.astype(np.float64)).sum()
    rel = 1e-5 if dt == np.float32 else 1e-12
    assert abs(clt.score(Y, sample_weight=wy) - want) <= rel * abs(want)
    assert abs(clt.score(Y) - -dist.min(axis=1).sum()) <= rel * dist.min(axis=1).sum()
