"""KMeans(n_init=R) and init="random" on CPU: the .cu sources under the emulation (tests/emu), driven through
kmeans.py.  Several starts of one fit run as one batch of problems that read the same rows
(OFC_KMEANS_SHARED_ROWS); every start must give exactly what it gives alone, the lockstep k-means++ seeding must give
the seeds of sequential kmeans_plusplus calls, and the fits must reproduce sklearn 1.9.0 (tests/golden,
make_ninit_golden.py).  The `-m gpu` twins are in tests/test_gpu_kmeans_ninit.py."""
import os
import sys
import warnings

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN

E = pytest.importorskip("tests.emu.emu_lib")
from opticalflowclustering_b200 import kmeans as km    # noqa: E402

sys.path.insert(0, GOLDEN)
import make_ninit_golden as MG                           # noqa: E402


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
    init[1, 1] = init[1, 0]          # two equal initial centres: an empty cluster, relocated in the first iteration
    return init


# uint8 through the d = 4 fused step (n % 4 != 0 too), the generic fused step (d = 7) and the two-kernel step
# (d = 40); float32 and float64 through the CUDA-core kernels (small and medium E-step)
@pytest.mark.parametrize("dt,n,d,k", [(np.uint8, 1000, 4, 5), (np.uint8, 1003, 4, 8), (np.uint8, 803, 7, 4),
                                      (np.uint8, 400, 40, 6), (np.float32, 700, 5, 4), (np.float32, 300, 40, 5),
                                      (np.float64, 600, 3, 4)])
@pytest.mark.parametrize("max_iter", [3, 300])
def test_shared_row_batch_equals_single_starts(L, dt, n, d, k, max_iter):
    X = _rows(dt, n, d, k, n + d)
    init = _starts(X, k, 4, k)
    got = km.lloyd(X, init, max_iter=max_iter)
    assert [t.shape[0] for t in got] == [4] * 4
    if max_iter == 300:
        assert len(set(got[3].tolist())) > 1                 # the starts stop at different iterations
    for r in range(4):
        one = km.lloyd(X, init[r], max_iter=max_iter)
        assert all(torch.equal(a[r], b) for a, b in zip(got, one)), r


def test_shared_row_batch_keeps_a_single_start(L):
    """init [1, k, d] over X [n, d]: a batch of one start, the bits of the single fit"""
    X = _rows(np.float64, 500, 3, 4, 9)
    init = _starts(X, 4, 2, 1)[:1]
    got = km.lloyd(X, init)
    one = km.lloyd(X, init[0])
    assert all(torch.equal(a[0], b) for a, b in zip(got, one))


def test_lockstep_seeds_equal_sequential_kmeans_plusplus(L):
    X = _rows(np.uint8, 2000, 4, 6, 4)
    R = 3
    c, idx = km.kmeans_plusplus_starts(X, 6, R, np.random.RandomState(11))
    rs = np.random.RandomState(11)
    for r in range(R):
        c1, i1 = km.kmeans_plusplus(X, 6, rs)
        assert (i1 == idx[r]).all() and torch.equal(c1, c[r]), r
    _, idx2 = km.kmeans_plusplus_starts(X, 6, R + 2, np.random.RandomState(11))
    assert (idx2[:R] == idx).all()                           # a start's seeds do not depend on the number of starts
    Xf = _rows(np.float32, 900, 5, 4, 6)
    _, i3 = km.kmeans_plusplus_starts(Xf, 4, 2, np.random.RandomState(2))
    rs = np.random.RandomState(2)
    assert all((km.kmeans_plusplus(Xf, 4, rs)[1] == i3[r]).all() for r in range(2))


@pytest.mark.parametrize("name", list(MG.NINIT_CASES))
def test_ninit_reproduces_sklearn(L, name):
    """KMeans(init, n_init, random_state) against sklearn 1.9.0: every start's seeds, inertia and n_iter, the winner,
    and the winner's labels / n_iter exactly, centres and inertia to the bars of the seeded test (float32: the bars
    of the float32 golden tests)"""
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_ninit.npz"))
    _, n, d, k, init, n_init, seed = MG.NINIT_CASES[name]
    X = MG.ninit_case(name)
    R = z[name + "_seed_idx"].shape[0]
    Xt = torch.from_numpy(X)
    if init == "random":
        cen, idx = km.random_starts(Xt, k, R, np.random.RandomState(seed))
    else:
        cen, idx = km.kmeans_plusplus_starts(Xt, k, R, np.random.RandomState(seed))
    assert (idx == z[name + "_seed_idx"]).all()
    labels, _, inertia, n_iter = km.lloyd(Xt, cen)
    assert (n_iter.numpy() == z[name + "_start_niter"]).all()
    assert np.all(np.abs(inertia.numpy() - z[name + "_start_inertia"]) <= 1e-5 * z[name + "_start_inertia"])
    assert km.best_start(labels, inertia, k) == int(z[name + "_best"])
    clt = km.KMeans(n_clusters=k, init=init, n_init=n_init, random_state=seed).fit(X)
    ref_c, ref_i = z[name + "_centers"], float(z[name + "_inertia"])
    if X.dtype == np.float32:
        assert (clt.labels_ == z[name + "_labels"]).mean() > 0.999 and clt.cluster_centers_.dtype == np.float32
        assert np.abs(clt.cluster_centers_ - ref_c).max() < 1e-3 and abs(clt.inertia_ - ref_i) <= 1e-5 * ref_i
    else:
        assert (clt.labels_ == z[name + "_labels"]).all() and clt.n_iter_ == int(z[name + "_niter"])
        assert np.abs(clt.cluster_centers_ - ref_c).max() < 1e-9 and abs(clt.inertia_ - ref_i) <= 1e-9 * ref_i
        assert np.all(np.abs(inertia.numpy() - z[name + "_start_inertia"]) <= 1e-9 * z[name + "_start_inertia"])


def test_choice_of_the_start():
    """sklearn's rule: a later start wins only with a strictly lower inertia AND a different clustering, where "same"
    means the map from its labels to the best start's labels is a function (not necessarily a bijection)"""
    best = torch.tensor([0, 0, 1, 1, 2, 2], dtype=torch.int32)
    perm = torch.tensor([2, 2, 0, 0, 1, 1], dtype=torch.int32)            # the same clustering, permuted
    merged = torch.tensor([0, 0, 0, 0, 1, 1], dtype=torch.int32)          # the best's clusters 0 and 1 merged
    split = torch.tensor([0, 1, 2, 2, 2, 2], dtype=torch.int32)           # a different clustering
    lab = torch.stack([best, perm])
    assert km.best_start(lab, torch.tensor([5.0, 4.0], dtype=torch.float64), 3) == 0
    assert km.best_start(torch.stack([best, split]), torch.tensor([5.0, 4.0], dtype=torch.float64), 3) == 1
    assert km.best_start(torch.stack([best, split]), torch.tensor([5.0, 5.0], dtype=torch.float64), 3) == 0
    assert not km._is_same_clustering(split, best, 3)          # the split's cluster 2 maps to best's 1 and 2
    # merged -> best: label 0 of `merged` covers best's 0 and 1: not a function; best -> merged is one
    assert not km._is_same_clustering(merged, best, 3) and km._is_same_clustering(best, merged, 3)
    # a start whose map to the best is a function (a coarser clustering of it) does not replace it
    assert km.best_start(torch.stack([merged, best]), torch.tensor([5.0, 4.0], dtype=torch.float64), 3) == 0
    assert km.best_start(torch.stack([best, merged, split]), torch.tensor([5.0, 4.0, 3.0], dtype=torch.float64), 3) == 2


def test_n_init_resolution():
    assert km._resolve_n_init("auto", "k-means++") == 1
    assert km._resolve_n_init("auto", "random") == 10
    assert km._resolve_n_init("auto", np.zeros((2, 3))) == 1
    assert km._resolve_n_init(3, "random") == 3 and km._resolve_n_init(np.int64(4), "k-means++") == 4
    for bad in (0, -1, "all", 2.5):
        with pytest.raises(ValueError):
            km._resolve_n_init(bad, "k-means++")
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        assert km._resolve_n_init(5, np.zeros((2, 3))) == 1
    assert any(issubclass(x.category, RuntimeWarning) and "performing only one init" in str(x.message) for x in w)
    with pytest.raises(ValueError):
        km.KMeans(n_clusters=2, init="kmeans").fit(np.zeros((4, 2)))


def test_explicit_init_runs_one_start(L):
    X = _rows(np.uint8, 600, 4, 3, 3)
    init = X[:3].astype(np.float64)
    with pytest.warns(RuntimeWarning, match="performing only one init"):
        clt = km.KMeans(n_clusters=3, init=init, n_init=4).fit(X)
    labels, centres, inertia, n_iter = km.lloyd(X, init)
    assert (clt.labels_ == labels.numpy()).all() and clt.n_iter_ == int(n_iter)
