"""KMeans(n_init=R) and init="random" on the GPU (twins of tests/test_emulated_kmeans_ninit.py at larger sizes): the
sklearn 1.9.0 goldens, every start of a shared-row batch bit-identical to the same start alone, the tensor-core regime
(sequential starts), and no copy of X per start."""
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu

sys.path.insert(0, GOLDEN)
import make_ninit_golden as MG                           # noqa: E402


@pytest.fixture(scope="module")
def km():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from opticalflowclustering_b200 import _lib, kmeans
    _lib.lib()
    return kmeans


def _rows(dt, n, d, k, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    cen = torch.rand((k + 2, d), generator=g, device="cuda", dtype=torch.float64) * 210 + 20
    X = cen[torch.randint(0, k + 2, (n,), generator=g, device="cuda")]
    X = X + torch.randn((n, d), generator=g, device="cuda", dtype=torch.float64) * 15
    return X.round().clamp(0, 255).to(torch.uint8) if dt == torch.uint8 else X.to(dt)


def _same_as_single_starts(km, X, init, max_iter=300):
    got = km.lloyd(X, init, max_iter=max_iter)
    for r in range(init.shape[0]):
        one = km.lloyd(X, init[r], max_iter=max_iter)
        assert all(torch.equal(a[r], b) for a, b in zip(got, one)), r
    return got


@pytest.mark.parametrize("name", list(MG.NINIT_CASES))
def test_ninit_reproduces_sklearn(km, name):
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_ninit.npz"))
    _, n, d, k, init, n_init, seed = MG.NINIT_CASES[name]
    X = MG.ninit_case(name)
    R = z[name + "_seed_idx"].shape[0]
    Xt = torch.from_numpy(X).cuda()
    if init == "random":
        cen, idx = km.random_starts(Xt, k, R, np.random.RandomState(seed))
    else:
        cen, idx = km.kmeans_plusplus_starts(Xt, k, R, np.random.RandomState(seed))
    assert (idx == z[name + "_seed_idx"]).all()
    labels, _, inertia, n_iter = _same_as_single_starts(km, Xt, cen)
    assert (n_iter.cpu().numpy() == z[name + "_start_niter"]).all()
    assert km.best_start(labels, inertia, k) == int(z[name + "_best"])
    clt = km.KMeans(n_clusters=k, init=init, n_init=n_init, random_state=seed).fit(X)
    ref_c, ref_i = z[name + "_centers"], float(z[name + "_inertia"])
    if X.dtype == np.float32:
        assert (clt.labels_ == z[name + "_labels"]).mean() > 0.999 and clt.cluster_centers_.dtype == np.float32
        assert np.abs(clt.cluster_centers_ - ref_c).max() < 1e-3 and abs(clt.inertia_ - ref_i) <= 1e-5 * ref_i
    else:
        assert (clt.labels_ == z[name + "_labels"]).all() and clt.n_iter_ == int(z[name + "_niter"])
        assert np.abs(clt.cluster_centers_ - ref_c).max() < 1e-9 and abs(clt.inertia_ - ref_i) <= 1e-9 * ref_i


def test_lockstep_seeds_1m_u8(km):
    """1 M x 4 uint8 pixels, k = 8, 10 starts: lockstep seeds = 10 sequential kmeans_plusplus calls, and the shared-row
    batch = the 10 single fits (the d = 4 fused step, several grid CTAs per start)"""
    X = _rows(torch.uint8, 1_000_000, 4, 8, 1)
    cen, idx = km.kmeans_plusplus_starts(X, 8, 10, np.random.RandomState(7))
    rs = np.random.RandomState(7)
    for r in range(10):
        c1, i1 = km.kmeans_plusplus(X, 8, rs)
        assert (i1 == idx[r]).all() and torch.equal(c1, cen[r]), r
    _same_as_single_starts(km, X, cen)
    clt = km.KMeans(n_clusters=8, n_init=10, random_state=7).fit(X)
    labels, centres, inertia, _ = km.lloyd(X, cen)
    b = km.best_start(labels, inertia, 8)
    assert (clt.labels_ == labels[b].cpu().numpy()).all() and clt.inertia_ == float(inertia[b])


@pytest.mark.parametrize("dt,n,d,k,R", [(torch.float32, 200_000, 16, 16, 10), (torch.float32, 1_000_000, 8, 8, 10),
                                        (torch.float64, 400_000, 3, 5, 6)])
def test_float_shared_rows_equal_single_starts(km, dt, n, d, k, R):
    """float M-step sums are folded per split: a start in a batch must use the split count of a single problem
    (1 M rows and 10 starts: 245 splits alone, 60 if the batch divided the cap)"""
    X = _rows(dt, n, d, k, n + d)
    init, _ = km.random_starts(X, k, R, np.random.RandomState(d))
    init[1, 1] = init[1, 0]                                  # an empty cluster in the first iteration
    _same_as_single_starts(km, X, init)
    _same_as_single_starts(km, X, init, max_iter=5)


def test_tensor_core_regime_runs_starts_one_by_one(km):
    """float32 1 M x 64, k = 64, 3 starts: the single fit runs on the tensor cores, so do the starts"""
    X = _rows(torch.float32, 1_000_000, 64, 64, 3)
    assert km._tc_wanted(X.unsqueeze(0), 64)
    init, _ = km.random_starts(X, 64, 3, np.random.RandomState(0))
    _same_as_single_starts(km, X, init)


def test_no_copy_of_x_per_start(km):
    """KMeans(init="random", n_init=10) on 1 M x 256 uint8 rows (256 MB, CUDA-core path: k*d < 4096): the peak
    allocation grows by far less than the 2.56 GB that ten copies of X would take"""
    X = torch.randint(0, 256, (1_000_000, 256), dtype=torch.uint8, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.max_memory_allocated()
    clt = km.KMeans(n_clusters=8, init="random", n_init=10, random_state=0).fit(X)
    grown = torch.cuda.max_memory_allocated() - base
    print(f"\npeak allocation grew by {grown / 1e9:.3f} GB for 10 starts over 256 MB of rows")
    assert grown < 1e9 and clt.labels_.shape == (1_000_000,)
