"""KMeans.fit(X, sample_weight=w) on the B200: the goldens of make_weighted_golden.py (the d = 64 float32 case on the
tensor cores), weights of all ones against the unweighted fit at the shapes of every kernel path, and a shared-row batch
of weighted starts against the single weighted starts.  The CPU twins are in tests/test_emulated_kmeans_weighted.py."""
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu

from opticalflowclustering_b200 import kmeans as km    # noqa: E402

sys.path.insert(0, GOLDEN)
import make_weighted_golden as WG                        # noqa: E402


def _rows(n, d, dt, k, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    cen = torch.rand((k + 2, d), generator=g, device="cuda", dtype=torch.float64) * 210 + 20
    X = cen[torch.randint(0, k + 2, (n,), generator=g, device="cuda")] + torch.randn((n, d), generator=g, device="cuda",
                                                                                       dtype=torch.float64) * 15
    return X.round().clamp(0, 255).to(torch.uint8) if dt == torch.uint8 else X.to(dt)


def _starts(X, k, R, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    init = torch.stack([X[torch.randperm(X.shape[0], generator=g, device="cuda")[:k]] for _ in range(R)]).to(torch.float64)
    init[:, 1] = init[:, 0]          # two equal initial centres: an empty cluster, relocated in the first iteration
    return init


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("name", list(WG.WEIGHTED_CASES))
def test_gpu_weighted_fit_reproduces_sklearn(name):
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_weighted.npz"))
    _, n, d, k, init, n_init, seed, _w = WG.WEIGHTED_CASES[name]
    X, w = WG.weighted_case(name)
    Xt = torch.from_numpy(X).cuda()
    wt = torch.from_numpy(w).cuda()
    f32 = X.dtype == np.float32
    if name == "f32_d64_k8_pp1":
        assert km._tc_wanted(Xt.unsqueeze(0), k)
    if init == "explicit":
        clt = km.KMeans(n_clusters=k, init=X[WG.PROBE_INIT_ROWS].astype(np.float64)).fit(Xt, sample_weight=wt)
    else:
        R = z[name + "_seed_idx"].shape[0]
        if init == "random":
            cen, idx = km.random_starts(Xt, k, R, np.random.RandomState(seed), wt)
        else:
            cen, idx = km.kmeans_plusplus_starts(Xt, k, R, np.random.RandomState(seed), wt)
        assert (idx == z[name + "_seed_idx"]).all()
        labels, _, inertia, n_iter = km.lloyd(Xt, cen, sample_weight=wt)
        assert (n_iter.cpu().numpy() == z[name + "_start_niter"]).all()
        rel = 1e-5 if f32 else 1e-9
        assert np.all(np.abs(inertia.cpu().numpy() - z[name + "_start_inertia"]) <= rel * z[name + "_start_inertia"])
        assert km.best_start(labels, inertia, k) == int(z[name + "_best"])
        clt = km.KMeans(n_clusters=k, init=init, n_init=n_init, random_state=seed).fit(Xt, sample_weight=wt)
    ref_c, ref_i = z[name + "_centers"], float(z[name + "_inertia"])
    assert (clt.labels_ == z[name + "_labels"]).all() and clt.n_iter_ == int(z[name + "_niter"])
    if f32:
        assert np.abs(clt.cluster_centers_ - ref_c).max() < 1e-3 and abs(clt.inertia_ - ref_i) <= 1e-5 * ref_i
    else:
        assert np.abs(clt.cluster_centers_ - ref_c).max() <= 1e-9
        assert abs(clt.inertia_ - ref_i) <= 1e-9 * max(ref_i, 1.0)


# the fused uint8 step (d = 4) against the weighted two-kernel iteration, the float32 CUDA-core path, and the tensor-core
# path for float32 (d = 64) and for uint8 (d = 352, k = 256)
@pytest.mark.parametrize("n,d,dt,k", [(1_000_000, 4, torch.uint8, 8), (200_000, 16, torch.float32, 16),
                                      (1_000_000, 64, torch.float32, 64), (1_000_000, 352, torch.uint8, 256)])
def test_gpu_unit_weights_give_the_unweighted_bits(n, d, dt, k):
    X = _rows(n, d, dt, k, d)
    init = _starts(X, k, 1, k)[0]
    if d >= 64:
        assert km._tc_wanted(X.unsqueeze(0), k)
    ones = torch.ones(n, dtype=torch.float64, device="cuda")
    assert _same(km.lloyd(X, init, max_iter=30, sample_weight=ones), km.lloyd(X, init, max_iter=30))


def test_gpu_weighted_shared_row_batch_equals_single_starts():
    X = _rows(1_000_000, 4, torch.uint8, 8, 1)
    w = torch.rand(1_000_000, generator=torch.Generator(device="cuda").manual_seed(2), device="cuda", dtype=torch.float64) * 3
    init = _starts(X, 8, 10, 3)
    got = km.lloyd(X, init, sample_weight=w)
    for r in range(10):
        assert _same([t[r] for t in got], km.lloyd(X, init[r], sample_weight=w)), r
