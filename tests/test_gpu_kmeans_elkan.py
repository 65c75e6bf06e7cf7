"""KMeans(algorithm="elkan") on the B200: the scikit-learn goldens (tests/golden/kmeans_sklearn_elkan.npz), every launch form
the Elkan kernels choose by shape at 1 M rows against the numpy restatement tests/kmeans_elkan_np.py (bit for bit, bounds
included), and a shared-row batch of starts against its single starts.  CPU twins: tests/test_emulated_kmeans_elkan.py."""
import ctypes as C
import sys
import warnings

import numpy as np
import pytest
import torch

from tests import kmeans_elkan_np as EN
from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu

sys.path.insert(0, GOLDEN)
import make_elkan_golden as EG                              # noqa: E402
from tests.test_emulated_kmeans_elkan import check_fit, fit_case  # noqa: E402


@pytest.fixture(scope="module")
def km():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    from opticalflowclustering_b200 import kmeans
    kmeans._use_test_library(None)
    return kmeans


@pytest.mark.parametrize("name", list(EG.ELKAN_CASES))
def test_goldens_on_the_gpu(km, name):
    check_fit(name, fit_case(name))


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


# one shape per launch form (`form`: kmeans_elkan_form in kmeans_elkan.cu): geometry in shared memory or global (past
# 48 KB of centres, chd and dnc), row in registers
# (d <= 4, d <= 16) or re-read from memory (d > 16)
@pytest.mark.parametrize("dt,d,k,form", [(np.uint8, 4, 8, 6), (np.float32, 12, 16, 5), (np.float64, 24, 8, 4),
                                         (np.uint8, 3, 80, 2), (np.float32, 16, 120, 1), (np.float64, 20, 80, 0)])
def test_launch_forms_at_1m_rows(km, dt, d, k, form):
    from opticalflowclustering_b200 import _lib
    L = _lib.lib()
    n = 1 << 20
    rng = np.random.default_rng(d * k)
    X = (rng.integers(0, 256, (n, d), dtype=np.uint8) if dt == np.uint8 else rng.normal(0, 30, (n, d)).astype(dt))
    wdt = np.float32 if dt == np.float32 else np.float64
    mean = X.astype(wdt).mean(axis=0).astype(wdt).astype(np.float64)
    Xc = X.astype(wdt) - mean.astype(wdt)
    C0 = Xc[rng.choice(n, k, replace=False)].astype(np.float64)
    C0[1] = C0[0]
    C1 = (C0 + rng.normal(0, 6.0, C0.shape)).astype(wdt).astype(np.float64)
    dev = torch.device("cuda")
    tX, tm = torch.from_numpy(X).to(dev), torch.from_numpy(mean).to(dev)
    tdt = torch.float32 if wdt == np.float32 else torch.float64
    code = {np.uint8: 0, np.float32: 1, np.float64: 2}[dt]
    geo = []
    for Cc in (C0, C1):
        tc = torch.from_numpy(Cc).to(dev)
        chd = torch.empty((k, k), dtype=tdt, device=dev)
        dnc = torch.empty(k, dtype=tdt, device=dev)
        ws = torch.empty(k * d * 4 + 256, dtype=torch.uint8, device=dev)
        _lib.check(L.ofc_kmeans_elkan_centres(code, 1, d, k, _ptr(tc), _ptr(chd), _ptr(dnc), _ptr(ws), ws.numel(), None))
        geo.append((tc, chd, dnc))
    lab0 = torch.empty(n, dtype=torch.int32, device=dev)
    lab1 = torch.empty(n, dtype=torch.int32, device=dev)
    up = torch.empty(n, dtype=tdt, device=dev)
    lo = torch.empty((n, k), dtype=tdt, device=dev)
    changed = torch.zeros(1, dtype=torch.int64, device=dev)
    _lib.check(L.ofc_kmeans_elkan_init(_ptr(tX), code, 1, n, d, k, _ptr(tm), _ptr(geo[0][0]), _ptr(geo[0][1]), _ptr(lab0), _ptr(up),
                                       _ptr(lo), None, None))
    chd0 = geo[0][1].cpu().numpy()
    ol0, ou0, ow0 = EN.elkan_init(Xc, C0.astype(wdt), chd0)
    assert np.array_equal(lab0.cpu().numpy(), ol0) and np.array_equal(up.cpu().numpy(), ou0) and np.array_equal(lo.cpu().numpy(), ow0)
    _lib.check(L.ofc_kmeans_elkan_step(_ptr(tX), code, 1, n, d, k, _ptr(tm), _ptr(geo[1][0]), _ptr(geo[1][1]), _ptr(geo[1][2]), _ptr(lab0),
                                       _ptr(lab1), _ptr(lab0), _ptr(up), _ptr(lo), _ptr(changed), None, None, None))
    ol1, ou1, ow1, _ = EN.elkan_step(Xc, C1.astype(wdt), geo[1][1].cpu().numpy(), geo[1][2].cpu().numpy(), ol0, ou0, ow0)
    assert np.array_equal(lab1.cpu().numpy(), ol1) and np.array_equal(up.cpu().numpy(), ou1) and np.array_equal(lo.cpu().numpy(), ow1)
    assert int(changed[0]) == int((ol1 != ol0).sum())


def test_batch_of_starts_equals_single_starts(km):
    rng = np.random.default_rng(7)
    X = rng.integers(0, 256, (200_000, 4), dtype=np.uint8)
    Xd = torch.from_numpy(X).cuda()
    init, _ = km.kmeans_plusplus_starts(Xd, 8, 4, np.random.RandomState(0))
    w = torch.from_numpy(rng.uniform(0.5, 2, X.shape[0])).cuda()
    for sw in (None, w):
        batch = km.lloyd(Xd, init, sample_weight=sw, algorithm="elkan")
        for r in range(4):
            one = km.lloyd(Xd, init[r], sample_weight=sw, algorithm="elkan")
            for a, b in zip(batch, one):
                assert torch.equal(a[r], b)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        a = km.lloyd(Xd, init[0], algorithm="elkan")
        b = km.lloyd(Xd, init[0], sample_weight=torch.ones(X.shape[0], dtype=torch.float64, device="cuda"), algorithm="elkan")
    assert all(torch.equal(u, v) for u, v in zip(a, b))
