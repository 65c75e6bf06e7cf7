"""KMeans(algorithm="elkan") on CPU: the ofc_kmeans_elkan_* kernels under the emulation (tests/emu) against the numpy
restatement tests/kmeans_elkan_np.py (bit for bit, bounds included) and whole fits against scikit-learn 1.9.0
(tests/golden/kmeans_sklearn_elkan.npz, make_elkan_golden.py).  The `-m gpu` twins are in tests/test_gpu_kmeans_elkan.py."""
import ctypes as C
import os
import sys
import warnings

import numpy as np
import pytest
import torch

from tests import kmeans_elkan_np as EN
from tests.conftest import GOLDEN

E = pytest.importorskip("tests.emu.emu_lib")
from opticalflowclustering_b200 import kmeans as km    # noqa: E402

sys.path.insert(0, GOLDEN)
import make_elkan_golden as EG                          # noqa: E402

_DT = {np.uint8: 0, np.float32: 1, np.float64: 2}


@pytest.fixture(scope="module")
def L():
    E.build()
    km._use_test_library(E.lib())
    yield E.lib()
    km._use_test_library(None)


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


def kernel_init_step(L, X, mean, C0, C1, chd0, chd1, dnc1):
    """init_bounds_dense from centres C0, then one step with centres C1, through the C-ABI (one problem)"""
    n, d = X.shape
    k = C0.shape[0]
    wdt = np.float32 if X.dtype == np.float32 else np.float64
    lab0 = np.zeros(n, np.int32)
    up = np.zeros(n, wdt)
    lo = np.full((n, k), 7, wdt)                              # garbage: init writes every lower bound
    dt = _DT[X.dtype.type]
    assert L.ofc_kmeans_elkan_init(_p(X), dt, 1, C.c_int64(n), d, k, _p(mean), _p(C0), _p(chd0), _p(lab0), _p(up), _p(lo), _p(None),
                                   C.c_void_p(0)) == 0
    init = (lab0.copy(), up.copy(), lo.copy())
    lab1 = np.zeros(n, np.int32)
    changed = np.zeros(1, np.uint64)
    nd = np.zeros(1, np.uint64)
    assert L.ofc_kmeans_elkan_step(_p(X), dt, 1, C.c_int64(n), d, k, _p(mean), _p(C1), _p(chd1), _p(dnc1), _p(lab0), _p(lab1), _p(lab0),
                                   _p(up), _p(lo), _p(changed), _p(nd), _p(None), C.c_void_p(0)) == 0
    return init, (lab1, up, lo, int(changed[0]), int(nd[0]))


def _rows(kind, n, d, rng):
    if kind == "ties_u8":
        return rng.integers(0, 6, (n, d), dtype=np.uint8)
    if kind == "u8":
        return rng.integers(0, 256, (n, d), dtype=np.uint8)
    return rng.normal(0, 30, (n, d)).astype(np.float32 if kind == "f32" else np.float64)


# (rows, n, d, k): small d (row in registers), d = 16 and d = 21 (row from memory); k = 90 puts chd past shared memory
@pytest.mark.parametrize("kind,n,d,k", [("ties_u8", 700, 3, 7), ("u8", 500, 4, 8), ("f32", 400, 6, 9), ("f64", 400, 16, 5),
                                        ("f64", 300, 21, 6), ("f32", 300, 3, 90), ("ties_u8", 600, 2, 90), ("f64", 200, 33, 90)])
def test_kernel_init_and_step_match_the_oracle(L, kind, n, d, k):
    rng = np.random.default_rng(n + d + k)
    X = _rows(kind, n, d, rng)
    wdt = np.float32 if X.dtype == np.float32 else np.float64
    mean = X.astype(wdt).mean(axis=0).astype(wdt).astype(np.float64)
    Xc = X.astype(wdt) - mean.astype(wdt)
    C0 = Xc[rng.choice(n, k, replace=False)].astype(np.float64)
    C0[1] = C0[0]                                             # duplicate centres: chd and dnc = 0
    C1 = (C0 + rng.normal(0, 1.5 if kind == "ties_u8" else 8.0, C0.shape)).astype(wdt).astype(np.float64)
    C1[3] = C1[2]
    if kind == "ties_u8":
        C1 = np.rint(C1 * 2) / 2                              # exact ties between lattice rows and half-integer centres
    geo = []
    for Cc in (C0, C1):
        chd = np.zeros((k, k), wdt)
        dnc = np.zeros(k, wdt)
        ws = np.zeros(k * d * 4 + 256, np.uint8)
        assert L.ofc_kmeans_elkan_centres(_DT[X.dtype.type], 1, d, k, _p(Cc), _p(chd), _p(dnc), _p(ws), C.c_size_t(ws.size),
                                          C.c_void_p(0)) == 0
        assert np.array_equal(dnc, np.partition(chd, kth=1, axis=0)[1]) and np.array_equal(chd, chd.T)
        geo.append((chd, dnc))
    assert geo[0][1][0] == 0 and geo[0][1][1] == 0
    (l0, u0, w0), (l1, u1, w1, changed, nd) = kernel_init_step(L, X, mean, C0, C1, geo[0][0], geo[1][0], geo[1][1])
    Cw0, Cw1 = C0.astype(wdt), C1.astype(wdt)
    ol0, ou0, ow0 = EN.elkan_init(Xc, Cw0, geo[0][0])
    assert np.array_equal(l0, ol0) and np.array_equal(u0, ou0) and np.array_equal(w0, ow0)
    ol1, ou1, ow1, ond = EN.elkan_step(Xc, Cw1, geo[1][0], geo[1][1], ol0, ou0, ow0)
    assert np.array_equal(l1, ol1) and np.array_equal(u1, ou1) and np.array_equal(w1, ow1)
    assert changed == int((ol1 != ol0).sum()) and nd == ond


def test_bound_update_matches_the_oracle(L):
    rng = np.random.default_rng(3)
    for wdt, dt in ((np.float32, 1), (np.float64, 2)):
        n, k, d = 300, 7, 5
        old = rng.normal(0, 10, (k, d)).astype(wdt).astype(np.float64)
        new = (old + rng.normal(0, 0.5, (k, d))).astype(wdt).astype(np.float64)
        new[2] = old[2]
        lab = rng.integers(0, k, n).astype(np.int32)
        up = rng.uniform(0, 5, n).astype(wdt)
        lo = rng.uniform(0, 2, (n, k)).astype(wdt)
        want_u, want_l = EN.update_bounds(lab, up, lo, EN.center_shift(old.astype(wdt), new.astype(wdt)))
        ws = np.zeros(k * 8 + 256, np.uint8)
        assert L.ofc_kmeans_elkan_bounds(dt, 1, C.c_int64(n), d, k, _p(old), _p(new), _p(lab), _p(up), _p(lo), _p(None), _p(None), _p(ws),
                                         C.c_size_t(ws.size), C.c_void_p(0)) == 0
        assert np.array_equal(up, want_u) and np.array_equal(lo, want_l) and (lo == 0).any()


def test_shapes_that_do_not_fit_are_errors(L):
    X = np.zeros((10, 3))
    out = np.zeros(100)
    assert L.ofc_kmeans_elkan_init(_p(X), 2, 1, C.c_int64(10), 3, 1, _p(None), _p(X), _p(out), _p(out), _p(out), _p(out), _p(None),
                                   C.c_void_p(0)) == -1                                          # k = 1
    assert L.ofc_kmeans_elkan_centres(1, 1, 3, 4, _p(X), _p(out), _p(out), _p(None), C.c_size_t(0), C.c_void_p(0)) == -4
    assert L.ofc_kmeans_elkan_bounds(2, 1, C.c_int64(10), 3, 4, _p(X), _p(X), _p(out), _p(out), _p(out), _p(None), _p(None), _p(out),
                                     C.c_size_t(8), C.c_void_p(0)) == -4


def check_fit(name, est):
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_elkan.npz"))
    X, _, _ = EG.elkan_case(name)
    lab, cen, inertia, n_iter = z[name + "_labels"], z[name + "_centers"], float(z[name + "_inertia"]), int(z[name + "_n_iter"])
    if X.dtype == np.float32:
        assert (est.labels_ == lab).mean() >= 0.9995 and est.n_iter_ == n_iter
        assert abs(est.inertia_ - inertia) <= 1e-5 * abs(inertia)
    else:
        assert np.array_equal(est.labels_, lab) and est.n_iter_ == n_iter
        assert np.abs(est.cluster_centers_ - cen).max() <= 1e-9
        assert abs(est.inertia_ - inertia) <= 1e-9 * abs(inertia)


def fit_case(name):
    _, n, d, k, init, n_init, rs, _, max_iter = EG.ELKAN_CASES[name]
    X, w, init_arr = EG.elkan_case(name)
    init_p = init_arr if not isinstance(init_arr, str) else init
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        return km.KMeans(k, init=init_p, n_init=n_init, random_state=rs, max_iter=max_iter, algorithm="elkan").fit(X, sample_weight=w)


@pytest.mark.parametrize("name", list(EG.ELKAN_CASES))
def test_fits_match_sklearn_elkan(L, name):
    est = fit_case(name)
    check_fit(name, est)
    if name.startswith("ties"):                                # where Elkan's labels differ from Lloyd's, they are Elkan's
        z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_elkan.npz"))
        assert (z[name + "_labels"] != z[name + "_lloyd_labels"]).any()


def test_shared_row_batch_gives_single_starts(L):
    X, _, _ = EG.elkan_case("ties_u8_k7_s0")
    rs = np.random.RandomState(1)
    init, _ = km.kmeans_plusplus_starts(torch.from_numpy(X), 7, 3, rs)
    w = np.random.default_rng(0).uniform(0.5, 2, X.shape[0])
    for sw in (None, w):
        batch = km.lloyd(X, init, sample_weight=sw, algorithm="elkan")
        for r in range(3):
            one = km.lloyd(X, init[r], sample_weight=sw, algorithm="elkan")
            for a, b in zip(batch, one):
                assert torch.equal(a[r], b)


@pytest.mark.parametrize("dt", [np.uint8, np.float32, np.float64])
def test_unit_weights_equal_unweighted(L, dt):
    rng = np.random.default_rng(5)
    X = rng.integers(0, 40, (900, 4)).astype(dt)
    init = X[[1, 50, 300, 600, 800]].astype(np.float64)
    a = km.lloyd(X, init, algorithm="elkan")
    b = km.lloyd(X, init, sample_weight=np.ones(900), algorithm="elkan")
    for u, v in zip(a, b):
        assert torch.equal(u, v)


def test_estimator_parameters(L):
    X, _, _ = EG.elkan_case("cell_u8_k1")
    with pytest.raises(ValueError, match="'algorithm' parameter of KMeans"):
        km.KMeans(3, algorithm="full").fit(X)
    with pytest.warns(RuntimeWarning, match="algorithm='elkan' doesn't make sense for a single cluster. Using 'lloyd' instead."):
        est = km.KMeans(1, algorithm="elkan", random_state=0).fit(X)
    check_fit("cell_u8_k1", est)
    X0 = X.copy()
    est = km.KMeans(4, random_state=0, copy_x=False, verbose=0, algorithm="elkan").fit(X)
    assert np.array_equal(X, X0) and est.labels_.shape == (X.shape[0],)
    with pytest.raises(ValueError):
        km.lloyd(X, X[:3].astype(np.float64), algorithm="hamerly")
