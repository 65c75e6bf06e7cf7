"""MiniBatchKMeans on the B200: the goldens of make_minibatch_weighted_golden.py, the centre update against the left
fold (tests/minibatch_weighted_np.py update_fold) up to a whole 1080p frame, partial_fit on a 1080p clip frame by frame
(CUDA tensors and numpy arrays alike) and the unique-colour fit.  The CPU twins are in
tests/test_emulated_minibatch_weighted.py."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu

from opticalflowclustering_b200 import _lib                      # noqa: E402
from opticalflowclustering_b200.minibatch import MiniBatchKMeans  # noqa: E402
from opticalflowclustering_b200.synthetic import synthetic_clip   # noqa: E402
from tests import minibatch_weighted_np as MB                    # noqa: E402

sys.path.insert(0, GOLDEN)
import make_minibatch_weighted_golden as MG                      # noqa: E402

DT = {torch.uint8: 0, torch.float32: 1, torch.float64: 2}


def _vp(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def update(X, labels, w, c_old, ws):
    """one centre update on the device (ofc_minibatch_update, or _weighted with w)"""
    k, d = c_old.shape
    c_new, ws_new = torch.empty_like(c_old), ws.clone()
    lib = _lib.lib()
    head = (_vp(X), DT[X.dtype], X.shape[0], d, k, _vp(labels))
    tail = (_vp(c_old), _vp(c_new), _vp(ws_new), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(lib.ofc_minibatch_update(*head, *tail) if w is None else lib.ofc_minibatch_update_weighted(*head, _vp(w), *tail))
    return c_new.cpu().numpy(), ws_new.cpu().numpy()


def _inputs(n, k, dt, wkind, seed):
    rng = np.random.default_rng(seed)
    W = np.float32 if dt == np.float32 else np.float64
    X = rng.integers(0, 256, (n, 3)).astype(dt)
    if dt == np.float32:
        X = (X + rng.uniform(0, 1, X.shape)).astype(dt)
    labels = rng.integers(0, k, n).astype(np.int32)
    w = None if wkind is None else (rng.integers(0, 5, n).astype(np.float64) if wkind == "int"
                                    else rng.uniform(0, 3, n).astype(W).astype(np.float64))
    c_old = rng.uniform(0, 255, (k, 3)).astype(W).astype(np.float64)
    ws = rng.integers(0, 10 ** 6, k).astype(np.float64)
    ws[0] = 0.0
    c_old[1], ws[1] = float(W((1024 - 1e-3) / 3)), 3.0
    return X, labels, w, c_old, ws


CASES = [(np.uint8, None), (np.uint8, "int"), (np.uint8, "real"), (np.float32, None)]


@pytest.mark.parametrize("dt,wkind", CASES)
@pytest.mark.parametrize("k", [8, 64])
@pytest.mark.parametrize("n", [1024, 51200, 2073600])
def test_update_equals_the_left_fold(n, k, dt, wkind):
    X, labels, w, c_old, ws = _inputs(n, k, dt, wkind, n + k)
    want = MB.update_fold(X, labels, w, c_old, ws)
    got = update(*[torch.from_numpy(a).cuda() if a is not None else None for a in (X, labels, w, c_old, ws)])
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def _check(m, z, prefix, f32, labels=True):
    assert int(m.n_steps_) == int(z[prefix + "_nsteps"]), prefix
    if labels:
        lab = m.labels_.cpu().numpy() if isinstance(m.labels_, torch.Tensor) else m.labels_
        assert (lab == z[prefix + "_labels"]).all(), prefix
    cen = m.cluster_centers_.cpu().numpy() if isinstance(m.cluster_centers_, torch.Tensor) else m.cluster_centers_
    tol, itol = (1e-3, 1e-5) if f32 else (1e-9, 1e-9)
    ref = z[prefix + "_centers"]
    assert np.abs(np.asarray(cen, np.float64) - ref).max() <= tol * max(1.0, np.abs(ref).max()), prefix
    assert np.abs(m._counts - z[prefix + "_counts"]).max() <= tol * max(1.0, z[prefix + "_counts"].max()), prefix
    assert abs(m.inertia_ - z[prefix + "_inertia"]) <= itol * max(1.0, abs(z[prefix + "_inertia"])), prefix


@pytest.mark.parametrize("name", list(MG.FIT_CASES))
def test_weighted_fit_reproduces_sklearn(name):
    z = np.load(os.path.join(GOLDEN, "minibatch_sklearn_weighted.npz"))
    X, w, k, kw = MG.fit_case(name)
    m = MiniBatchKMeans(n_clusters=k, **kw).fit(X, sample_weight=w)
    _check(m, z, name, X.dtype == np.float32, kw.get("compute_labels", True))


@pytest.mark.parametrize("name", list(MG.PARTIAL_CASES))
@pytest.mark.parametrize("as_tensor", [False, True])
def test_partial_fit_sequence_reproduces_sklearn(name, as_tensor):
    z = np.load(os.path.join(GOLDEN, "minibatch_sklearn_weighted.npz"))
    k, kw, seq = MG.partial_case(name)
    m = MiniBatchKMeans(n_clusters=k, **kw)
    for i, (call, X, w) in enumerate(seq):
        getattr(m, call)(torch.from_numpy(X).cuda() if as_tensor and call == "partial_fit" else X, sample_weight=w)
        _check(m, z, f"{name}_{i}", X.dtype == np.float32)


def test_partial_fit_1080p_clip_tensors_equal_numpy():
    clip = synthetic_clip(3, 1080, 1920, seed=4)
    a, b = MiniBatchKMeans(n_clusters=8, random_state=0), MiniBatchKMeans(n_clusters=8, random_state=0)
    for f in clip:
        px = f.reshape(-1, 3)
        a.partial_fit(px.cuda())
        b.partial_fit(px.numpy())
        assert isinstance(a.labels_, torch.Tensor) and a.labels_.is_cuda and a.cluster_centers_.is_cuda
        assert np.array_equal(a.labels_.cpu().numpy(), b.labels_) and np.array_equal(a.cluster_centers_.cpu().numpy(),
                                                                                     b.cluster_centers_)
        assert a.inertia_ == b.inertia_


def test_partial_fit_1080p_frame_reproduces_sklearn_restatement():
    """the whole-frame step (the exact-integer path) against the numpy restatement of sklearn's partial_fit"""
    px = synthetic_clip(1, 1080, 1920, seed=9)[0].reshape(-1, 3)
    m = MiniBatchKMeans(n_clusters=8, random_state=0).partial_fit(px.cuda())
    o = MB.MiniBatch(8, random_state=0).partial_fit(px.numpy())
    assert (m.labels_.cpu().numpy() == o.labels_).all()
    assert np.abs(m.cluster_centers_.cpu().numpy() - o.cluster_centers_).max() <= 1e-9


def test_fit_on_unique_colours_with_counts():
    X, w, k, kw = MG.fit_case("u8_unique_counts")
    m = MiniBatchKMeans(n_clusters=k, **kw).fit(torch.from_numpy(X).cuda(), sample_weight=w)
    o = MB.MiniBatch(k, **kw).fit(X, sample_weight=w)
    assert m.n_steps_ == o.n_steps_ and (m.labels_ == o.labels_).all()
    assert np.abs(m.cluster_centers_ - o.cluster_centers_).max() <= 1e-9
