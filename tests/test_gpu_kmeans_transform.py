"""KMeans.transform / fit_transform and MiniBatchKMeans.transform on the B200: the goldens of make_transform_golden.py,
every shape of tools/kmeans_transform_bench.py against a float64 direct-difference reference on the GPU, the
independence of an element from the kernel form and the neighbouring rows at 1 M rows, CUDA tensors in and out, and an
output of more than 2^31 elements.  The CPU twins are in tests/test_emulated_kmeans_transform.py."""
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN
from tests.transform_bars import check_exact, check_sklearn

pytestmark = pytest.mark.gpu

from opticalflowclustering_b200 import kmeans as km    # noqa: E402
from opticalflowclustering_b200 import minibatch as mb  # noqa: E402

sys.path.insert(0, GOLDEN)
import make_transform_golden as TG                      # noqa: E402

# the shapes of tools/kmeans_transform_bench.py: (n, d, dtype, k)
BENCH_SHAPES = [(2_073_600, 3, torch.uint8, 8), (2_073_600, 4, torch.uint8, 8), (1_000_000, 16, torch.float32, 16),
                (1_000_000, 128, torch.float32, 256), (1_000_000, 512, torch.float32, 256)]


def _rows(n, d, dt, seed, off=0.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.randn((n, d), generator=g, device="cuda", dtype=torch.float64) * 40 + 120 + off
    return X.round().clamp(0, 255).to(torch.uint8) if dt == torch.uint8 else X.to(dt)


def _reference(X, C, chunk=1 << 17):
    """float64 direct difference, chunked over rows (a reduction of its own: within (d + 2) 2^-53 of the exact value)"""
    Cd = C.to(torch.float64)
    out = torch.empty((X.shape[0], C.shape[0]), dtype=torch.float64, device=X.device)
    for a in range(0, X.shape[0], chunk):
        xs = X[a:a + chunk].to(torch.float64)
        acc = torch.zeros((xs.shape[0], C.shape[0]), dtype=torch.float64, device=X.device)
        for t in range(X.shape[1]):
            df = xs[:, t:t + 1] - Cd[None, :, t]
            acc.addcmul_(df, df)
        out[a:a + chunk] = acc.sqrt_()
    return out


def _check_against_reference(out, ref, d):
    """the exact bar, widened by the reference's own error"""
    rel = (d + 2) * 2.0 ** -53
    if out.dtype == torch.float32:
        ulp = torch.abs(torch.nextafter(ref.float(), torch.tensor(float("inf"), device=ref.device)) - ref.float()).double()
        tol = ulp * (1 + 1e-6) + 2 * rel * ref
    else:
        tol = 2 * rel * ref
    assert bool(((out.double() - ref).abs() <= tol).all())


@pytest.mark.parametrize("name", list(TG.TRANSFORM_CASES))
def test_transform_goldens(name):
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_transform.npz"))
    X, Y, w = TG.transform_case(name)
    sk_c = z[name + "_centers"]
    Yc = TG.with_centres(Y, sk_c)
    got = km.transform(Yc, torch.from_numpy(sk_c)).cpu().numpy()
    check_sklearn(got, Yc, sk_c, z[name + "_transform"])
    check_exact(got, Yc, sk_c)
    est, _, _, _, _, k, _, _, rs = TG.TRANSFORM_CASES[name]
    e = (km.KMeans if est == "KMeans" else mb.MiniBatchKMeans)(n_clusters=k, random_state=rs)
    ft = e.fit_transform(X, sample_weight=w)
    rows = TG.FT_ROWS[TG.FT_ROWS < X.shape[0]]
    c_gap = np.sqrt(((e.cluster_centers_.astype(np.float64) - sk_c.astype(np.float64)) ** 2).sum(1))
    check_sklearn(ft[rows], X[rows], sk_c, z[name + "_fit_transform"], extra=c_gap[None])


@pytest.mark.parametrize("n,d,dt,k", BENCH_SHAPES)
def test_bench_shapes_against_reference(n, d, dt, k):
    X = _rows(n, d, dt, d)
    Cc = _rows(k, d, torch.float64, k + 1)
    if dt == torch.float32:
        Cc = Cc.to(torch.float32)
    Cc[1] = X[7].to(Cc.dtype)
    out = km.transform(X, Cc)
    assert out.is_cuda and out.dtype == (torch.float32 if dt == torch.float32 else torch.float64)
    _check_against_reference(out, _reference(X, Cc), d)
    assert float(out[7, 1]) == 0.0


@pytest.mark.parametrize("dt", [torch.float32, torch.float64])
def test_element_does_not_depend_on_form_or_neighbours_at_1m_rows(dt):
    X = _rows(1_000_000, 16, dt, 3, 1e3)
    Cc = _rows(200, 16, dt, 4, 1e3)
    full = km.transform(X, Cc)                                   # k = 200: the dense form
    assert torch.equal(full[:, :8], km.transform(X, Cc[:8]))     # k = 8: the small form
    assert torch.equal(km.transform(X[123_457:876_543], Cc), full[123_457:876_543])


@pytest.mark.parametrize("cls", [km.KMeans, mb.MiniBatchKMeans])
def test_cuda_tensor_in_gives_cuda_tensor_out(cls):
    X = _rows(300_000, 4, torch.uint8, 5)
    e = cls(n_clusters=8, random_state=0)
    ft = e.fit_transform(X)
    assert isinstance(ft, torch.Tensor) and ft.is_cuda and ft.dtype == torch.float64 and ft.shape == (300_000, 8)
    Y = _rows(50_000, 4, torch.uint8, 6)
    t = e.transform(Y)
    assert t.is_cuda and torch.equal(t, km.transform(Y, e._centres_t))
    Xf = _rows(200_000, 16, torch.float32, 7)
    tf = cls(n_clusters=16, random_state=0).fit(Xf).transform(Xf)
    assert tf.is_cuda and tf.dtype == torch.float32
    assert isinstance(e.transform(Y.cpu().numpy()), np.ndarray)


def test_output_beyond_two_to_the_31_elements():
    n, d, k = 2_200_000, 4, 1024                                  # n k = 2.25e9
    X = _rows(n, d, torch.float32, 8)
    Cc = _rows(k, d, torch.float32, 9)
    out = km.transform(X, Cc)
    rows = np.r_[0, 1, n - 2, n - 1, np.random.default_rng(0).integers(0, n, 2000)]
    rows_t = torch.from_numpy(rows).cuda()
    check_exact(out[rows_t].cpu().numpy(), X[rows_t].cpu().numpy(), Cc.cpu().numpy())
