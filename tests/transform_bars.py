"""The accuracy bars of KMeans.transform, shared by tests/test_emulated_kmeans_transform.py and
tests/test_gpu_kmeans_transform.py (not a test module).

* against the exact distance (direct difference in np.longdouble): float32 output within one float32 ulp, float64
  output within a relative (d + 2) 2^-53, a row equal to a centre exactly 0;
* against scikit-learn's transform: |lib - sk| <= sqrt((d + 2) 2^-52 (|x|^2 + |c|^2)) + 2 ulp(sk) in the output dtype --
  the cancellation error of sklearn's norm form, not the library's."""
import numpy as np


def exact_distances(X, C):
    """[n, k] Euclidean distances in np.longdouble, by the direct difference"""
    Xl = np.asarray(X).astype(np.longdouble)
    Cl = np.asarray(C).astype(np.longdouble)
    return np.sqrt(((Xl[:, None, :] - Cl[None]) ** 2).sum(-1))


def check_exact(out, X, C):
    out = np.asarray(out)
    d = np.asarray(X).shape[1]
    ex = exact_distances(X, C)
    if out.dtype == np.float32:
        tol = np.spacing(ex.astype(np.float32)).astype(np.longdouble)
    else:
        assert out.dtype == np.float64
        tol = ex * ((d + 2) * 2.0 ** -53)
    err = np.abs(out.astype(np.longdouble) - ex)
    assert (err <= tol).all(), f"worst {float((err / np.maximum(tol, 1e-300)).max())} of the exact bar"
    same = (np.asarray(X, np.float64)[:, None, :] == np.asarray(C, np.float64)[None]).all(-1)
    assert (out[same] == 0).all()


def sklearn_bar(X, C, sk):
    """the per-element bar of the library against sklearn's transform of the same X and centres"""
    d = np.asarray(X).shape[1]
    x2 = (np.asarray(X, np.float64) ** 2).sum(1)
    c2 = (np.asarray(C, np.float64) ** 2).sum(1)
    return np.sqrt((d + 2) * 2.0 ** -52 * (x2[:, None] + c2[None])) + 2 * np.spacing(np.abs(sk)).astype(np.float64)


def check_sklearn(out, X, C, sk, extra=0.0):
    """``extra``: added to the bar per centre (the distance between the library's and sklearn's fitted centres)"""
    out = np.asarray(out)
    assert out.dtype == sk.dtype and out.shape == sk.shape
    bar = sklearn_bar(X, C, sk) + extra
    err = np.abs(out.astype(np.float64) - sk.astype(np.float64))
    assert (err <= bar).all(), f"worst {float((err / bar).max())} of the sklearn bar"
