import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def unpack_images(z):
    """inverse of tests/golden/make_golden.py:pack_images"""
    out, o = [], 0
    for s in z["shapes"]:
        n = int(np.prod(s))
        out.append(z["flat"][o:o + n].reshape(s))
        o += n
    return out


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


def run_without_gpu(code):
    """Run ``code`` in a child Python started in the repository root that sees no CUDA device (``CUDA_VISIBLE_DEVICES``
    empty), so that the no-GPU behaviour is checked on machines with a GPU too; returns the child's stdout."""
    import subprocess
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return r.stdout


def have_cv2():
    try:
        import cv2  # noqa: F401
        return True
    except Exception:
        return False


def flow_parity_stats(flow, ref, RA=None, RB=None, winsize=15):
    """BASELINE.md section 5: distribution of the end-point error against cv2 -- mean / p99 / p99.9 / max, and the max
    over the well-conditioned pixels.  Well-conditioned = det of the box-blurred 2x2 system matrix > 1e-2, with the
    matrix formed from the polynomial coefficients of the first frame (``RA[..., 2:4]``, ``RB``: the r4, r5, r6 of
    SURVEY.md A.2 at zero displacement; the blur is the iteration's winsize x winsize box mean)."""
    e = np.linalg.norm(np.asarray(flow, np.float64) - np.asarray(ref, np.float64), axis=-1)
    out = {"mean": float(e.mean()), "p99": float(np.percentile(e, 99)), "p99.9": float(np.percentile(e, 99.9)),
           "max": float(e.max())}
    if RA is not None and RB is not None:
        r4, r5, r6 = RA[..., 2].astype(np.float64), RA[..., 3].astype(np.float64), 0.5 * RB.astype(np.float64)

        def box(a):
            r = winsize // 2
            p = np.pad(a, r, mode="edge")
            c = np.cumsum(np.cumsum(p, 0), 1)
            c = np.pad(c, ((1, 0), (1, 0)))
            k = 2 * r + 1
            return (c[k:, k:] - c[:-k, k:] - c[k:, :-k] + c[:-k, :-k]) / (winsize * winsize)
        g11, g12, g22 = box(r4 * r4 + r6 * r6), box((r4 + r5) * r6), box(r5 * r5 + r6 * r6)
        mask = (g11 * g22 - g12 * g12) > 1e-2
        out["well_conditioned_share"] = float(mask.mean())
        out["max_well_conditioned"] = float(e[mask].max()) if mask.any() else 0.0
    return out
