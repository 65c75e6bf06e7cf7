"""Empty clusters and weights on the B200, through every path kmeans.lloyd picks by shape: the relocation goldens of
make_relocation_golden.py (scikit-learn 1.9.0), and its generated cases scaled up -- uint8 d = 4 (fused step; weighted:
two kernels) up to 1 M rows, the small / medium / generic E-steps in float32 and float64, the tensor cores -- against the
oracle (itself pinned to sklearn on the goldens); shared-row batches, per-problem [B, n] weights, lloyd_cells on a
350-cell frame with probe cells planted in it, and KMeans.fit end to end.  Then non-unit weights on the same paths without
empty clusters.  The CPU twins are in tests/test_emulated_kmeans_relocation.py."""
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN

pytestmark = pytest.mark.gpu

from opticalflowclustering_b200 import kmeans as km    # noqa: E402
from oracle import kmeans_np as K                       # noqa: E402

sys.path.insert(0, GOLDEN)
import make_relocation_golden as RG                      # noqa: E402


@pytest.fixture(scope="module")
def Z():
    return np.load(os.path.join(GOLDEN, "kmeans_sklearn_relocation.npz"))


def _case(key):
    if key.startswith("probe_"):
        p, f = key[len("probe_"):].rsplit("_", 1)
        return RG.probe_form(p, f)
    return RG.gen_case(key[len("gen_"):])


def _fit(X, init, w=None, max_iter=300):
    wt = None if w is None else torch.from_numpy(w).cuda()
    return km.lloyd(torch.from_numpy(X).cuda(), init, max_iter=max_iter, sample_weight=wt)


@pytest.mark.parametrize("key", [f"probe_{p}_{f}" for p, f in RG.PROBE_FORMS] + [f"gen_{g}" for g in RG.GEN_CASES])
def test_gpu_relocation_goldens(Z, key):
    X, init, w = _case(key)
    for m in RG.MAX_ITERS:
        RG.check_fit(f"gpu {key} max_iter={m}", _fit(X, init, w, m), RG.golden_fit(Z, key, m), X)


# (n, d, dtype, k, weighted, below, runs on the tensor cores): every E-step / M-step form of kmeans.lloyd
PATHS = {
    "u8_d4_fused_1M": (1_000_000, 4, np.uint8, 8, False, True, False),
    "u8_d4_weighted_1M": (1_000_000, 4, np.uint8, 8, True, False, False),
    "f32_d42_medium": (20000, 42, np.float32, 6, False, True, False),
    "f64_d42_medium_w": (20000, 42, np.float64, 6, True, False, False),
    "f32_d130_medium_w": (20000, 130, np.float32, 5, True, True, False),
    "f64_d390_medium": (12000, 390, np.float64, 4, False, False, False),
    "f32_d602_generic": (8000, 602, np.float32, 4, False, True, False),
    "f64_d602_generic_w": (8000, 602, np.float64, 4, True, True, False),
    "f32_d64_tc": (30000, 64, np.float32, 8, False, True, True),
    "f32_d64_tc_w": (30000, 64, np.float32, 8, True, False, True),
    "f32_d128_tc_w": (30000, 128, np.float32, 5, True, True, True),
    "u8_d128_k32_tc": (30000, 128, np.uint8, 32, False, True, True),
    "u8_d128_k32_tc_w": (30000, 128, np.uint8, 32, True, False, True),
}


@pytest.mark.parametrize("name", list(PATHS))
def test_gpu_relocation_paths_against_oracle(name):
    n, d, dt, k, weighted, below, tc = PATHS[name]
    X, init, w = RG.relocation_case(n, d, dt, k, weighted, below, seed=1)
    assert km._tc_wanted(torch.empty((1, 1, d), dtype=torch.from_numpy(X[:1]).dtype, device="cuda"), k) == tc
    for m in (1, 300):
        RG.check_fit(f"gpu {name} max_iter={m}", _fit(X, init, w, m), K.kmeans_fit(X, init, max_iter=m, sample_weight=w), X)


@pytest.mark.parametrize("dt", [np.uint8, np.float64])
def test_gpu_shared_row_batch(dt):
    """X [n, d] with init [R, k, d]: starts that hit the relocation (both layouts) beside one that does not"""
    X, init, _ = RG.relocation_case(40000, 4 if dt == np.uint8 else 42, dt, 8, below=False, seed=2)
    init_b = init.copy()
    init_b[[1, 7]] = init[[7, 1]]                         # the outlier's cluster below the blobs
    rng = np.random.default_rng(3)
    other = X[rng.choice(X.shape[0], 8, replace=False)].astype(np.float64)
    inits = np.stack([init, other, init_b])
    got = km.lloyd(torch.from_numpy(X).cuda(), inits)
    for r in range(3):
        RG.check_fit(f"shared batch {dt.__name__} start {r}", [t[r] for t in got], K.kmeans_fit(X, inits[r]), X)


@pytest.mark.parametrize("dt", [np.uint8, np.float32, np.float64])
def test_gpu_per_problem_weights(dt):
    """[B, n] weights that differ per problem: only problems 0 and 2 hit the relocation (2 with its far row at weight 0)"""
    X, init, w = RG.relocation_case(20000, 4 if dt == np.uint8 else 42, dt, 6, weighted=True, seed=3)
    rng = np.random.default_rng(4)
    quiet = init.copy()
    quiet[0] = init[1]
    quiet[0, 0] += 5.0                                   # beside a blob: no empty cluster
    quiet[-1] = X[np.argmin(np.abs(X[:, 0].astype(np.float64) - 3.0) + np.abs(X[:, 1].astype(np.float64) - 3.0))]
    w2 = w.copy()
    far = int(np.argmin(np.abs(X[:, 0].astype(np.float64) - 3.0) + np.abs(X[:, 1].astype(np.float64) - 3.0)))
    w2[far] = 0
    ws = np.stack([w, rng.integers(1, 5, X.shape[0]).astype(w.dtype), w2])
    inits = np.stack([init, quiet, init])
    got = km.lloyd(torch.from_numpy(np.stack([X] * 3)).cuda(), inits, sample_weight=torch.from_numpy(ws).cuda())
    for b in range(3):
        RG.check_fit(f"per-problem weights {dt.__name__} problem {b}", [t[b] for t in got],
                     K.kmeans_fit(X, inits[b], sample_weight=ws[b]), X)


@pytest.mark.parametrize("fast", ["1", "0"])
@pytest.mark.parametrize("k", [3, 8, 16])
def test_gpu_cells_frame_with_planted_probes(monkeypatch, fast, k):
    """lloyd_cells on a 350-cell frame of 1500-pixel cells (random blob data, init from the cell's own rows), with the
    generated relocation case planted in a few cells (both layouts): every cell against the oracle"""
    monkeypatch.setenv("OFC_CELLS_FAST", fast)
    cells, n = 350, 1500
    rng = np.random.default_rng(10 + k)
    X = np.empty((cells, n, 4), np.uint8)
    inits = np.empty((cells, k, 4))
    for c in range(cells):
        cen = rng.uniform(20, 235, (k + 2, 4))
        X[c] = np.clip(np.rint(cen[rng.integers(k + 2, size=n)] + rng.normal(0, 12, (n, 4))), 0, 255)
        X[c, :, 3] = 255
        inits[c] = X[c, rng.choice(n, k, replace=False)]
    planted = {7: False, 180: True, 349: False}
    for c, below in planted.items():
        Xc, ic, _ = RG.relocation_case(n, 4, np.uint8, k, below=below, seed=c)
        X[c], inits[c] = Xc, ic
    lab, cen, inertia, n_iter, _ = km.lloyd_cells(torch.from_numpy(X).cuda(), k, init=torch.from_numpy(inits).cuda())
    lab, cen, inertia, n_iter = lab.cpu().numpy(), cen.cpu().numpy(), inertia.cpu().numpy(), n_iter.cpu().numpy()
    bad = []
    for c in range(cells):
        ref = K.kmeans_fit(X[c], inits[c])
        ok = ((lab[c] == ref[0]).all() and int(n_iter[c]) == ref[3]
              and (np.abs(cen[c] - ref[1]) <= 1e-9 + 1e-12 * np.abs(ref[1])).all()
              and abs(inertia[c] - ref[2]) <= 1e-9 * ref[2])
        if not ok:
            bad.append(c)
    print(f"cells k={k} fast={fast}: {len(bad)} of {cells} cells differ from the oracle: {bad[:10]}")
    assert not bad


def test_gpu_kmeans_fit_end_to_end(Z):
    """KMeans(init, n_init=1).fit(X, sample_weight=w) on the zero-weight probe: the public estimator, one iteration"""
    X, init, w = RG.probe_form("zero_weight_move", "f64")
    for m in RG.MAX_ITERS:
        est = km.KMeans(n_clusters=3, init=init, n_init=1, max_iter=m).fit(X, sample_weight=w)
        RG.check_fit(f"KMeans.fit max_iter={m}", (est.labels_, est.cluster_centers_, est.inertia_, est.n_iter_),
                     RG.golden_fit(Z, "probe_zero_weight_move_f64", m), X)


# ---- non-unit weights on the same paths, without empty clusters ----------------------------------------------------
def _blobs(n, d, dt, k, seed):
    """k tight, well-separated blobs; init = each blob's centre moved by a few units (no cluster empties)"""
    rng = np.random.default_rng(seed)
    side = int(np.ceil(np.sqrt(k)))
    grid = np.linspace(40, 215, max(side, 2))
    bc = np.full((k, d), 100.0)
    bc[:, :2] = [[grid[i % side], grid[i // side]] for i in range(k)]
    bc[:, 2:] = rng.uniform(60, 190, (k, d - 2))
    X = bc[rng.integers(k, size=n)] + rng.normal(0, 4.0, (n, d))
    X = np.clip(np.rint(X), 0, 255).astype(np.uint8) if dt == np.uint8 else X.astype(dt)
    return X, bc + rng.uniform(-6, 6, bc.shape)


@pytest.mark.parametrize("wkind", ["real", "int"])
@pytest.mark.parametrize("shape", [(500_000, 4, np.uint8, 8), (20000, 42, np.float64, 6), (20000, 130, np.float32, 5),
                                   (8000, 602, np.float64, 4), (30000, 64, np.float32, 8), (30000, 128, np.uint8, 32)],
                         ids=["u8_d4", "f64_d42", "f32_d130", "f64_d602", "f32_d64_tc", "u8_d128_tc"])
def test_gpu_weighted_paths_against_oracle(shape, wkind):
    n, d, dt, k = shape
    X, init = _blobs(n, d, dt, k, seed=d + k)
    rng = np.random.default_rng(d)
    wdt = np.float32 if dt == np.float32 else np.float64
    w = (rng.uniform(0.05, 4.0, n) if wkind == "real" else rng.integers(1, 7, n)).astype(wdt)
    ref = K.kmeans_fit(X, init, sample_weight=w)
    assert (np.bincount(ref[0], minlength=k) > 0).all()
    RG.check_fit(f"weighted {dt.__name__} d={d} {wkind}", _fit(X, init, w), ref, X)
