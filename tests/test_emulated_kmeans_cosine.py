"""k-means / cosine kernels + their Python host loop on CPU: the .cu sources under the fiber
emulation (tests/emu), driven through the product's own host code (kmeans.py / cosine.py
with the emulated library passed explicitly), compared with the oracle and with the
sklearn / reference goldens.  The `-m gpu` twins are in tests/test_gpu_kmeans_cosine.py."""
import csv
import os

import numpy as np
import pytest
import torch

from oracle import grid_np as G
from oracle import kmeans_np as K
from tests.conftest import GOLDEN

E = pytest.importorskip("tests.emu.emu_lib")
from opticalflowclustering_b200 import cosine as cosm  # noqa: E402
from opticalflowclustering_b200 import kmeans as km    # noqa: E402


@pytest.fixture(scope="module")
def L():
    """the .cu sources compiled for the host; kmeans.py / cosine.py are routed to it through their private test hook"""
    E.build()
    km._use_test_library(E.lib())
    yield E.lib()
    km._use_test_library(None)


def _hue_col(path):
    with open(path, encoding="utf-8-sig") as f:
        return np.array([int(r[1]) for r in csv.reader(f) if r])


@pytest.mark.parametrize("name", ["u8_d4_k3", "u8_d4_k8"])
def test_lloyd_vs_sklearn_golden_u8(L, name):
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn.npz"))
    X = z[name + "_X"][:6000] if name == "u8_d4_k8" else z[name + "_X"]
    init = z[name + "_init"]
    labels, centres, inertia, n_iter = km.lloyd(X, init)
    want = K.kmeans_fit(X, init)
    assert (labels.numpy() == want[0]).all()
    assert np.abs(centres.numpy() - want[1]).max() < 1e-9
    assert abs(float(inertia) - want[2]) <= 1e-9 * want[2]
    assert int(n_iter) == want[3]
    if X.shape[0] == z[name + "_X"].shape[0]:
        assert (labels.numpy() == z[name + "_labels"]).all()
        assert int(n_iter) == int(z[name + "_niter"])
        assert abs(float(inertia) - float(z[name + "_inertia"])) <= 1e-5 * float(z[name + "_inertia"])
        assert (km.predict(X, centres).numpy() == z[name + "_predict"]).all()


def test_lloyd_f32_golden(L):
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn.npz"))
    X, init = z["f32_d32_k16_X"][:1500], z["f32_d32_k16_init"]
    labels, centres, inertia, n_iter = km.lloyd(X, init)
    want = K.kmeans_fit(X, init)
    assert (labels.numpy() == want[0]).mean() > 0.999
    assert np.abs(centres.numpy() - want[1]).max() < 1e-3
    assert abs(float(inertia) - want[2]) <= 1e-5 * want[2]


def test_lloyd_batched_matches_single_and_freezes(L):
    rng = np.random.default_rng(3)
    B, n, d, k = 5, 700, 4, 3
    cen = rng.uniform(10, 240, (B, k, d))
    X = np.clip(np.rint(cen[np.arange(B)[:, None], rng.integers(k, size=(B, n))] + rng.normal(0, 9, (B, n, d))), 0, 255)
    X = X.astype(np.uint8)
    init = X[:, :k].astype(np.float64)
    labels, centres, inertia, n_iter = km.lloyd(X, init)
    assert len(set(n_iter.tolist())) > 1 or B == 1     # problems stop at different iterations
    for b in range(B):
        w = K.kmeans_fit(X[b], init[b])
        assert (labels[b].numpy() == w[0]).all()
        assert np.abs(centres[b].numpy() - w[1]).max() < 1e-9
        assert int(n_iter[b]) == w[3]
        assert abs(float(inertia[b]) - w[2]) <= 1e-9 * max(w[2], 1.0)


def test_generic_path_large_d(L):
    rng = np.random.default_rng(5)
    n, d, k = 300, 70, 5
    cen = rng.uniform(0, 255, (k, d))
    X = np.clip(np.rint(cen[rng.integers(k, size=n)] + rng.normal(0, 20, (n, d))), 0, 255).astype(np.uint8)
    init = X[:k].astype(np.float64)
    labels, centres, inertia, n_iter = km.lloyd(X, init)
    w = K.kmeans_fit(X, init)
    assert (labels.numpy() == w[0]).all() and int(n_iter) == w[3]
    assert np.abs(centres.numpy() - w[1]).max() < 1e-9


def test_empty_cluster_relocation(L):
    # a duplicated initial centre: its second copy starts empty (ties -> lowest index) and is relocated
    rng = np.random.default_rng(11)
    X = np.clip(np.rint(rng.normal(100, 20, (400, 4))), 0, 255).astype(np.uint8)
    init = np.array([[100, 100, 100, 100], [100, 100, 100, 100], [70, 70, 70, 70]], np.float64)
    labels, centres, inertia, n_iter = km.lloyd(X, init)
    w = K.kmeans_fit(X, init)
    assert int(n_iter) == w[3]
    assert (labels.numpy() == w[0]).all()
    assert abs(float(inertia) - w[2]) <= 1e-9 * w[2]


def test_lloyd_cells_device_loop_equals_stepwise(L):
    """one-launch per-cell kernel == the stepwise host loop == the oracle, for the same initial centres"""
    rng = np.random.default_rng(31)
    B, n, d, k = 6, 900, 4, 4
    cen = rng.uniform(10, 240, (B, k, d))
    X = np.clip(np.rint(cen[np.arange(B)[:, None], rng.integers(k, size=(B, n))] + rng.normal(0, 10, (B, n, d))), 0, 255).astype(np.uint8)
    init = X[:, :k].astype(np.float64)
    init[2, 1] = init[2, 0]                                  # duplicated centre -> an empty cluster gets relocated
    lab, cen_d, inertia, n_iter, counts = km.lloyd_cells(X, k, init=init)
    l2, c2, i2, n2 = km.lloyd(X, init)
    assert torch.equal(lab, l2) and torch.equal(cen_d, c2) and (n_iter.long() == n2).all()
    assert ((inertia - i2).abs() <= 1e-12 * i2).all()
    for b in range(B):
        w = K.kmeans_fit(X[b], init[b])
        assert (lab[b].numpy() == w[0]).all() and int(n_iter[b]) == w[3]
        assert (counts[b].numpy() == np.bincount(w[0], minlength=k)).all()


def test_lloyd_cells_kmeanspp_seeding(L):
    rng = np.random.default_rng(32)
    X = np.clip(np.rint(np.concatenate([rng.normal(50, 5, (300, 4)), rng.normal(130, 5, (300, 4)), rng.normal(210, 5, (300, 4))])), 0, 255)
    X = np.stack([X.astype(np.uint8), X[::-1].astype(np.uint8)])
    a = km.lloyd_cells(X, 3, seed=7)
    b = km.lloyd_cells(X, 3, seed=7)
    assert all(torch.equal(u, v) for u, v in zip(a, b))                      # deterministic in the seed
    lab, cen_d, inertia, n_iter, counts = a
    assert sorted(counts[0].tolist()) == [300, 300, 300] and sorted(counts[1].tolist()) == [300, 300, 300]
    assert np.allclose(np.sort(cen_d[0].numpy()[:, 0]), [50, 130, 210], atol=1.5)
    with pytest.raises(Exception):
        km.lloyd_cells(X[:, :2], 3)                         # n < k


def test_k1_is_the_mean_and_matches_g2_rint(L):
    z = np.load(os.path.join(GOLDEN, "g23_cells.npz"))
    cells = z["cells"][0, :40]                              # 40 cells of one frame, 51x51x3
    X = np.stack([G.preprocess_image(c[..., ::-1].copy()).reshape(-1, 4) for c in cells])
    labels, centres, inertia, n_iter = km.lloyd(X, X[:, :1].astype(np.float64))
    assert (labels.numpy() == 0).all() and (n_iter.numpy() <= 2).all()
    for b in range(len(cells)):
        c, _ = G.cluster_colors_k1(X[b].reshape(51, 51, 4))
        assert (np.rint(centres[b, 0].numpy()) == c).all()


def test_kmeans_class_api(L):
    rng = np.random.default_rng(2)
    X = np.clip(np.rint(np.concatenate([rng.normal(60, 6, (300, 4)), rng.normal(190, 6, (200, 4))])), 0, 255).astype(np.uint8)
    clt = km.KMeans(n_clusters=2, random_state=0).fit(X)
    pred = clt.predict(X)
    assert (pred == clt.labels_).all()
    counts = np.bincount(pred)
    assert sorted(counts.tolist()) == [200, 300]
    assert clt.cluster_centers_.shape == (2, 4) and clt.inertia_ > 0 and clt.n_iter_ >= 1
    with pytest.raises(ValueError):
        km.KMeans(n_clusters=5).fit(X[:3])


@pytest.mark.parametrize("name", ["blobs_k5_rs0", "blobs_k5_rs42", "cell_k8_rs3"])
def test_kmeans_random_state_reproduces_sklearn(L, name):
    """SURVEY section 8f-3: KMeans(n_clusters=k, random_state=int) end to end -- k-means++ with sklearn's RNG call
    sequence (same seed indices), then Lloyd: labels, n_iter bit-exact, centres / inertia to rounding"""
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_seeded.npz"))
    X = z[name + "_X"]
    k, rs = (int(v) for v in z[name + "_k_rs"])
    _, idx = km.kmeans_plusplus(X, k, random_state=rs)
    assert (idx == z[name + "_seed_idx"]).all()
    clt = km.KMeans(n_clusters=k, random_state=rs).fit(X)
    assert (clt.labels_ == z[name + "_labels"]).all() and clt.n_iter_ == int(z[name + "_niter"])
    assert np.abs(clt.cluster_centers_ - z[name + "_centers"]).max() < 1e-9
    assert abs(clt.inertia_ - float(z[name + "_inertia"])) <= 1e-9 * float(z[name + "_inertia"])


@pytest.mark.parametrize("shape", [(5000, 4, 8, 1), (3001, 7, 5, 3), (1500, 32, 4, 1)])
def test_fused_uint8_step_equals_two_kernel_iteration(L, shape, monkeypatch):
    """ofc_kmeans_step (E-step + exact integer sums in one pass) against ofc_kmeans_assign + ofc_kmeans_sums"""
    n, d, k, B = shape
    X = np.random.default_rng(1).integers(0, 256, (B, n, d), dtype=np.uint8)
    init = X[:, :k].astype(np.float64)
    monkeypatch.setenv("OFC_KMEANS_FUSED", "0")
    a = km.lloyd(X, init)
    monkeypatch.setenv("OFC_KMEANS_FUSED", "1")
    b = km.lloyd(X, init)
    assert all(torch.equal(x, y) for x, y in zip(a, b))


def test_medium_assign_kernel_equals_generic(L, monkeypatch):
    """kmeans_assign_medium_kernel (centres in shared memory, row in registers) keeps the generic kernel's arithmetic
    order: whole fits must be bit-identical"""
    rng = np.random.default_rng(2)
    for dt, (n, d, k, B) in [(np.uint8, (260, 350, 8, 1)), (np.float32, (300, 70, 9, 2)), (np.float64, (200, 130, 5, 1)),
                             (np.uint8, (200, 33, 12, 1))]:
        X = (rng.integers(0, 256, (B, n, d)) if dt == np.uint8 else rng.normal(0, 3, (B, n, d))).astype(dt)
        init = X[:, :k].astype(np.float64)
        monkeypatch.setenv("OFC_KMEANS_MEDIUM", "0")
        a = km.lloyd(X, init, max_iter=4)
        monkeypatch.setenv("OFC_KMEANS_MEDIUM", "1")
        b = km.lloyd(X, init, max_iter=4)
        assert all(torch.equal(x, y) for x, y in zip(a, b)), (dt, n, d, k, B)


def test_sliding_cosine_goldens(L):
    short = _hue_col(os.path.join(GOLDEN, "bounce.csv"))
    for name, want_sim, want_frame in [("601_3_3_cropped.csv", 0.91448231723348, 24),
                                       ("cropped_trimmed2.csv", 0.963475622684391, 7)]:
        long_ = _hue_col(os.path.join(GOLDEN, name))
        best, frame, sims = cosm.sliding_cosine(short, long_, return_sims=True)
        ob, of = G.sliding_cosine(short, long_)
        assert best == ob and frame == of                    # bit-exact vs the numpy restatement
        assert frame == want_frame and abs(best - want_sim) < 1e-14
        ref = np.array([G.cosine_similarity(short, long_[i:i + len(short)]) for i in range(len(sims))])
        assert (sims == ref).all()


def test_sliding_cosine_edge_cases(L):
    assert cosm.sliding_cosine([1, 2, 3], [1, 2]) == (-1, -1)
    best, frame = cosm.sliding_cosine([0, 0], [0, 0, 5, 0])
    assert best == 0 and frame == 2                            # zero norms -> 0; ties -> last index
    best, frame = cosm.sliding_cosine([1, 1], [2, 2, 0, 3, 3])
    assert frame == 3 and abs(best - 1.0) < 1e-15
    assert cosm.calculate_cosine_similarity([0, 0], [1, 2]) == 0


def test_vector_distance_golden(L):
    a = _hue_col(os.path.join(GOLDEN, "file1.csv"))
    b = _hue_col(os.path.join(GOLDEN, "file2.csv"))
    cos, row, dist = cosm.vector_distance(a, b)
    ocos, orow, odist = G.vector_distance(a, b)
    assert abs(cos[0, 0] - ocos[0, 0]) < 1e-15 and str(np.array([[round(cos[0, 0], 12)]])) == "[[1.]]"
    assert np.array_equal(row, orow, equal_nan=True)
    assert dist == odist == 0.0
    assert np.allclose(row[:6], [1., 1.09756098, 0.91836735, 0.83333333, 0.8490566, 0.52023121])


def test_row_cosine(L):
    rng = np.random.default_rng(9)
    for d, dt in [(3, np.uint8), (16, np.uint8), (350, np.uint8), (40, np.float32)]:
        X = rng.integers(0, 180, (257, d)).astype(dt)
        X[5] = 0
        q = rng.integers(0, 180, d).astype(np.float64)
        out = cosm.row_cosine(X, q).numpy()
        ref = np.array([G.cosine_similarity(X[i].astype(np.float64), q) for i in range(len(X))], dtype=np.float64)
        assert out[5] == 0
        assert np.abs(out - ref).max() < 1e-14


def test_extract_cells_matches_reference_rois(L):
    import ctypes as C
    rng = np.random.default_rng(4)
    H, W, rows, cols = 60, 100, 3, 4
    frame = rng.integers(0, 256, (2, H, W, 3), dtype=np.uint8)
    ys, xs = H // rows, W // cols
    out = np.zeros((2, rows * cols, ys * xs, 4), np.uint8)
    rc = L.ofc_grid_extract_cells(C.c_void_p(frame.ctypes.data), 2, H, W, rows, cols, 1, 30, 0,
                                  C.c_void_p(out.ctypes.data), C.c_void_p(0))
    assert rc == 0
    for f in range(2):
        fr = frame[f].copy()
        _, _, rois = G.grid_mean_hues(fr, rows, cols)        # draws the rectangles like the reference
        for c, roi in enumerate(rois):
            want = G.preprocess_image(roi.copy()).reshape(-1, 4)
            assert (out[f, c] == want).all()


def _cells_both(L, X, k, monkeypatch, **kw):
    """the same problems through the shared-memory / filtered kernel (cells_kmeans.cu) and the first kernel"""
    monkeypatch.setenv("OFC_CELLS_FAST", "1")
    fast = km.lloyd_cells(X, k, **kw)
    monkeypatch.setenv("OFC_CELLS_FAST", "0")
    slow = km.lloyd_cells(X, k, **kw)
    monkeypatch.delenv("OFC_CELLS_FAST")
    return fast, slow


@pytest.mark.parametrize("k", [1, 3, 8, 13])
def test_cells_fast_kernel_is_bit_identical_to_the_first_kernel(L, k, monkeypatch):
    """labels, centres, inertia, n_iter, counts: identical bits, with given centres and with k-means++ seeding"""
    rng = np.random.default_rng(40 + k)
    B, n = 4, 700
    cen = rng.uniform(10, 240, (B, max(k, 2), 4))
    X = np.clip(np.rint(cen[np.arange(B)[:, None], rng.integers(max(k, 2), size=(B, n))] + rng.normal(0, 14, (B, n, 4))), 0, 255).astype(np.uint8)
    X[3] = rng.integers(0, 256, (n, 4), dtype=np.uint8)            # one unclustered problem: many iterations, near-ties
    init = X[:, :k].astype(np.float64)
    for kw in ({"init": init}, {"seed": 5}):
        fast, slow = _cells_both(L, X, k, monkeypatch, **kw)
        for u, v in zip(fast, slow):
            assert torch.equal(u, v)
    lab, cen_d, inertia, n_iter, counts = fast
    assert int(n_iter.max()) > 1 or k == 1


def test_cells_fast_kernel_degenerate_cells(L, monkeypatch):
    """fewer distinct colours than clusters (a black cell with its white grid lines): relocation of empty clusters,
    exact ties between duplicated centres -- still the first kernel's bits, and the oracle's labels for a given init"""
    n = 26 * 25
    X = np.zeros((3, n, 4), np.uint8)
    X[0, :60] = 255                                                 # two colours
    X[1, :] = (40, 90, 200, 255)                                    # one colour
    X[2, ::3] = (255, 0, 0, 255); X[2, 1::3] = (0, 255, 0, 255)     # three colours, integer-symmetric (exact ties)
    for k in (2, 8):
        for kw in ({"seed": 1}, {"init": X[:, :k].astype(np.float64)}):
            fast, slow = _cells_both(L, X, k, monkeypatch, **kw)
            for u, v in zip(fast, slow):
                assert torch.equal(u, v)
    init = X[:, :2].astype(np.float64)
    lab = km.lloyd_cells(X, 2, init=init)[0]
    for b in range(3):
        assert (lab[b].numpy() == K.kmeans_fit(X[b], init[b])[0]).all()


def test_grid_kmeans_cells_fused_equals_gather_then_cluster(L):
    """ofc_grid_kmeans_cells (cells gathered inside the k-means kernel) == ofc_grid_extract_cells + ofc_kmeans_cells
    + the host-side dominant-cluster rule, and first_frame shifts the random stream as documented"""
    import ctypes as C
    rng = np.random.default_rng(50)
    F, H, W, rows, cols, k = 2, 50, 66, 3, 4, 3
    base = rng.integers(0, 256, (F, rows, cols, 1, 1, 3))
    img = np.clip(np.repeat(np.repeat(base, H // rows, 3), W // cols, 4).transpose(0, 1, 3, 2, 4, 5).reshape(F, rows * (H // rows), cols * (W // cols), 3)
                  + rng.normal(0, 25, (F, rows * (H // rows), cols * (W // cols), 3)), 0, 255).astype(np.uint8)
    frames = np.zeros((F, H, W, 3), np.uint8)
    frames[:, :img.shape[1], :img.shape[2]] = img
    cells, n = rows * cols, (H // rows) * (W // cols)
    p = lambda a: C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)

    def fused(first_frame, fr):
        nf = fr.shape[0]
        dc, dh = np.zeros((nf, cells, 4), np.uint8), np.zeros((nf, cells), np.uint8)
        cen, cnt, nit = np.zeros((nf, cells, k, 4)), np.zeros((nf, cells, k), np.int64), np.zeros((nf, cells), np.int32)
        L.ofc_grid_kmeans_cells_workspace_bytes.restype = C.c_size_t
        ws = np.zeros(max(8, L.ofc_grid_kmeans_cells_workspace_bytes(nf, H, W, rows, cols, k)), np.uint8)
        rc = L.ofc_grid_kmeans_cells(p(fr), nf, H, W, rows, cols, 1, 30, 0, k, C.c_uint64(9), C.c_uint64(first_frame), 300,
                                     C.c_double(1e-4), p(dc), p(dh), p(cen), p(cnt), p(nit), p(ws), C.c_size_t(ws.size), None)
        assert rc == 0, L.ofc_last_error()
        return dc, dh, cen, cnt, nit

    dc, dh, cen, cnt, nit = fused(0, frames)
    out = np.zeros((F, cells, n, 4), np.uint8)
    assert L.ofc_grid_extract_cells(p(frames), F, H, W, rows, cols, 1, 30, 0, p(out), None) == 0
    lab, c2, inertia, n2, counts = km.lloyd_cells(out.reshape(F * cells, n, 4), k, seed=9)
    assert (cen.reshape(-1, k, 4) == c2.numpy()).all() and (cnt.reshape(-1, k) == counts.numpy()).all()
    assert (nit.reshape(-1) == n2.numpy()).all()
    top = counts.numpy().argmax(1)                                              # first largest
    want = np.rint(c2.numpy()[np.arange(F * cells), top])
    assert (dc.reshape(-1, 4) == want.astype(np.uint8)).all()
    from oracle import viz_np
    hues = np.array([viz_np.bgr2hsv_u8(want[i, :3].astype(np.uint8).reshape(1, 1, 3))[0, 0, 0] for i in range(F * cells)])
    assert (dh.reshape(-1) == hues).all()
    # frame 1 processed alone with first_frame = 1 reproduces its row of the two-frame call
    dc1, dh1, cen1, cnt1, nit1 = fused(1, frames[1:])
    assert (dc1[0] == dc[1]).all() and (dh1[0] == dh[1]).all() and (cen1[0] == cen[1]).all()


def test_cells_seeding_and_dominant_hue_vs_numpy_oracle(L):
    """the device-resident seeding (counter-based stream), the fit and the dominant-cluster hue against the
    independent numpy restatement (oracle/kmeans_np.py: cells_seed_indices / cells_fit / dominant_centre_hue)"""
    rng = np.random.default_rng(61)
    B, n, k = 5, 640, 4
    cen = rng.uniform(10, 240, (B, k, 4))
    X = np.clip(np.rint(cen[np.arange(B)[:, None], rng.integers(k, size=(B, n))] + rng.normal(0, 9, (B, n, 4))), 0, 255).astype(np.uint8)
    lab, cen_d, inertia, n_iter, counts = km.lloyd_cells(X, k, seed=123)
    for b in range(B):
        wl, wc, wi, wn, idx = K.cells_fit(X[b], k, 123, b)
        assert (lab[b].numpy() == wl).all() and int(n_iter[b]) == wn
        assert np.abs(cen_d[b].numpy() - wc).max() <= 1e-9 and abs(float(inertia[b]) - wi) <= 1e-9 * wi


@pytest.mark.parametrize("name", ["u8_d2_k8", "f32_d2_k8"])
def test_lloyd_d2_lattice_vs_sklearn_golden(L, name):
    """D = 2 end of BASELINE configs[4]'s sweep: uint8 rows on a 2-D lattice sit EXACTLY on bisectors, so the last bit of
    ||c||^2 decides labels -- it is evaluated in numpy's einsum order (what sklearn's row_norms does); a sequential fma
    chain flips 31 of these 20 000 labels"""
    import sys
    sys.path.insert(0, GOLDEN)
    import make_golden as MG
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_sweep.npz"))
    X, init = MG.sweep_case(name)
    labels, centres, inertia, n_iter = km.lloyd(X, init)
    assert int((labels.numpy() != z[name + "_labels"]).sum()) == 0 and int(n_iter) == int(z[name + "_niter"])
    assert abs(float(inertia) - float(z[name + "_inertia"])) <= 1e-5 * float(z[name + "_inertia"])


def test_grid_kmeans_cells_on_flow_visualisation_vs_oracle(L):
    """the k > 1 pipeline stage on REAL visualisation data (oracle flow -> HSV image of a small synthetic clip: heavily
    duplicated colours, rows exactly on bisectors): every cell's KMeans(8) fit -- seeding, n_iter, centres -- equals the
    numpy oracle (oracle/kmeans_np.py cells_fit)"""
    import ctypes as C
    from oracle import farneback_np as FB, viz_np as V
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, rows, cols, k = 144, 200, 6, 8, 8
    clip = synthetic_clip(3, H, W, seed=13).numpy()
    g = np.stack([V.bgr2gray(f) for f in clip])
    viz = np.ascontiguousarray(np.stack([V.flow_to_bgr(FB.calc_optical_flow_farneback(g[p], g[p + 1]))[0] for p in range(2)]))
    cells = rows * cols
    p_ = lambda a: C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)
    dc, dh = np.zeros((2, cells, 4), np.uint8), np.zeros((2, cells), np.uint8)
    cen, cnt, nit = np.zeros((2, cells, k, 4)), np.zeros((2, cells, k), np.int64), np.zeros((2, cells), np.int32)
    L.ofc_grid_kmeans_cells_workspace_bytes.restype = C.c_size_t
    ws = np.zeros(max(8, L.ofc_grid_kmeans_cells_workspace_bytes(2, H, W, rows, cols, k)), np.uint8)
    rc = L.ofc_grid_kmeans_cells(p_(viz), 2, H, W, rows, cols, 1, 30, 0, k, C.c_uint64(3), C.c_uint64(0), 300, C.c_double(1e-4),
                                 p_(dc), p_(dh), p_(cen), p_(cnt), p_(nit), p_(ws), C.c_size_t(ws.size), None)
    assert rc == 0
    for p in range(2):
        fr = viz[p].copy()
        _, _, rois = G.grid_mean_hues(fr, rows, cols)
        for c in range(0, cells, 2):
            X = G.preprocess_image(rois[c].copy()).reshape(-1, 4)
            lab, ce, inertia, n_iter, idx = K.cells_fit(X, k, 3, p * cells + c)
            assert int(nit[p, c]) == n_iter and np.abs(cen[p, c] - ce).max() < 1e-9, (p, c)
            assert (cnt[p, c] == np.bincount(lab, minlength=k)).all()
            want_c, want_h = K.dominant_centre_hue(X, lab, ce)
            assert (dc[p, c] == want_c.astype(np.uint8)).all() and int(dh[p, c]) == want_h


@pytest.mark.parametrize("name", ["lab_k8_rs0", "lab_k4_rs7"])
def test_minibatch_kmeans_reproduces_sklearn(L, name):
    """SURVEY section 8f-4 (color-quantization/quant.py:18-20): MiniBatchKMeans(n_clusters=k, random_state=rs) through the
    product's host loop and the emulated kernels == scikit-learn 1.9.0 (same mini-batches, steps, centres, labels)"""
    import sys
    sys.path.insert(0, GOLDEN)
    import make_golden as MG
    from opticalflowclustering_b200.minibatch import MiniBatchKMeans
    z = np.load(os.path.join(GOLDEN, "minibatch_sklearn.npz"))
    X, k, rs = MG.minibatch_case(name)
    clt = MiniBatchKMeans(n_clusters=k, random_state=rs).fit(X)
    assert clt.n_steps_ == int(z[name + "_nsteps"])
    assert np.abs(clt.cluster_centers_ - z[name + "_centers"]).max() <= 1e-9
    assert (clt.labels_ == z[name + "_labels"]).all()
    assert abs(clt.inertia_ - float(z[name + "_inertia"])) <= 1e-9 * float(z[name + "_inertia"])
    assert (clt.predict(X[:500]) == z[name + "_labels"][:500]).all()


def test_minibatch_oracle_vs_sklearn_golden():
    import sys
    sys.path.insert(0, GOLDEN)
    import make_golden as MG
    from oracle import minibatch_np as MB
    z = np.load(os.path.join(GOLDEN, "minibatch_sklearn.npz"))
    for name in MG.MINIBATCH_CASES:
        X, k, rs = MG.minibatch_case(name)
        lab, cen, inertia, ns = MB.minibatch_fit(X, k, rs)
        assert ns == int(z[name + "_nsteps"]) and (lab == z[name + "_labels"]).all()
        assert np.abs(cen - z[name + "_centers"]).max() <= 1e-12
