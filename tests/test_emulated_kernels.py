"""Kernel logic on CPU: the .cu sources compiled with g++ against a fiber-based
CUDA emulation (tests/emu), compared with the oracle.  Debug tooling for a
container without a GPU; the real parity tests are the `-m gpu` ones."""
import os

import numpy as np
import pytest

from oracle import farneback_np as FB
from oracle import grid_np as G
from oracle import viz_np as V
from tests.conftest import GOLDEN

E = pytest.importorskip("tests.emu.emu_lib")


@pytest.fixture(scope="module", autouse=True)
def _build():
    E.build()


def test_emu_farneback_golden_96x128():
    z = np.load(os.path.join(GOLDEN, "flow_96x128.npz"))
    H, W = z["gray"].shape[1:]
    pl = E.Plan(W, H, max_frames=3)
    flow, mm = pl.sequence(z["gray"], want_minmax=True)
    ref, inter = FB.calc_optical_flow_farneback(z["gray"][0], z["gray"][1], return_intermediates=True)
    for l, it in enumerate(inter):
        assert np.abs(pl.buffer(l, 0, 0)[..., 0] - it["I0"]).max() < 1e-4
        assert np.abs(pl.buffer(l, 1, 0) - it["R0"][..., :4]).max() < 1e-4
        assert np.abs(pl.buffer(l, 2, 0)[..., 0] - it["R0"][..., 4]).max() < 1e-4
    for p in range(2):
        epe = np.linalg.norm(flow[p] - z["flow"][p], axis=-1)
        assert epe.mean() < 2e-6 and epe.max() < 1e-4
    mag = V.cart_to_polar(flow[..., 0], flow[..., 1])[0].reshape(2, -1)
    assert (mm.view(np.float32)[:, 0] == mag.min(1)).all() and (mm.view(np.float32)[:, 1] == mag.max(1)).all()


def test_emu_odd_size_and_params():
    from opticalflowclustering_b200.synthetic import synthetic_clip
    clip = synthetic_clip(2, 101, 150, seed=9).numpy()
    g = E.bgr2gray(clip)
    assert (g == np.stack([V.bgr2gray(f) for f in clip])).all()
    for kw in [dict(), dict(pyr_scale=0.6, levels=2, winsize=11, iterations=2, poly_n=7, poly_sigma=1.5)]:
        pl = E.Plan(150, 101, max_frames=2, **kw)
        f = pl.sequence(g)[0]
        ref = FB.calc_optical_flow_farneback(g[0], g[1], **kw)
        epe = np.linalg.norm(f - ref, axis=-1)
        assert epe.mean() < 2e-6 and epe.max() < 2e-4, (kw, epe.mean(), epe.max())


def test_emu_viz_and_grid_exact():
    z = np.load(os.path.join(GOLDEN, "flow_135x240.npz"))
    bgr, mag, _ = E.flow_to_bgr(z["flow"])
    assert (bgr == z["viz"]).all()                       # the reference's own compute() output
    out = E.grid_cells(z["viz"], 14, 25)
    for i in range(2):
        fr = z["viz"][i].copy()
        avg, hue, rois = G.grid_mean_hues(fr, 14, 25)
        assert (avg == out["avg_bgr"][i]).all() and (hue == out["avg_hue"][i]).all()
        kc = np.array([G.cluster_colors_k1(G.preprocess_image(r))[0] for r in rois])
        assert (kc == out["km_centre"][i]).all()
        lined = z["viz"][i].copy()                      # fr itself was thresholded in place (Q4)
        G.grid_mean_hues(lined, 14, 25)
        assert (E.draw_grid(z["viz"][i:i + 1], 14, 25)[0] == lined).all()


def test_emu_grid_quad_path_and_ragged_grid():
    """cells whose width is a multiple of 4 take the word-load path; ragged right/bottom remainders are ignored"""
    rng = np.random.default_rng(12)
    for (H, W, rows, cols) in [(70, 100, 4, 4), (1080 // 8, 1920 // 8, 7, 5), (50, 64, 3, 8)]:
        fr = rng.integers(0, 256, (2, H, W, 3), dtype=np.uint8)
        out = E.grid_cells(fr, rows, cols)
        for i in range(2):
            work = fr[i].copy()
            avg, hue, rois = G.grid_mean_hues(work, rows, cols)
            assert (avg == out["avg_bgr"][i]).all() and (hue == out["avg_hue"][i]).all()
            kc = np.array([G.cluster_colors_k1(G.preprocess_image(r))[0] for r in rois])
            kh = np.array([G.cluster_colors_k1(G.preprocess_image(r))[1] for r in rois])
            assert (kc == out["km_centre"][i]).all() and (kh == out["km_hue"][i]).all()


def test_emu_unsupported_flags():
    with pytest.raises(RuntimeError, match="flags"):
        E.Plan(64, 64, flags=8)
    with pytest.raises(RuntimeError, match="INITIAL_FLOW"):          # a flag-4 plan needs the initial flow
        E.Plan(64, 64, flags=4).sequence(np.zeros((2, 64, 64), np.uint8))


@pytest.mark.parametrize("flags,kw", [(256, dict()), (256, dict(winsize=9, levels=1)), (4, dict()),
                                      (260, dict(pyr_scale=0.6, levels=2, winsize=11)),
                                      (0, dict(winsize=10, levels=2, iterations=2)),     # even window: cv2's 1/winsize^2 quirk
                                      (0, dict(winsize=17, levels=1, iterations=2))])    # no unrolled kernel: run-time radius
def test_emu_flow_flags_vs_oracle(flags, kw):
    """SURVEY section 8f-2: OPTFLOW_FARNEBACK_GAUSSIAN (Gaussian window kernel) and OPTFLOW_USE_INITIAL_FLOW
    (INTER_AREA seed of the coarsest level) against the cv2-pinned oracle"""
    from opticalflowclustering_b200.synthetic import synthetic_clip
    clip = synthetic_clip(3, 77, 131, seed=4).numpy()
    g = np.stack([V.bgr2gray(f) for f in clip])
    a = dict(pyr_scale=0.5, levels=3, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2)
    a.update(kw)
    init = FB.calc_optical_flow_farneback(g[0], g[1])
    ref = FB.calc_optical_flow_farneback(g[1], g[2], init.copy(), flags=flags, **a)
    plan = E.Plan(131, 77, flags=flags, **a)
    got = plan.pair_init(g[1], g[2], init) if flags & 4 else plan.sequence(g[1:3])[0]
    epe = np.linalg.norm(got - ref, axis=-1)
    assert epe.mean() <= 5e-6 and epe.max() <= 1e-3, (epe.mean(), epe.max())


@pytest.mark.parametrize("env", [{"OFC_STRIP_MIN_W": "1", "OFC_ITER_TMEM": "1"},            # ring in TMEM + cp.async landing
                                 {"OFC_STRIP_MIN_W": "1", "OFC_ITER_TMEM": "0"},            # ring in smem, register taps
                                 {"OFC_ITER_VARIANT": "1"}])                               # square tiles everywhere
def test_emu_production_iteration_kernels_on_small_frames(env):
    """The strip-walk kernels normally only see levels wider than 512 px; the dispatch switches are read once
    per process, so a child process forces them onto small odd-sized frames (partial strips, strips that
    stick out of the frame, ragged last row groups) and compares with cv2's golden flow / the oracle."""
    import subprocess
    import sys
    code = r'''
import os, sys, numpy as np
sys.path.insert(0, os.getcwd())
from tests.emu import emu_lib as E
from oracle import farneback_np as FB
from opticalflowclustering_b200.synthetic import synthetic_clip
z = np.load("tests/golden/flow_96x128.npz")
flow = E.Plan(128, 96, max_frames=3).sequence(z["gray"])
for p in range(2):
    e = np.linalg.norm(flow[p] - z["flow"][p], axis=-1)
    assert e.mean() < 2e-6 and e.max() < 1e-4, (p, e.mean(), e.max())
for (H, W) in [(61, 250), (101, 150)]:
    g = E.bgr2gray(synthetic_clip(2, H, W, seed=H).numpy())
    f = E.Plan(W, H, max_frames=2).sequence(g)[0]
    ref = FB.calc_optical_flow_farneback(g[0], g[1])
    e = np.linalg.norm(f - ref, axis=-1)
    assert e.mean() < 2e-6 and e.max() < 2e-4, (H, W, e.mean(), e.max())
    if os.environ.get("OFC_ITER_TMEM") == "1":
        # the coarse flow up-sampled inside the walk (OFC_FUSE_UPSAMPLE=1) == the separate up-sample launch, bit for bit
        os.environ["OFC_FUSE_UPSAMPLE"] = "1"
        f2 = E.Plan(W, H, max_frames=2).sequence(g)[0]
        del os.environ["OFC_FUSE_UPSAMPLE"]
        assert (f2 == f).all(), (H, W, np.abs(f2 - f).max())
print("ok")
'''
    e = dict(os.environ)
    e.update(env)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", code], cwd=root, env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-2000:] + r.stderr[-2000:]


def test_emu_pyramid_prefilter_equals_tile_kernel(monkeypatch):
    """the one-launch pyramid pre-filter (levels that are an exact 1/2, 1/4, 1/8 of the frame) writes the bits of the
    per-level tile kernel, and both match the oracle's GaussianBlur + resize"""
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W = 256, 328                                     # 328 = 8 * 41: ragged last column block, not a multiple of 16
    g = E.bgr2gray(synthetic_clip(2, H, W, seed=23).numpy())
    got = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("OFC_PREFILTER_PYR", mode)
        pl = E.Plan(W, H, max_frames=2, iterations=1)
        assert pl.n_levels == 4
        pl.sequence(g)
        got[mode] = [pl.buffer(l, 0, f)[..., 0].copy() for l in range(pl.n_levels) for f in range(2)]
    monkeypatch.delenv("OFC_PREFILTER_PYR")
    for a, b in zip(got["1"], got["0"]):
        assert a.shape == b.shape and (a == b).all()
    _, inter = FB.calc_optical_flow_farneback(g[0], g[1], iterations=1, return_intermediates=True)
    for l, it in enumerate(inter):
        assert np.abs(got["1"][2 * l] - it["I0"]).max() < 1e-4


def test_emu_fast_encode_exhaustive_hue_boundaries():
    """the fast visualisation arithmetic (approximate hue with exact re-evaluation near byte boundaries, FADD.RZ
    truncation, per-hue multiplier table) against the oracle's statement of cv2 on flows chosen to sit ON the
    boundaries: every hue byte edge, axis-aligned and zero vectors, magnitudes at value-byte edges"""
    rng = np.random.default_rng(5)
    ang = np.concatenate([np.arange(0, 360, 2.0), np.arange(0, 360, 2.0) + 1e-4, np.arange(0, 360, 2.0) - 1e-4,
                          rng.uniform(0, 360, 4000)])
    mag = rng.uniform(0.01, 9.0, ang.size)
    mag[:97] = np.linspace(0, 9, 97)                               # includes the exact minimum and maximum
    fx = (mag * np.cos(np.deg2rad(ang))).astype(np.float32)
    fy = (mag * np.sin(np.deg2rad(ang))).astype(np.float32)
    fx[100:110] = 0.0
    fy[110:120] = 0.0
    fx[120], fy[120] = 0.0, 0.0
    n = fx.size - fx.size % 33
    flow = np.stack([fx[:n], fy[:n]], -1).reshape(1, n // 33, 33, 2)           # width 33: one scalar-tail pixel per row
    bgr, mag_sum, _ = E.flow_to_bgr(flow)
    want, m = V.flow_to_bgr(flow[0])
    assert (bgr[0] == want).all()
    assert abs(mag_sum[0] - m.astype(np.float64).sum()) <= 1e-9 * m.sum()
    bgr2, hsv = E.flow_to_hsv(flow)
    assert (bgr2 == bgr).all()
    mg, an = V.cart_to_polar(flow[0, ..., 0], flow[0, ..., 1])
    assert (hsv[0, ..., 0] == V.hue_byte(an)).all() and (hsv[0, ..., 1] == 255).all()
    assert (hsv[0, ..., 2] == V.normalize_minmax_u8(mg)).all()


@pytest.mark.parametrize("shape", [(2, 135, 240, 14, 25), (1, 77, 100, 3, 4), (1, 64, 96, 4, 6)])
def test_emu_fused_encode_grid_equals_separate_kernels(shape):
    """ofc_flow_to_bgr_grid == ofc_flow_to_bgr followed by ofc_grid_cells: quad path (cells a multiple of 4 wide),
    scalar path, and grids that leave a right / bottom remainder"""
    n, H, W, rows, cols = shape
    if (H, W) == (135, 240):
        flow = np.load(os.path.join(GOLDEN, "flow_135x240.npz"))["flow"][:n]
    else:
        rng = np.random.default_rng(H)
        flow = rng.normal(0, 2.0, (n, H, W, 2)).astype(np.float32)
    bgr, mag, mm = E.flow_to_bgr(flow)
    want = E.grid_cells(bgr, rows, cols)
    bgr2, mag2, got = E.flow_to_bgr_grid(flow, rows, cols, minmax=mm)
    assert (bgr2 == bgr).all()
    assert np.abs(mag2 - mag).max() <= 1e-9 * np.abs(mag).max()
    for k in got:
        assert (got[k] == want[k]).all(), k


def test_emu_streaming_form_equals_pairs():
    """ofc_farneback_stream_begin / _next (the previous frame's expansion stays in the workspace, two frame slots used
    alternately) gives the bits of ofc_farneback_sequence on the same frames"""
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W = 64, 96
    g = E.bgr2gray(synthetic_clip(4, H, W, seed=6).numpy())
    want = E.Plan(W, H, max_frames=4).sequence(g)
    pl = E.Plan(W, H, max_frames=2)
    pl.stream_begin(g[0])
    for t in range(1, 4):
        assert (pl.stream_next(g[t]) == want[t - 1]).all(), t
    with pytest.raises(RuntimeError, match="stream_begin"):
        E.Plan(W, H, max_frames=2).stream_next(g[1])


@pytest.mark.parametrize("levels", [0, 1])
def test_emu_pair_flow_independent_of_pair_count(levels):
    """DESIGN 5a: a pair's flow bits do not depend on how many pairs share the call.  The iteration kernel of a level is
    chosen from its geometry alone: a 240-px-wide level (a whole 240-column strip) must not switch from the square-tile
    kernel to the strip walk once n_pairs * rows passes a multiple of the SM count (the emulation reports 3 SMs, so 5
    pairs of 72 rows are past any such line and 2 pairs are short of it)."""
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W = 72, 240
    g = E.bgr2gray(synthetic_clip(6, H, W, seed=3).numpy())
    two = E.Plan(W, H, max_frames=3, levels=levels).sequence(g[:3])
    five = E.Plan(W, H, max_frames=6, levels=levels).sequence(g)
    pl = E.Plan(W, H, max_frames=2, levels=levels)
    pl.stream_begin(g[0])
    streamed = pl.stream_next(g[1])
    for name, got in (("5-pair sequence", five[0]), ("stream form", streamed)):
        d = np.abs(got - two[0])
        assert (got == two[0]).all(), (name, int((d.max(-1) > 0).sum()), float(d.max()))
    assert (five[1] == two[1]).all()
    ref = FB.calc_optical_flow_farneback(g[0], g[1], levels=levels)
    e = np.linalg.norm(two[0] - ref, axis=-1)
    assert e.mean() < 2e-6 and e.max() < 1e-4, (e.mean(), e.max())
