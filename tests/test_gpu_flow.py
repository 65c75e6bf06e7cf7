"""GPU parity tests (run on the B200 box): the CUDA path, through the C-ABI, against
the oracle, the committed goldens and -- when the wheel is importable -- live cv2.

Tolerances (north_star): flow mean end-point error <= 1e-2 px vs
cv2.calcOpticalFlowFarneback; we assert far tighter bounds on textured frames
(mean <= 5e-6 px, max <= 1e-3 px) and report the distribution.  Integer stages
(gray, visualisation given the flow, grid, k=1 clusters) are bit-exact.
"""
import os

import numpy as np
import pytest
import torch

from oracle import farneback_np as FB
from oracle import grid_np as G
from oracle import viz_np as V
from tests.conftest import GOLDEN, have_cv2

pytestmark = pytest.mark.gpu

MEAN_EPE, MAX_EPE = 5e-6, 1e-3


def _epe(a, b):
    return np.linalg.norm(a - b, axis=-1)


def _record_parity(key, stats):
    """the measured distributions also go to gpurun_out/flow_parity.json (copied to profiles/ as evidence)"""
    import json
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "flow_parity.json")
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        cur = json.load(open(path)) if os.path.exists(path) else {}
        cur[key] = stats
        json.dump(cur, open(path, "w"), indent=1)
    except OSError:
        pass


@pytest.fixture(scope="module")
def ofc():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from opticalflowclustering_b200 import _lib, flow, grid, pipeline  # noqa: F401
    _lib.lib()          # fails loudly if libofc.so is missing
    import opticalflowclustering_b200 as pkg
    return pkg


@pytest.mark.parametrize("name", ["flow_96x128", "flow_135x240", "flow_270x480"])
def test_flow_sequence_vs_golden_cv2(ofc, name):
    from opticalflowclustering_b200.flow import FarnebackPlan
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    gray = torch.from_numpy(z["gray"]).cuda()
    H, W = gray.shape[1:]
    plan = FarnebackPlan(W, H, max_frames=3)
    mm = torch.empty((2, 2), dtype=torch.int32, device="cuda")
    flow = plan.sequence(gray, minmax=mm).cpu().numpy()
    for p in range(2):
        e = _epe(flow[p], z["flow"][p])
        assert e.mean() <= MEAN_EPE and e.max() <= MAX_EPE, (name, p, e.mean(), e.max())
    # fused min/max of |flow| equals the magnitude range of the produced flow, bit for bit
    mag = V.cart_to_polar(flow[..., 0], flow[..., 1])[0].reshape(2, -1)
    got = mm.cpu().numpy().view(np.float32)
    assert (got[:, 0] == mag.min(1)).all() and (got[:, 1] == mag.max(1)).all()


def test_flow_intermediates_vs_oracle(ofc):
    from opticalflowclustering_b200.flow import FarnebackPlan
    z = np.load(os.path.join(GOLDEN, "flow_135x240.npz"))
    gray = torch.from_numpy(z["gray"]).cuda()
    plan = FarnebackPlan(240, 135, max_frames=3).keep_intermediates()
    plan.sequence(gray)
    torch.cuda.synchronize()
    _, inter = FB.calc_optical_flow_farneback(z["gray"][0], z["gray"][1], return_intermediates=True)
    assert plan.num_levels == len(inter) == 3
    for l, it in enumerate(inter):
        assert np.abs(plan.buffer(l, 0, 0).cpu().numpy()[..., 0] - it["I0"]).max() < 1e-4
        assert np.abs(plan.buffer(l, 0, 1).cpu().numpy()[..., 0] - it["I1"]).max() < 1e-4
        assert np.abs(plan.buffer(l, 1, 0).cpu().numpy() - it["R0"][..., :4]).max() < 1e-4
        assert np.abs(plan.buffer(l, 2, 1).cpu().numpy()[..., 0] - it["R1"][..., 4]).max() < 1e-4


@pytest.mark.parametrize("kw", [dict(), dict(levels=1, winsize=9, iterations=2), dict(levels=5),
                                dict(pyr_scale=0.6, levels=2, winsize=11, poly_n=7, poly_sigma=1.5),
                                dict(winsize=21), dict(winsize=5, iterations=1),
                                dict(winsize=10), dict(winsize=17, levels=2), dict(winsize=33, levels=1), dict(winsize=4)])
def test_cv2_signature_drop_in(ofc, kw):
    """calc_optical_flow_farneback(prev, next, None, ...) numpy in -> numpy out, odd size."""
    from opticalflowclustering_b200.flow import calc_optical_flow_farneback
    from opticalflowclustering_b200.synthetic import synthetic_clip
    clip = synthetic_clip(2, 101, 150, seed=9).numpy()
    g = np.stack([V.bgr2gray(f) for f in clip])
    a = dict(pyr_scale=0.5, levels=3, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2)
    a.update(kw)
    got = calc_optical_flow_farneback(g[0], g[1], None, a["pyr_scale"], a["levels"], a["winsize"], a["iterations"],
                                      a["poly_n"], a["poly_sigma"], 0)
    assert isinstance(got, np.ndarray) and got.dtype == np.float32 and got.shape == (101, 150, 2)
    ref = FB.calc_optical_flow_farneback(g[0], g[1], **a)
    e = _epe(got, ref)
    assert e.mean() <= MEAN_EPE and e.max() <= MAX_EPE, (kw, e.mean(), e.max())
    if have_cv2():
        import cv2
        ref2 = cv2.calcOpticalFlowFarneback(g[0], g[1], None, a["pyr_scale"], a["levels"], a["winsize"],
                                            a["iterations"], a["poly_n"], a["poly_sigma"], 0)
        e = _epe(got, ref2)
        assert e.mean() <= MEAN_EPE and e.max() <= MAX_EPE, (kw, e.mean(), e.max())


@pytest.mark.parametrize("flags,kw", [(256, dict()), (256, dict(winsize=21, levels=1)), (4, dict()),
                                      (260, dict(pyr_scale=0.6, levels=2, winsize=11))])
def test_flow_flags_vs_oracle_and_cv2(ofc, flags, kw):
    """SURVEY section 8f-2: cv2.OPTFLOW_FARNEBACK_GAUSSIAN (256) and cv2.OPTFLOW_USE_INITIAL_FLOW (4) through the
    cv2-signature call; bar as for flags=0 (mean EPE <= 5e-6 px, max <= 1e-3 px)"""
    from opticalflowclustering_b200.flow import calc_optical_flow_farneback
    from opticalflowclustering_b200.synthetic import synthetic_clip
    clip = synthetic_clip(3, 270, 480, seed=21).numpy()
    g = np.stack([V.bgr2gray(f) for f in clip])
    a = dict(pyr_scale=0.5, levels=3, winsize=15, iterations=3, poly_n=5, poly_sigma=1.2)
    a.update(kw)
    init = calc_optical_flow_farneback(g[0], g[1], None, 0.5, 3, 15, 3, 5, 1.2, 0)
    got = calc_optical_flow_farneback(g[1], g[2], init.copy(), a["pyr_scale"], a["levels"], a["winsize"], a["iterations"],
                                      a["poly_n"], a["poly_sigma"], flags)
    ref = FB.calc_optical_flow_farneback(g[1], g[2], init.copy(), flags=flags, **a)
    e = _epe(got, ref)
    assert e.mean() <= MEAN_EPE and e.max() <= MAX_EPE, (flags, kw, e.mean(), e.max())
    if have_cv2():
        import cv2
        ref2 = cv2.calcOpticalFlowFarneback(g[1], g[2], init.copy(), a["pyr_scale"], a["levels"], a["winsize"],
                                            a["iterations"], a["poly_n"], a["poly_sigma"], flags)
        e = _epe(got, ref2)
        assert e.mean() <= MEAN_EPE and e.max() <= MAX_EPE, (flags, kw, e.mean(), e.max())


def test_unsupported_flags_raise(ofc):
    from opticalflowclustering_b200.flow import calc_optical_flow_farneback
    g = np.zeros((64, 64), np.uint8)
    with pytest.raises(NotImplementedError):
        calc_optical_flow_farneback(g, g, None, 0.5, 3, 15, 3, 5, 1.2, 8)        # not a Farneback flag
    with pytest.raises(ValueError):
        calc_optical_flow_farneback(g, g, None, 0.5, 3, 15, 3, 5, 1.2, 4)        # OPTFLOW_USE_INITIAL_FLOW without a flow
    with pytest.raises(ValueError):
        calc_optical_flow_farneback(g, g[:32], None, 0.5, 3, 15, 3, 5, 1.2, 0)


def test_constant_frames_zero_flow(ofc):
    from opticalflowclustering_b200.flow import calc_optical_flow_farneback, flow_to_bgr
    g = np.full((80, 96), 77, np.uint8)
    fl = calc_optical_flow_farneback(g, g, None, 0.5, 3, 15, 3, 5, 1.2, 0)
    assert np.all(fl == 0)
    bgr = flow_to_bgr(torch.from_numpy(fl[None]).cuda()).cpu().numpy()
    assert np.all(bgr == 0)                                      # constant magnitude -> V = 0 -> black


@pytest.mark.parametrize("name", ["flow_96x128", "flow_135x240", "flow_270x480"])
def test_visualisation_bit_exact_given_flow(ofc, name):
    """golden viz = the reference's ComputeOpticalFLow.compute output for the cv2 flow"""
    from opticalflowclustering_b200.flow import bgr2gray, flow_to_bgr
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    assert (bgr2gray(torch.from_numpy(z["clip"]).cuda()).cpu().numpy() == z["gray"]).all()
    fl = torch.from_numpy(z["flow"]).cuda()
    bgr, mean_mag = flow_to_bgr(fl, want_mean_magnitude=True)
    assert (bgr.cpu().numpy() == z["viz"]).all()
    mag = V.cart_to_polar(z["flow"][..., 0], z["flow"][..., 1])[0]
    assert np.allclose(mean_mag.cpu().numpy(), mag.reshape(2, -1).astype(np.float64).mean(1), rtol=1e-12)


def test_visualisation_row_tail_rounding(ofc):
    """cv2's HSV2BGR rounds in the scalar tail (W % 32 pixels) and truncates elsewhere"""
    from opticalflowclustering_b200.flow import flow_to_bgr
    rng = np.random.default_rng(2)
    for W in (33, 50, 64, 100):
        fl = (rng.standard_normal((2, 40, W, 2)) * 3).astype(np.float32)
        got = flow_to_bgr(torch.from_numpy(fl).cuda()).cpu().numpy()
        want = np.stack([V.flow_to_bgr(f)[0] for f in fl])
        assert (got == want).all(), W
        if have_cv2():
            import cv2
            for i in range(2):
                m, a = cv2.cartToPolar(fl[i, ..., 0], fl[i, ..., 1])
                mask = np.zeros((40, W, 3), np.uint8)
                mask[..., 1] = 255
                mask[..., 0] = a * 180 / np.pi / 2
                mask[..., 2] = cv2.normalize(m, None, 0, 255, cv2.NORM_MINMAX)
                assert (got[i] == cv2.cvtColor(mask, cv2.COLOR_HSV2BGR)).all(), W


def test_compute_optical_flow_class_drop_in(ofc):
    """ComputeOpticalFLow(firstframe).compute(frame) vs the reference's output (golden viz).

    Residual differences come only from ~1e-7 px flow differences crossing uint8
    truncation boundaries (SURVEY.md H3): a handful of bytes, off by one step."""
    from opticalflowclustering_b200.computeOpticalFlowModule import ComputeOpticalFLow
    z = np.load(os.path.join(GOLDEN, "flow_270x480.npz"))
    cof = ComputeOpticalFLow(z["clip"][0].copy())
    assert (cof.width, cof.height) == (480, 270)
    for p in range(2):
        out = cof.compute(z["clip"][p + 1].copy())
        assert isinstance(out, np.ndarray) and out.dtype == np.uint8 and out.shape == (270, 480, 3)
        bad = (out != z["viz"][p]).any(-1).mean()
        assert bad < 2e-3, bad
        assert (cof.prev_gray == z["gray"][p + 1]).all()


def test_grid_stage_bit_exact(ofc):
    from opticalflowclustering_b200.grid import draw_grid, grid_cells
    z = np.load(os.path.join(GOLDEN, "flow_270x480.npz"))
    viz = torch.from_numpy(z["viz"]).cuda()
    out = {k: v.cpu().numpy() for k, v in grid_cells(viz, 14, 25).items()}
    for i in range(2):
        fr = z["viz"][i].copy()
        avg, hue, rois = G.grid_mean_hues(fr, 14, 25)
        assert (avg == out["avg_bgr"][i]).all() and (hue == out["avg_hue"][i]).all()
        lined = fr.copy()
        kc, kh = zip(*[G.cluster_colors_k1(G.preprocess_image(r)) for r in rois])
        assert (np.array(kc) == out["km_centre"][i]).all() and (np.array(kh) == out["km_hue"][i]).all()
        assert (draw_grid(viz[i].clone(), 14, 25).cpu().numpy() == lined).all()


def test_grid_golden_g2_g3(ofc):
    """the reference's saved 51x51 cells -> OutCSV hues (G2) and rgb_values hues (G3)"""
    from opticalflowclustering_b200.grid import grid_cells
    z = np.load(os.path.join(GOLDEN, "g23_cells.npz"))
    cells = z["cells"]                                           # [3,350,51,51,3] BGR as saved
    rgb = np.ascontiguousarray(cells[..., ::-1]).reshape(-1, 51, 51, 3)    # read_image swaps to RGB (Q5)
    out = grid_cells(torch.from_numpy(rgb).cuda(), 1, 1, draw_lines=False, threshold=30, want=("km_hue",))
    assert (out["km_hue"].cpu().numpy().reshape(3, 350) == z["outcsv_hues"]).all()
    out = grid_cells(torch.from_numpy(cells.reshape(-1, 51, 51, 3)).cuda(), 1, 1, draw_lines=False, threshold=0,
                     want=("avg_hue",))
    got = out["avg_hue"].cpu().numpy().reshape(3, 350)
    interior = np.array([(c // 25 > 0) and (c % 25 > 0) for c in range(350)])
    assert (got[:, interior] == z["rgb_values_hues"][:, interior]).all()


def test_pipeline_chunking_invariance_and_oracle(ofc):
    """clip pipeline: chunked (with 1-frame halo) == one shot, and hues follow the oracle chain"""
    from opticalflowclustering_b200.pipeline import ClipPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, T = 144, 208, 7
    clip = synthetic_clip(T, H, W, seed=21)
    a = ClipPipeline(W, H, chunk_frames=T, rows=6, cols=8).process_clip(clip)
    b = ClipPipeline(W, H, chunk_frames=3, rows=6, cols=8).process_clip(clip)
    for k in a:
        assert torch.equal(a[k], b[k]), k
    # carry=True: new frames only, the shared frame stays on the device as prev_gray
    c = ClipPipeline(W, H, chunk_frames=4, rows=6, cols=8)
    dev_clip = clip.cuda()
    assert c.run_chunk(dev_clip[0:3]) == 2
    got = [c.avg_hue[:2].cpu()]
    assert c.run_chunk(dev_clip[3:6], carry=True) == 3
    got.append(c.avg_hue[:3].cpu())
    assert c.run_chunk(dev_clip[6:7], carry=True) == 1
    got.append(c.avg_hue[:1].cpu())
    assert torch.equal(torch.cat(got), a["avg_hue"])
    with pytest.raises(ValueError):
        ClipPipeline(W, H, chunk_frames=4, rows=6, cols=8).run_chunk(dev_clip[0:2], carry=True)
    # streaming ingest from a host frame iterator (pinned staging + copy stream) gives the same rows
    st = ClipPipeline(W, H, chunk_frames=3, rows=6, cols=8).process_stream(iter(clip.numpy()))
    for k in a:
        assert torch.equal(a[k], st[k]), k
    seen = []
    n = ClipPipeline(W, H, chunk_frames=4, rows=6, cols=8).process_stream(
        (f for f in clip.numpy()), on_pairs=lambda first, res: seen.append((first, res["viz"].shape[0])), want_viz=True)
    assert n == T - 1 and seen == [(0, 3), (3, 3)]
    pipe = ClipPipeline(W, H, chunk_frames=T, rows=6, cols=8)
    pipe.run_chunk(clip.cuda())
    flow = pipe.flow.cpu().numpy()
    viz = pipe.viz.cpu().numpy()
    for p in range(T - 1):
        want, mag = V.flow_to_bgr(flow[p])
        assert (viz[p] == want).all()
        fr = viz[p].copy()
        _, hue, rois = G.grid_mean_hues(fr, 6, 8)
        assert (a["avg_hue"][p].numpy() == hue).all()
        kh = [G.cluster_colors_k1(G.preprocess_image(r))[1] for r in rois]
        assert (a["km_hue"][p].numpy() == np.array(kh)).all()
        assert abs(a["mean_magnitude"][p].item() - mag.astype(np.float64).mean()) < 1e-9


@pytest.mark.parametrize("size", [(720, 1280), (1080, 1920)])
def test_full_size_properties(ofc, size):
    """BASELINE sizes: parity through properties that do not need a CPU oracle run --
    (a) translation recovery: mean flow of the synthetic warp within 0.1 px of truth
        (Farneback's own accuracy on noisy frames; cv2 gives the same error);
    (b) batch invariance: pair t in a sequence == the same pair computed alone, bit for bit;
    (c) determinism: two runs are bit-identical."""
    from opticalflowclustering_b200.flow import FarnebackPlan, bgr2gray
    from opticalflowclustering_b200.synthetic import synthetic_clip, true_flow
    H, W = size
    clip = synthetic_clip(3, H, W, seed=5, device="cuda")
    gray = bgr2gray(clip)
    plan = FarnebackPlan(W, H, max_frames=3)
    f1 = plan.sequence(gray).clone()
    f2 = plan.sequence(gray).clone()
    assert torch.equal(f1, f2)
    solo = FarnebackPlan(W, H, max_frames=2).pair(gray[1], gray[2])
    assert torch.equal(solo, f1[1])
    truth = true_flow(H, W, device="cuda")
    inner = (slice(40, H - 40), slice(40, W - 40))
    err = (f1[0][inner] - truth[inner]).norm(dim=-1)
    assert err.mean().item() < 0.1, err.mean().item()
    if have_cv2():
        # the direct comparison at BOTH BASELINE sizes (1080p is the headline config and the one width whose strips
        # are never ragged), with the distribution BASELINE.md section 5 asks for
        import cv2
        from tests.conftest import flow_parity_stats
        g = gray.cpu().numpy()
        ref = cv2.calcOpticalFlowFarneback(g[0], g[1], None, 0.5, 3, 15, 3, 5, 1.2, 0)
        top = plan.num_levels - 1
        st = flow_parity_stats(f1[0].cpu().numpy(), ref, plan.buffer(top, 1, 0).cpu().numpy(), plan.buffer(top, 2, 0).cpu().numpy()[..., 0])
        print(f"\nflow parity vs cv2 {W}x{H}: {st}")
        _record_parity(f"{W}x{H}_L3", st)
        assert st["mean"] <= MEAN_EPE and st["max"] <= MAX_EPE, st
        assert st["p99"] <= 1e-4 and st["p99.9"] <= 5e-4 and st["max_well_conditioned"] <= MAX_EPE, st
        assert st["well_conditioned_share"] > 0.5


def test_4k_five_level_pyramid_properties(ofc):
    """BASELINE configs[3] geometry: 3840x2160, levels=5 (6 scales down to 120x68, 79-tap pre-filter).
    Too large for the numpy oracle, so: determinism, pair-vs-sequence invariance, translation recovery,
    and agreement with live cv2 on the same frames when the wheel is importable."""
    from opticalflowclustering_b200.flow import FarnebackPlan, bgr2gray
    from opticalflowclustering_b200.synthetic import synthetic_clip, true_flow
    H, W = 2160, 3840
    clip = synthetic_clip(3, H, W, seed=8, device="cuda")
    gray = bgr2gray(clip)
    plan = FarnebackPlan(W, H, max_frames=3, levels=5)
    assert plan.num_levels == 6 and plan.level_size(0) == (120, 68)
    f1 = plan.sequence(gray).clone()
    f2 = plan.sequence(gray).clone()
    assert torch.equal(f1, f2)
    solo = FarnebackPlan(W, H, max_frames=2, levels=5).pair(gray[0], gray[1])
    assert torch.equal(solo, f1[0])
    truth = true_flow(H, W, device="cuda")
    inner = (slice(60, H - 60), slice(60, W - 60))
    assert (f1[0][inner] - truth[inner]).norm(dim=-1).mean().item() < 0.1
    if have_cv2():
        import cv2
        g = gray.cpu().numpy()
        ref = cv2.calcOpticalFlowFarneback(g[0], g[1], None, 0.5, 5, 15, 3, 5, 1.2, 0)
        from tests.conftest import flow_parity_stats
        top = plan.num_levels - 1
        st = flow_parity_stats(f1[0].cpu().numpy(), ref, plan.buffer(top, 1, 0).cpu().numpy(), plan.buffer(top, 2, 0).cpu().numpy()[..., 0])
        print(f"\nflow parity vs cv2 {W}x{H} levels=5: {st}")
        _record_parity(f"{W}x{H}_L5", st)
        assert st["mean"] <= MEAN_EPE and st["max"] <= 5 * MAX_EPE, st
        assert st["p99"] <= 1e-4 and st["max_well_conditioned"] <= 5 * MAX_EPE, st


# ---- round-2 kernels: every fused / fast form against the form it replaces, at the BASELINE sizes -------------------
def _flow_with_env(monkeypatch, env, W, H, gray, levels=3):
    from opticalflowclustering_b200.flow import FarnebackPlan
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    plan = FarnebackPlan(W, H, max_frames=int(gray.shape[0]), levels=levels).keep_intermediates()
    out = plan.sequence(gray).clone()
    inter = [plan.buffer(l, 0, 1).clone() for l in range(plan.num_levels)]
    for k in env:
        monkeypatch.delenv(k)
    return out, inter


@pytest.mark.parametrize("size,levels", [((1080, 1920), 3), ((720, 1280), 3), ((2160, 3840), 5)])
def test_pyramid_prefilter_bit_identical(ofc, size, levels, monkeypatch):
    """one-launch pyramid pre-filter == per-level tile kernels: I of every level and the final flow, bit for bit"""
    from opticalflowclustering_b200.flow import bgr2gray
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W = size
    gray = bgr2gray(synthetic_clip(2, H, W, seed=31, device="cuda"))
    new, inew = _flow_with_env(monkeypatch, {"OFC_PREFILTER_PYR": "1"}, W, H, gray, levels)
    old, iold = _flow_with_env(monkeypatch, {"OFC_PREFILTER_PYR": "0"}, W, H, gray, levels)
    for a, b in zip(inew, iold):
        assert torch.equal(a, b)
    assert torch.equal(new, old)


@pytest.mark.parametrize("size,levels", [((1080, 1920), 3), ((720, 1280), 3), ((2160, 3840), 5)])
def test_round2b_fast_forms_bit_identical(ofc, size, levels, monkeypatch):
    """the forms added late in round 2 against the ones they replace, final flow and I of every level bit for bit: lower
    taps shared between rows (OFC_TMEM_SHARE), exact x2 up-sample kernel (OFC_UPSAMPLE_X2), staged 8-bit rows in the
    full-resolution polynomial expansion (OFC_POLY_STAGE)"""
    from opticalflowclustering_b200.flow import bgr2gray
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W = size
    gray = bgr2gray(synthetic_clip(3, H, W, seed=37, device="cuda"))
    new, inew = _flow_with_env(monkeypatch, {"OFC_TMEM_SHARE": "1", "OFC_UPSAMPLE_X2": "1", "OFC_POLY_STAGE": "1"}, W, H, gray, levels)
    for off in ("OFC_TMEM_SHARE", "OFC_UPSAMPLE_X2", "OFC_POLY_STAGE"):
        old, iold = _flow_with_env(monkeypatch, {off: "0"}, W, H, gray, levels)
        for a, b in zip(inew, iold):
            assert torch.equal(a, b), off
        assert torch.equal(new, old), off


@pytest.mark.parametrize("size,grid", [((1080, 1920), (14, 25)), ((720, 1280), (14, 25)), ((270, 484), (5, 7))])
def test_fused_encode_grid_equals_separate_kernels(ofc, size, grid):
    """ofc_flow_to_bgr_grid == ofc_flow_to_bgr + ofc_grid_cells on real flow fields: word path (1080p cells are 76 px
    wide), scalar path (720p: 51 px), ragged remainder; and both equal the oracle's statement of cv2"""
    from opticalflowclustering_b200.pipeline import ClipPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W = size
    rows, cols = grid
    clip = synthetic_clip(3, H, W, seed=41, device="cuda")
    a = ClipPipeline(W, H, chunk_frames=3, rows=rows, cols=cols)
    assert a.fuse_grid
    a.run_chunk(clip)
    b = ClipPipeline(W, H, chunk_frames=3, rows=rows, cols=cols)
    b.fuse_grid = False
    b.run_chunk(clip)
    for name in ("viz", "avg_bgr", "avg_hue", "km_centre", "km_hue"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert (a.mag_sum - b.mag_sum).abs().max().item() <= 1e-9 * b.mag_sum.abs().max().item()
    want, _ = V.flow_to_bgr(a.flow[0].cpu().numpy())
    assert (a.viz[0].cpu().numpy() == want).all()


def test_compute_optical_flow_mask_attribute(ofc):
    """ComputeOpticalFLow.mask follows the reference (computeOpticalFlowModule.py:14-15, 28-31): S = 255 always, H and V
    bytes of the latest pair after compute()"""
    from opticalflowclustering_b200.computeOpticalFlowModule import ComputeOpticalFLow
    from opticalflowclustering_b200.synthetic import synthetic_clip
    clip = synthetic_clip(3, 120, 168, seed=3).numpy()
    cf = ComputeOpticalFLow(clip[0])
    m0 = cf.mask
    assert m0.shape == clip[0].shape and (m0[..., 1] == 255).all() and (m0[..., 0] == 0).all() and (m0[..., 2] == 0).all()
    for f in clip[1:]:
        out = cf.compute(f)
        fl = cf.last_flow.cpu().numpy()
        mag, ang = V.cart_to_polar(fl[..., 0], fl[..., 1])
        m = cf.mask
        assert (m[..., 0] == V.hue_byte(ang)).all() and (m[..., 1] == 255).all() and (m[..., 2] == V.normalize_minmax_u8(mag)).all()
        assert (out == V.flow_to_bgr(fl)[0]).all()


def test_one_process_two_devices(ofc):
    """the > 48 KB shared-memory opt-in of every kernel is recorded per device: the same process runs the pipeline on
    cuda:0 and then on cuda:1 (skipped on a one-GPU box)"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from opticalflowclustering_b200.pipeline import ClipPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    clip = synthetic_clip(3, 288, 720, seed=2)
    res = []
    for d in (0, 1):
        with torch.cuda.device(d):
            pipe = ClipPipeline(720, 288, chunk_frames=3, rows=6, cols=8, device=f"cuda:{d}", n_clusters=2)
            pipe.run_chunk(clip.to(f"cuda:{d}"))
            torch.cuda.synchronize(d)
            res.append((pipe.avg_hue.cpu(), pipe.km_hue.cpu(), pipe.flow.cpu()))
    for u, v in zip(res[0], res[1]):
        assert torch.equal(u, v)


@pytest.mark.parametrize("lanes,n_clusters", [(2, 1), (3, 1), (2, 3)])
def test_laned_pipeline_equals_single_pipeline(ofc, lanes, n_clusters):
    """LanedPipeline (chunks dealt over pipelines on their own streams, the shared frame's gray image handed from lane to
    lane) gives the hue rows, k-means hues and magnitudes of one ClipPipeline walking the same clip"""
    from opticalflowclustering_b200.pipeline import ClipPipeline, LanedPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, T, F = 144, 200, 14, 4
    clip = synthetic_clip(T, H, W, seed=23, device="cuda")
    one = ClipPipeline(W, H, chunk_frames=F, rows=6, cols=8, n_clusters=n_clusters, kmeans_seed=9).process_clip(clip)
    many = LanedPipeline(W, H, lanes=lanes, chunk_frames=F, rows=6, cols=8, n_clusters=n_clusters, kmeans_seed=9).process_clip(clip)
    for key in ("avg_hue", "km_hue", "mean_magnitude"):
        assert torch.equal(one[key], many[key]), key
    # and twice on the same object (events and the lane order are reused)
    lp = LanedPipeline(W, H, lanes=lanes, chunk_frames=F, rows=6, cols=8, n_clusters=n_clusters, kmeans_seed=9)
    a = lp.process_clip(clip)
    b = lp.process_clip(clip)
    for key in ("avg_hue", "km_hue", "mean_magnitude"):
        assert torch.equal(a[key], b[key]) and torch.equal(a[key], one[key]), key
