"""The flow at the shapes the benchmark runs and on hard motion, against live cv2 (run on the B200 box).

test_gpu_flow.py compares 2- and 3-frame sequences of the gentle `synthetic_clip` with cv2.  Here:
(a) a pair's flow bits do not depend on the call it is computed in (DESIGN 5a) at the production shapes: 32-pair 1080p
    chunks, tail chunks, `FarnebackPlan.pair`, the per-frame drop-in, 28-pair 4K sequences;
(b) the benchmark's own 33-frame 1080p chunk against cv2, and its visualisation / grid / hues against the oracle;
(c) hard motion -- large translation, rotation with zoom, motion boundaries, expansion -- against cv2, with the shared
    lower taps of the strip walk on and off (OFC_TMEM_SHARE);
(d) ragged strip layouts at production widths against cv2.

cv2 is the reference and must be importable: a missing cv2 fails these tests.  Bars as in test_gpu_flow.py: mean EPE
<= 5e-6 px, p99 <= 1e-4 px, max over the well-conditioned pixels <= 1e-3 px (see LOST_* for the fields the pyramid
cannot follow everywhere).
"""
import importlib

import numpy as np
import pytest
import torch

from oracle import grid_np as G
from oracle import viz_np as V
from tests.conftest import flow_parity_stats

pytestmark = pytest.mark.gpu

MEAN_EPE, P99_EPE, MAX_WELL = 5e-6, 1e-4, 1e-3
FB_ARGS = (0.5, 3, 15, 3, 5, 1.2, 0)            # the reference's calcOpticalFlowFarneback literals


@pytest.fixture(scope="module")
def ofc():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from opticalflowclustering_b200 import _lib
    _lib.lib()
    import opticalflowclustering_b200 as pkg
    return pkg


@pytest.fixture(scope="module")
def cv2():
    return importlib.import_module("cv2")       # the reference: no skip when it is missing


def _gray(clip):
    from opticalflowclustering_b200.flow import bgr2gray
    return bgr2gray(clip if clip.is_cuda else clip.cuda())


# Where a field moves content further than the pyramid can follow (rotation with zoom and expansion at these sizes: up to
# 80 px at the corners of a 1080p frame, cv2 itself ends tens of px from the truth there), the iteration solves systems
# warped to unrelated texture and amplifies the last-bit differences of any two implementations.  The float64 oracle
# differs from cv2 by as much there: on a 320 x 200 corner crop of the 720p rotation clip it gives mean 3.9e-6 / p99
# 3.6e-5 / max 1.1e-4 px against 3.2e-7 / 2.0e-6 / 7.0e-6 px on a crop the pyramid follows (the emulated build: 5.7e-6 /
# 6.1e-5 / 1.8e-4 and 1.2e-6 / 5.0e-6 / 2.2e-5).  So for those fields the bars above hold on the pixels cv2 tracks
# (within TRACKED_PX of the true flow), and the whole frame gets the bars below (B200 runs: at most mean 1.1e-5,
# p99 1.4e-4, max 6.7e-3 px).
TRACKED_PX = 0.5
LOST_MEAN, LOST_P99, LOST_MAX = 3e-5, 5e-4, 2e-2


def _parity(cv2, tag, plan, flow, gray, p, levels=3, truth=None):
    """stats of pair p (frames p, p+1 of the uint8 numpy `gray`) against cv2; the well-conditioned mask comes from the
    plan's level-0 polynomial expansion of frame p.  ``truth``: the true flow of a field the pyramid cannot follow
    everywhere -- the bars then hold on the tracked pixels and the whole frame gets the LOST_* bars"""
    ref = cv2.calcOpticalFlowFarneback(gray[p], gray[p + 1], None, 0.5, levels, 15, 3, 5, 1.2, 0)
    top = plan.num_levels - 1
    st = flow_parity_stats(flow, ref, plan.buffer(top, 1, p).cpu().numpy(), plan.buffer(top, 2, p).cpu().numpy()[..., 0])
    print(f"\nflow parity vs cv2 {tag} pair {p}: {st}")
    assert st["well_conditioned_share"] > 0.5, (tag, p, st)
    if truth is None:
        assert st["mean"] <= MEAN_EPE and st["p99"] <= P99_EPE and st["max_well_conditioned"] <= MAX_WELL, (tag, p, st)
        return st
    assert st["mean"] <= LOST_MEAN and st["p99"] <= LOST_P99 and st["max"] <= LOST_MAX, (tag, p, st)
    tracked = np.linalg.norm(ref - truth, axis=-1) < TRACKED_PX
    e = np.linalg.norm(np.asarray(flow, np.float64) - ref, axis=-1)[tracked]
    tst = {"tracked_share": float(tracked.mean()), "mean": float(e.mean()), "p99": float(np.percentile(e, 99)),
           "max": float(e.max())}
    print(f"flow parity vs cv2 {tag} pair {p}, pixels cv2 tracks: {tst}")
    assert tst["tracked_share"] > 0.05, (tag, p, tst)
    assert tst["mean"] <= MEAN_EPE and tst["p99"] <= P99_EPE and tst["max"] <= MAX_WELL, (tag, p, tst)
    return st


# ---- hard-motion clips ------------------------------------------------------------------------------------------------
def _texture(cv2, h, w, seed):
    """blurred uniform noise (sigma 2.5, as synthetic.py) stretched to 0..255, float32"""
    rng = np.random.default_rng(seed)
    b = cv2.GaussianBlur(rng.uniform(0, 255, (h, w)).astype(np.float32), (0, 0), 2.5)
    return ((b - b.min()) / (b.max() - b.min()) * 255.0).astype(np.float32)


def _affine_powers(A, k):
    M = np.eye(2)
    for _ in range(abs(k)):
        M = M @ (A if k > 0 else np.linalg.inv(A))
    return M


def hard_clip(cv2, field, n, H, W, seed=0, alternate=False):
    """uint8 gray frames [n,H,W] of one of the hard-motion fields and the true flow [H,W,2] of pair 0.

    Frame k shows the texture moved k times by the field (``alternate``: moved back and forth, so pair k+1 undoes pair
    k and a long chunk keeps its texture scale).  The texture is larger than the frame, so content enters from outside.
      translation: (+9.5, -6.25) px per frame;
      rotation:    3.5 degrees with zoom 1.04 about the centre -- both components change down every column;
      boundaries:  16 x 32 px textured tiles in a checkerboard moving (+3.5, +2.25) px against the rest, which moves
                   (-2.75, -1.5) px: motion boundaries and occlusions every 16 rows;
      expansion:   zoom 1.03 about the centre -- the warped samples leave the frame on all four sides."""
    rng = np.random.default_rng(seed + 1000)
    M = 160
    base = _texture(cv2, H + 2 * M, W + 2 * M, seed)
    tiles = _texture(cv2, H + 2 * M, W + 2 * M, seed + 1)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    cx, cy = (W - 1) / 2.0, (H - 1) / 2.0

    def sample(img, X, Y):
        return cv2.remap(img, (X + M).astype(np.float32), (Y + M).astype(np.float32), cv2.INTER_LINEAR,
                         borderMode=cv2.BORDER_REFLECT)

    if field in ("rotation", "expansion"):
        th = np.deg2rad(3.5) if field == "rotation" else 0.0
        s = 1.04 if field == "rotation" else 1.03
        A = s * np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        truth = np.stack([(A[0, 0] - 1) * (xx - cx) + A[0, 1] * (yy - cy), A[1, 0] * (xx - cx) + (A[1, 1] - 1) * (yy - cy)], -1)
    elif field == "translation":
        truth = np.broadcast_to(np.array([9.5, -6.25]), (H, W, 2)).copy()
    elif field == "boundaries":
        fg, bg = np.array([3.5, 2.25]), np.array([-2.75, -1.5])
        in_tile = lambda X, Y: ((np.floor(Y / 16) + np.floor(X / 32)) % 2) == 0     # noqa: E731  (frame-0 coordinates)
        truth = np.where(in_tile(xx, yy)[..., None], fg, bg)
    else:
        raise ValueError(field)
    frames = []
    for k in range(n):
        j = (k % 2) if alternate else k
        if field in ("rotation", "expansion"):
            Mi = _affine_powers(A, -j)        # frame j at x shows the texture at c + A^-j (x - c)
            X = cx + Mi[0, 0] * (xx - cx) + Mi[0, 1] * (yy - cy)
            Y = cy + Mi[1, 0] * (xx - cx) + Mi[1, 1] * (yy - cy)
            img = sample(base, X, Y)
        elif field == "translation":
            img = sample(base, xx - j * 9.5, yy + j * 6.25)
        else:
            Xf, Yf = xx - j * fg[0], yy - j * fg[1]
            Xb, Yb = xx - j * bg[0], yy - j * bg[1]
            img = np.where(in_tile(Xf, Yf), sample(tiles, Xf, Yf), sample(base, Xb, Yb))
        img = img + rng.normal(0, 3.0, (H, W))
        frames.append(np.clip(np.rint(img), 0, 255).astype(np.uint8))
    return np.stack(frames), truth


def unshared_tap_share(flow):
    """share of pixels whose warped tap address in the strip walk (clamp(floor(y + v), 0, h - 2) * w + clamp(floor(x + u),
    0, w - 2), flow_kernels.cu request_row) is not the previous row's address + w: the rows that request their upper taps
    themselves instead of taking them from the row above"""
    h, w = flow.shape[:2]
    fl = np.asarray(flow, np.float32)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    x1 = np.clip(np.floor(xx + fl[..., 0]), 0, w - 2).astype(np.int64)
    y1 = np.clip(np.floor(yy + fl[..., 1]), 0, h - 2).astype(np.int64)
    o1 = y1 * w + x1
    return float((o1[1:] != o1[:-1] + w).mean())


# ---- (a) invariance at production shapes ------------------------------------------------------------------------------
def test_1080p_chunk_pairs_equal_pair_and_per_frame_dropin(ofc):
    """32 pairs of a 33-frame 1080p sequence == each pair alone == ComputeOpticalFLow fed frame by frame; the fused per-pair
    min/max of |flow| (atomics whose CTA row ranges cross pair boundaries) == the range of the produced flow"""
    from opticalflowclustering_b200.computeOpticalFlowModule import ComputeOpticalFLow
    from opticalflowclustering_b200.flow import FarnebackPlan
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, T = 1080, 1920, 33
    clip = synthetic_clip(T, H, W, seed=51, device="cuda")
    gray = _gray(clip)
    mm = torch.empty((T - 1, 2), dtype=torch.int32, device="cuda")
    seq = FarnebackPlan(W, H, max_frames=T).sequence(gray, minmax=mm).clone()
    solo = FarnebackPlan(W, H, max_frames=2)
    cof = ComputeOpticalFLow(clip[0])
    bad_pair, bad_frame = [], []
    for p in range(T - 1):
        if not torch.equal(solo.pair(gray[p], gray[p + 1]), seq[p]):
            bad_pair.append(p)
        cof.compute(clip[p + 1])
        if not torch.equal(cof.last_flow, seq[p]):
            bad_frame.append(p)
    assert not bad_pair and not bad_frame, (bad_pair, bad_frame)
    got = mm.cpu().numpy().view(np.float32)
    for p in range(T - 1):
        f = seq[p].cpu().numpy()
        mag = V.cart_to_polar(f[..., 0], f[..., 1])[0]
        assert got[p, 0] == mag.min() and got[p, 1] == mag.max(), (p, got[p], mag.min(), mag.max())


def _walk_chunks(pipe, clip):
    """ClipPipeline over a whole device clip in chunks with the one-frame halo (as process_clip), keeping the flow"""
    T = int(clip.shape[0])
    out = {"flow": [], "avg_hue": [], "km_hue": [], "mean_magnitude": []}
    t = 0
    while t < T - 1:
        first = t == 0
        n = min(pipe.F, T - t) if first else min(pipe.F - 1, T - 1 - t)
        P = pipe.run_chunk(clip[t:t + n] if first else clip[t + 1:t + 1 + n], carry=not first)
        out["flow"].append(pipe.flow[:P].clone())
        out["avg_hue"].append(pipe.avg_hue[:P].cpu())
        out["km_hue"].append(pipe.km_hue[:P].cpu())
        out["mean_magnitude"].append(pipe.mag_sum[:P].cpu() / float(pipe.H * pipe.W))
        t += P
    return {k: torch.cat(v) for k, v in out.items()}


def test_1080p_pipeline_chunk_size_invariance(ofc):
    """ClipPipeline at 1080p with chunks of 33 (32 pairs, then a 7-pair tail), 9 and 3 frames, and process_stream: the
    flow, hue rows, k-means hues and mean magnitudes of a 40-frame clip are identical"""
    from opticalflowclustering_b200.pipeline import ClipPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, T = 1080, 1920, 40
    clip = synthetic_clip(T, H, W, seed=52, device="cuda")
    res = {F: _walk_chunks(ClipPipeline(W, H, chunk_frames=F), clip) for F in (33, 9, 3)}
    for F in (9, 3):
        for k in res[33]:
            assert torch.equal(res[33][k], res[F][k]), (F, k)
    st = ClipPipeline(W, H, chunk_frames=33).process_stream(iter(clip.cpu().numpy()))
    for k in ("avg_hue", "km_hue", "mean_magnitude"):
        assert torch.equal(st[k], res[33][k]), ("stream", k)


def test_4k_five_levels_28_pairs_equal_pairs_alone(ofc):
    """3840 x 2160, levels=5: pairs of a 29-frame sequence == the same pairs computed alone"""
    from opticalflowclustering_b200.flow import FarnebackPlan
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, T = 2160, 3840, 29
    gray = _gray(synthetic_clip(T, H, W, seed=53, device="cuda"))
    seq = FarnebackPlan(W, H, max_frames=T, levels=5).sequence(gray)
    solo = FarnebackPlan(W, H, max_frames=2, levels=5)
    for p in (0, 13, T - 2):
        assert torch.equal(solo.pair(gray[p], gray[p + 1]), seq[p]), p


# ---- (b) the benchmark's chunk against cv2 and the oracle -------------------------------------------------------------
def test_bench_chunk_vs_cv2_and_oracle(ofc, cv2):
    """The first 33-frame chunk of bench.py's clip (synthetic_clip, seed 0) through ClipPipeline: 8 of its 32 pairs against
    cv2, and the visualisation, grid hues, k = 1 hues and mean magnitude of those pairs against the oracle applied to the
    pipeline's own flow, bit for bit"""
    from opticalflowclustering_b200.pipeline import ClipPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, T = 1080, 1920, 33
    clip = synthetic_clip(T, H, W, seed=0, device="cuda")
    pipe = ClipPipeline(W, H, chunk_frames=T, rows=14, cols=25)
    assert pipe.run_chunk(clip) == T - 1
    torch.cuda.synchronize()
    gray = pipe.gray.cpu().numpy()
    for p in (0, 3, 8, 13, 17, 22, 27, 31):
        flow = pipe.flow[p].cpu().numpy()
        _parity(cv2, "bench chunk 1920x1080", pipe.plan, flow, gray, p)
        viz = pipe.viz[p].cpu().numpy()
        want, mag = V.flow_to_bgr(flow)
        assert (viz == want).all(), p
        fr = viz.copy()
        _, hue, rois = G.grid_mean_hues(fr, 14, 25)
        assert (pipe.avg_hue[p].cpu().numpy() == hue).all(), p
        kh = np.array([G.cluster_colors_k1(G.preprocess_image(r))[1] for r in rois])
        assert (pipe.km_hue[p].cpu().numpy() == kh).all(), p
        assert abs(pipe.mag_sum[p].item() / float(H * W) - mag.astype(np.float64).mean()) < 1e-9, p


# ---- (c) hard motion against cv2 -------------------------------------------------------------------------------------
def _flow_share(monkeypatch, W, H, gray_dev, share):
    from opticalflowclustering_b200.flow import FarnebackPlan
    monkeypatch.setenv("OFC_TMEM_SHARE", share)
    plan = FarnebackPlan(W, H, max_frames=int(gray_dev.shape[0]))
    flow = plan.sequence(gray_dev).clone()
    monkeypatch.delenv("OFC_TMEM_SHARE")
    return plan, flow


@pytest.mark.parametrize("field", ["translation", "rotation", "boundaries", "expansion"])
@pytest.mark.parametrize("size", [(720, 1280), (1080, 1920)])
def test_hard_motion_vs_cv2(ofc, cv2, monkeypatch, field, size):
    from opticalflowclustering_b200.synthetic import true_flow
    H, W = size
    gray, truth = hard_clip(cv2, field, 3, H, W, seed=H + len(field))
    share = unshared_tap_share(truth)
    gentle = unshared_tap_share(true_flow(H, W).numpy())
    print(f"\n{field} {W}x{H}: rows requesting their own upper taps {share:.2%} (synthetic_clip: {gentle:.2%})")
    if field in ("rotation", "boundaries"):
        assert share >= 0.05, share
    g = torch.from_numpy(gray).cuda()
    plan, flow = _flow_share(monkeypatch, W, H, g, "1")
    _, flow0 = _flow_share(monkeypatch, W, H, g, "0")
    assert torch.equal(flow, flow0)
    flow = flow.cpu().numpy()
    lost = field in ("rotation", "expansion")
    for p in range(2):          # an affine field about the centre moves every pair alike: pair 1 has pair 0's true flow
        _parity(cv2, f"{field} {W}x{H}", plan, flow[p], gray, p, truth=truth if lost else None)


def test_rotation_33_frame_chunk_vs_cv2(ofc, cv2, monkeypatch):
    """a 32-pair 1080p chunk of the rotation field (rotated and zoomed back and forth): sharing on == off over the whole
    chunk, and the first, a middle and the last forward pair against cv2"""
    H, W, T = 1080, 1920, 33
    gray, truth = hard_clip(cv2, "rotation", T, H, W, seed=7, alternate=True)
    g = torch.from_numpy(gray).cuda()
    plan, flow = _flow_share(monkeypatch, W, H, g, "1")
    _, flow0 = _flow_share(monkeypatch, W, H, g, "0")
    assert torch.equal(flow, flow0)
    for p in (0, 16, T - 3):    # even pairs move forward, like pair 0
        _parity(cv2, f"rotation chunk {W}x{H}", plan, flow[p].cpu().numpy(), gray, p, truth=truth)


# ---- (d) ragged strip layouts at production widths --------------------------------------------------------------------
@pytest.mark.parametrize("size", [(768, 1366), (1440, 2560), (540, 960), (289, 513)])
def test_ragged_widths_vs_cv2(ofc, cv2, size):
    """widths that are not a whole number of 240-column strips (513: the narrowest that walks; its last strip is 33
    columns)"""
    from opticalflowclustering_b200.flow import FarnebackPlan
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W = size
    g = _gray(synthetic_clip(3, H, W, seed=W, device="cuda"))
    plan = FarnebackPlan(W, H, max_frames=3)
    flow = plan.sequence(g).cpu().numpy()
    gray = g.cpu().numpy()
    for p in range(2):
        _parity(cv2, f"{W}x{H}", plan, flow[p], gray, p)
