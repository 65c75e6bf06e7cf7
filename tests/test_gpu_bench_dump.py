"""bench.py --dump-outputs writes what its last timed step computed: the rows, magnitudes, flow and visualisation of
one ClipPipeline run over that step's chunk of the benchmark's seeded clip, bit for bit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import ROOT

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_timed_step(tmp_path):
    import bench
    from opticalflowclustering_b200.pipeline import ClipPipeline
    from opticalflowclustering_b200.synthetic import synthetic_clip
    H, W, F, T, steps, warmup = 720, 1280, 5, 12, 3, 1
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", "720p", "--chunk", str(F),
                        "--clip-frames", str(T), "--steps", str(steps), "--warmup", str(warmup), "--lanes", "2",
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    P = F - 1
    first = ((warmup + steps - 1) * P) % (T - F + 1)          # the chunk of the last timed step
    assert res["steps"] == steps and res["dump_outputs"]["frames"] == [first, first + F]

    clip = synthetic_clip(T, H, W, seed=0, device="cuda")
    pipe = ClipPipeline(W, H, chunk_frames=F, rows=14, cols=25)
    pipe.run_chunk(clip[first:first + F])
    idx = bench.dump_sample_index(P * H * W).cuda()
    assert idx.numel() == bench.DUMP_SAMPLE_PX
    want = {"avg_hue": pipe.avg_hue, "km_hue": pipe.km_hue, "km_centre": pipe.km_centre, "avg_bgr": pipe.avg_bgr,
            "mean_magnitude": pipe.mag_sum.cpu() / float(H * W),
            "flow_sample": pipe.flow.reshape(-1, 2)[idx], "viz_sample": pipe.viz.reshape(-1, 3)[idx]}
    assert sorted(res["dump_outputs"]["arrays"]) == sorted(want)
    total = 0
    for name, w in want.items():
        got = np.load(out / (name + ".npy"))
        total += got.nbytes
        w = w.cpu().numpy()
        assert got.dtype == (np.float64 if w.dtype == np.float64 else np.float32), name
        assert got.shape == w.shape and np.array_equal(got, w), name
    assert total <= 64 << 20
