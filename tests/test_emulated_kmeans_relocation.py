"""Empty clusters on CPU: the oracle and the .cu sources under the emulation (tests/emu) against scikit-learn 1.9.0 on fits
in which clusters go empty (tests/golden/make_relocation_golden.py).  sklearn lists the empty clusters once, so a cluster
that a relocation move empties stays empty; and its in-place _average_centers gives an empty cluster below the heaviest
one that cluster's centred sum, not its mean.  Every relocation form is driven here: the single-CTA kernel, the
two-kernel form (unweighted and weighted, single fits, shared-row and per-problem batches), both per-cell kernels, and the
row-sharded merges of a world-2 gloo fit.  The `-m gpu` twins are in tests/test_gpu_kmeans_relocation.py."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from tests.conftest import GOLDEN

E = pytest.importorskip("tests.emu.emu_lib")
from opticalflowclustering_b200 import kmeans as km    # noqa: E402
from oracle import kmeans_np as K                       # noqa: E402

sys.path.insert(0, GOLDEN)
import make_relocation_golden as RG                      # noqa: E402
import make_weighted_golden as WG                        # noqa: E402

MAX_ITERS = RG.MAX_ITERS
PROBE_KEYS = [f"probe_{p}_{f}" for p, f in RG.PROBE_FORMS]
#: the generated cases small enough for the emulation (one fiber per CUDA thread)
SMALL_GEN = ["u8_d4_k8", "u8_d4_k3_w_below", "f64_d42_k6_below", "f32_d42_k6_w_below"]


@pytest.fixture(scope="module")
def Z():
    return np.load(os.path.join(GOLDEN, "kmeans_sklearn_relocation.npz"))


@pytest.fixture(scope="module")
def L():
    E.build()
    km._use_test_library(E.lib())
    yield E.lib()
    km._use_test_library(None)


def _case(key):
    if key.startswith("probe_"):
        p, f = key[len("probe_"):].rsplit("_", 1)
        return RG.probe_form(p, f)
    return RG.gen_case(key[len("gen_"):])


# ---- the oracle -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("key", PROBE_KEYS + [f"gen_{g}" for g in RG.GEN_CASES])
def test_oracle_reproduces_relocation_goldens(Z, key):
    X, init, w = _case(key)
    for m in MAX_ITERS:
        RG.check_fit(f"oracle {key} max_iter={m}", K.kmeans_fit(X, init, max_iter=m, sample_weight=w),
                     RG.golden_fit(Z, key, m), X)


@pytest.mark.parametrize("name", list(WG.WEIGHTED_CASES))
def test_oracle_reproduces_weighted_goldens(name):
    """the weighted oracle against sklearn's kept start of every case of kmeans_sklearn_weighted.npz"""
    z = np.load(os.path.join(GOLDEN, "kmeans_sklearn_weighted.npz"))
    X, w = WG.weighted_case(name)
    seeds = WG.PROBE_INIT_ROWS if name.startswith("probe") else z[name + "_seed_idx"][int(z[name + "_best"])]
    init = X[seeds].astype(np.float64)
    ref = (z[name + "_labels"], z[name + "_centers"], float(z[name + "_inertia"]), int(z[name + "_niter"]))
    RG.check_fit(f"oracle {name}", K.kmeans_fit(X, init, sample_weight=w), ref, X)


def test_oracle_probes_show_both_rules(Z):
    """what the probes are for, stated on sklearn's own results: the cluster a move empties stays empty, and an empty
    cluster below the heaviest takes its centred sum"""
    lab, cen, _, _ = RG.golden_fit(Z, "probe_cascade_f64", 1)
    assert (lab == [1, 1, 1, 0]).all() and np.allclose(cen[:, 0], [60, 4 / 3, 4 / 3])
    assert RG.golden_fit(Z, "probe_cascade_f64", 300)[3] == 3
    assert np.allclose(RG.golden_fit(Z, "probe_in_place_f64", 1)[1][:, 0], [60, -28, 4 / 3])
    assert np.allclose(RG.golden_fit(Z, "probe_zero_weight_move_f64", 1)[1][:, 0], [-8.2, 2.5, 0.5])


# ---- kmeans.lloyd under the emulation -------------------------------------------------------------------------------
@pytest.mark.parametrize("key", PROBE_KEYS + [f"gen_{g}" for g in SMALL_GEN])
def test_emulated_lloyd_reproduces_sklearn(L, Z, key):
    X, init, w = _case(key)
    for m in MAX_ITERS:
        RG.check_fit(f"lloyd {key} max_iter={m}", km.lloyd(X, init, max_iter=m, sample_weight=w), RG.golden_fit(Z, key, m), X)


def test_emulated_shared_row_batch(L, Z):
    """X [n, d] with init [R, k, d]: the start that hits the relocation reproduces sklearn, the other its oracle fit"""
    X, init, w = RG.gen_case("u8_d4_k8")
    rng = np.random.default_rng(5)
    other = X[rng.choice(X.shape[0], init.shape[0], replace=False)].astype(np.float64)
    got = km.lloyd(X, np.stack([other, init]))
    RG.check_fit("shared batch, start 1", [t[1] for t in got], RG.golden_fit(Z, "gen_u8_d4_k8", 300), X)
    RG.check_fit("shared batch, start 0", [t[0] for t in got], K.kmeans_fit(X, other), X)


@pytest.mark.parametrize("form", ["f64", "u8"])
def test_emulated_per_problem_weights(L, form):
    """[B, n] weights that differ per problem (and per-problem init): problem 0 hits the cascade, problem 1 no empty
    cluster, problem 2 moves a row of weight 0 -- each against the weighted oracle"""
    X, init, w = RG.probe_form("cascade", "w")
    if form == "u8":
        X = np.concatenate([X, np.zeros((X.shape[0], 1)), np.full((X.shape[0], 1), 255.0)], axis=1).astype(np.uint8)
        init = np.concatenate([init, np.zeros((3, 1)), np.full((3, 1), 255.0)], axis=1)
    inits = np.stack([init, X[[0, 2, 5]].astype(np.float64), init])
    ws = np.stack([w, np.linspace(0.5, 3.0, X.shape[0]), np.where(np.arange(X.shape[0]) == 3, 0.0, w + 1.0)])
    got = km.lloyd(np.stack([X] * 3), inits, sample_weight=ws, max_iter=1)
    for b in range(3):
        RG.check_fit(f"per-problem weights {form}, problem {b}", [t[b] for t in got],
                     K.kmeans_fit(X, inits[b], max_iter=1, sample_weight=ws[b]), X)
    assert got[1][2][0, 0] < -1.0         # problem 2: the row of weight 0 left cluster 0 empty -> the sum of cluster 1


# ---- the per-cell kernels -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fast", ["1", "0"])
def test_emulated_cells_reproduce_sklearn(L, Z, monkeypatch, fast):
    """lloyd_cells, fast per-cell kernel (OFC_CELLS_FAST=1) and kmeans_cells_kernel (0): the unweighted uint8 probes as
    cells, beside a cell of the same size without an empty cluster; and the generated uint8 case"""
    monkeypatch.setenv("OFC_CELLS_FAST", fast)
    for p in ("cascade", "in_place"):
        X, init, _ = RG.probe_form(p, "u8")
        quiet = X.copy()
        quiet[:, 0] = [10, 40, 70, 100, 130][:X.shape[0]]
        q_init = quiet[[0, 1, 2]].astype(np.float64)
        for m in MAX_ITERS:
            lab, cen, inertia, n_iter, _ = km.lloyd_cells(np.stack([X, quiet]), 3, init=np.stack([init, q_init]), max_iter=m)
            RG.check_fit(f"cells fast={fast} {p} max_iter={m}", (lab[0], cen[0], inertia[0], n_iter[0]),
                         RG.golden_fit(Z, f"probe_{p}_u8", m), X)
            RG.check_fit(f"cells fast={fast} quiet cell", (lab[1], cen[1], inertia[1], n_iter[1]),
                         K.kmeans_fit(quiet, q_init, max_iter=m), quiet)
    X, init, _ = RG.gen_case("u8_d4_k8")
    for m in MAX_ITERS:
        got = km.lloyd_cells(X, init.shape[0], init=init, max_iter=m)[:4]
        RG.check_fit(f"cells fast={fast} gen u8_d4_k8 max_iter={m}", got, RG.golden_fit(Z, "gen_u8_d4_k8", m), X)


# ---- the single-CTA relocation kernel, called directly --------------------------------------------------------------
@pytest.mark.parametrize("form", ["f64", "u8"])
def test_emulated_single_cta_relocation(L, form):
    """ofc_kmeans_relocate with scratch = NULL runs kmeans_relocate_kernel: after the cascade probe's first E-step, cluster
    0 takes row 3, and cluster 2 -- emptied by that move -- stays empty (it must not take row 2)"""
    X, init, _ = RG.probe_form("cascade", form)
    Xd = X.astype(np.float64)
    mean = Xd.mean(axis=0)
    cen = np.ascontiguousarray(init - mean)
    labels = K._e_step(Xd - mean, cen).astype(np.int32)
    raw = form == "u8"                                       # uint8 sums stay raw (exact integers)
    rows = Xd if raw else Xd - mean
    sums = np.zeros((3, X.shape[1]))
    np.add.at(sums, labels, rows)
    counts = np.bincount(labels, minlength=3).astype(np.int64)
    assert (counts == [0, 3, 1]).all()
    Xc = np.ascontiguousarray(X)
    dtype = 0 if raw else 2
    p = E._p
    rc = L.ofc_kmeans_relocate(p(Xc), dtype, 1, C.c_int64(X.shape[0]), X.shape[1], 3, p(mean), p(labels), p(cen), p(sums),
                               p(counts), int(raw), C.c_void_p(0), C.c_void_p(0), C.c_void_p(0))
    assert rc == 0
    print("counts after the relocation", counts.tolist())
    assert (counts == [1, 3, 0]).all()
    assert np.allclose(sums[0], rows[3], atol=1e-12) and np.allclose(sums[2], 0.0, atol=1e-12)
    assert np.allclose(sums[1], rows[:3].sum(axis=0), atol=1e-12)


# ---- row-sharded: world-2 gloo --------------------------------------------------------------------------------------
def _gloo_worker(rank, world, port, out_dir, key, host):
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from opticalflowclustering_b200 import kmeans as kmw
    from opticalflowclustering_b200.sharding import shard_range
    from tests.emu import emu_lib as Ew
    sys.path.insert(0, GOLDEN)
    import make_relocation_golden as RGw
    kmw._use_test_library(Ew.lib())
    X, init, _ = (RGw.probe_form("cascade", "u8") if key == "probe_cascade_u8" else RGw.gen_case(key[len("gen_"):]))
    lo, hi = shard_range(len(X), rank, world)
    out = {}
    for m in RGw.MAX_ITERS:
        lab, cen, inertia, n_iter = kmw.lloyd(X[lo:hi], init, max_iter=m, group=dist.group.WORLD, _host_relocation=host)
        out.update({f"labels{m}": lab.numpy(), f"centres{m}": cen.numpy(), f"inertia{m}": float(inertia),
                    f"n_iter{m}": int(n_iter)})
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), lo=lo, hi=hi, **out)
    dist.destroy_process_group()


@pytest.mark.parametrize("host", [False, True], ids=["device_merge", "host_merge"])
@pytest.mark.parametrize("key", ["probe_cascade_u8", "gen_u8_d4_k8"])
def test_sharded_relocation_reproduces_sklearn(Z, tmp_path, key, host):
    """world 2, rows split in two: the outlier lives on one rank, the rows the emptied cluster later takes on the other
    (the probe: row 3 on rank 1, rows 0-1 on rank 0); ofc_kmeans_far_payload + ofc_kmeans_relocate_merge, and the
    host-merged relocation, against sklearn"""
    import torch.multiprocessing as mp
    from tests.test_distributed_gloo import _free_port
    E.build()
    X = _case(key)[0]
    mp.spawn(_gloo_worker, args=(2, _free_port(), str(tmp_path), key, host), nprocs=2, join=True)
    got = [np.load(tmp_path / f"r{r}.npz") for r in range(2)]
    for m in MAX_ITERS:
        lab = np.concatenate([g[f"labels{m}"] for g in got])
        for r, g in enumerate(got):
            RG.check_fit(f"gloo {key} host={host} rank {r} max_iter={m}", (lab, g[f"centres{m}"], g[f"inertia{m}"],
                                                                            g[f"n_iter{m}"]), RG.golden_fit(Z, key, m), X)
