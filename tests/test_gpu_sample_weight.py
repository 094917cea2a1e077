"""Frequency weights (`sample_weight`) on the device: the weighted K4 / K2 / post-pass kernels against the unweighted
ones, repeated rows, the oracle and themselves."""
import numpy as np
import pytest

import _datasets
import _weighted_oracle as WO
from oracle import som_oracle as O

pytestmark = pytest.mark.gpu

GAP = 1e-6


def engine(**kw):
    from dbgsom_b200.engine import DeviceEngine

    return DeviceEngine(**kw)


def run_epochs(X, m_side, n_epochs, weight=None, y=None, n_classes=0, entropy=False, rows=None, backend="tensor",
               start=None):
    """Epochs of one engine from a fixed start; returns (stats, [(W, error, counts, change, part, winners)])."""
    from dbgsom_b200.topology import MapTopology

    gx, gy = m_side
    m = gx * gy
    e = engine(bmu_backend=backend)
    stats = e.load_data(X, y, n_classes, sample_weight=weight) if weight is not None else e.load_data(X, y, n_classes)
    if start is not None:
        e.set_map(start)
    else:
        e.init_map_from_rows(rows, capacity=m)
    e.set_hops_from_topology(MapTopology.full_grid(gx, gy))
    outs = []
    for ep in range(n_epochs):
        W0 = e.weights()
        r = e.epoch(max(2.0, 0.1 * gx) - 0.3 * ep, True, entropy)
        part = e.part[: m * e.ldx + 3 * m].cpu().numpy()
        outs.append(dict(W0=W0, W=e.weights(), error=r["error"], counts=r["counts"], change=r["change"], part=part,
                         winners=e.last_winners_host()))
    e.close()
    return stats, outs


SHAPES = {
    "selective": (300_000, 64, 32, 32),   # D <= 256, M >= 1024: the second epoch runs the selective search
    "wide_teams": (20_000, 768, 8, 8),    # D > 512: teams of several warps in K2
    "tiny": (5, 8, 2, 2),                 # fewer samples than K2 has teams
}


@pytest.mark.parametrize("shape", list(SHAPES), ids=list(SHAPES))
def test_weight_two_equals_unweighted_bitwise(shape):
    """w = 2 doubles every sum exactly: total variance, prototypes and change are the unweighted ones bit for bit,
    counts and E exactly twice theirs."""
    n, d, gx, gy = SHAPES[shape]
    X = _datasets.gmm(n, d, 16, 7)
    rows = np.random.default_rng(3).choice(n, gx * gy, replace=n < gx * gy)
    s0, a = run_epochs(X, (gx, gy), 2, rows=rows)
    s1, b = run_epochs(X, (gx, gy), 2, weight=np.full(n, 2.0), rows=rows)
    assert s0["total_variance"] == s1["total_variance"]
    for u, w in zip(a, b):
        np.testing.assert_array_equal(u["W"], w["W"])
        assert u["change"] == w["change"]
        np.testing.assert_array_equal(2.0 * u["counts"], w["counts"])
        np.testing.assert_array_equal(2.0 * u["error"], w["error"])
        np.testing.assert_array_equal(u["winners"], w["winners"])


def test_integer_weights_equal_repeated_rows():
    n, d, side = 20_000, 32, 8
    X = _datasets.gmm(n, d, 16, 11)
    w = np.random.default_rng(5).integers(1, 5, n).astype(np.float64)
    X_rep = np.repeat(X, w.astype(np.int64), axis=0)
    start = X[np.random.default_rng(6).choice(n, side * side, replace=False)].astype(np.float64)
    s_w, a = run_epochs(X, (side, side), 1, weight=w, start=start)
    s_r, b = run_epochs(X_rep, (side, side), 1, start=start)
    assert s_w["total_variance"] == pytest.approx(s_r["total_variance"], rel=1e-12)
    ra, rb = a[0], b[0]
    gap = O.relative_gap(X.astype(np.float64), start)
    rep_win = rb["winners"][np.cumsum(w.astype(np.int64)) - 1]
    assert not np.any((ra["winners"] != rep_win) & (gap >= GAP))
    assert np.array_equal(ra["winners"], rep_win), "a near-tie went another way: the sums below would not match"
    np.testing.assert_array_equal(ra["counts"], rb["counts"])
    np.testing.assert_allclose(ra["part"], rb["part"], rtol=1e-12, atol=1e-12 * np.abs(rb["part"]).max())
    np.testing.assert_allclose(ra["W"], rb["W"], rtol=1e-12, atol=1e-12 * np.abs(rb["W"]).max())


@pytest.mark.parametrize("backend", ["simt", "tensor"])
def test_fractional_weights_match_the_weighted_oracle(backend):
    n, d, side = 30_000, 48, 8
    X = _datasets.gmm(n, d, 16, 13)
    rng = np.random.default_rng(7)
    w = rng.uniform(0.1, 3.0, n)
    w[rng.random(n) < 0.1] = 0.0
    start = X[np.flatnonzero(w > 0)[:side * side]].astype(np.float64)
    stats, outs = run_epochs(X, (side, side), 1, weight=w, start=start, backend=backend)
    r = outs[0]
    X64 = X.astype(np.float64)
    assert stats["total_variance"] == pytest.approx(WO.total_variance(X64, w), rel=1e-12)
    _, own, gap = O.bmu_with_gap(X64, start)
    strict = gap >= GAP
    assert strict.mean() > 0.99
    assert not np.any((r["winners"] != own) & strict)
    hop = O.hop_matrix_grid(side, side)
    ref = WO.epoch_step(X64, start, hop, max(2.0, 0.1 * side), stats["total_variance"], pack=True,
                       winners=r["winners"], freq_weight=w)
    np.testing.assert_allclose(r["counts"], ref["n"], rtol=1e-12)
    np.testing.assert_allclose(r["error"], ref["E"], rtol=1e-5, atol=1e-6)
    fin = np.isfinite(ref["W_new"])
    assert np.array_equal(np.isfinite(r["W"]), fin)
    assert np.abs(r["W"][fin] - ref["W_new"][fin]).max() / np.abs(ref["W_new"][fin]).max() < 1e-5
    assert r["change"] == pytest.approx(ref["change"], rel=1e-5)


@pytest.mark.parametrize("entropy", [False, True], ids=["qe", "entropy"])
@pytest.mark.parametrize("n,d,gx,gy", [
    (300_000, 64, 16, 16),
    (20_000, 768, 8, 8),
    (60_000, 16, 100, 100),
    (5, 8, 2, 2),
], ids=["selective", "wide_teams", "large_map", "tiny"])
def test_weighted_epochs_repeat_bit_for_bit(n, d, gx, gy, entropy):
    X, y = _datasets.gmm(n, d, 16, 7), np.arange(n) % 5
    rng = np.random.default_rng(9)
    w = rng.uniform(0.0, 2.0, n)
    w[rng.random(n) < 0.1] = 0.0
    w[: min(n, 4)] = 1.0
    rows = np.random.default_rng(3).choice(n, gx * gy, replace=n < gx * gy)
    runs = [run_epochs(X, (gx, gy), 4, weight=w, y=y if entropy else None, n_classes=5 if entropy else 0,
                       entropy=entropy, rows=rows) for _ in range(2)]
    assert runs[0][0]["total_variance"] == runs[1][0]["total_variance"]
    for a, b in zip(runs[0][1], runs[1][1]):
        for key in ("W", "error", "counts", "part"):
            np.testing.assert_array_equal(a[key], b[key])
        assert a["change"] == b["change"]


def test_weighted_post_passes_match_bincount():
    import torch

    from dbgsom_b200 import _native as nat

    lib = nat.load()
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(1)
    n, m, c = 200_003, 300, 7
    idx = rng.integers(0, m, (n, 2)).astype(np.int32)
    dist = rng.uniform(0.0, 3.0, (n, 2))
    pos = rng.integers(0, 20, (m, 2)).astype(np.int32)
    labels = rng.integers(0, c, n).astype(np.int32)
    w = rng.uniform(0.0, 2.0, n)
    w[rng.random(n) < 0.2] = 0.0
    t = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in
         dict(idx=idx, dist=dist, pos=pos, labels=labels, w=w, idx0=idx[:, 0].copy()).items()}
    stream = torch.cuda.current_stream(dev).cuda_stream
    bw = 0.7
    out = torch.empty(2 + 2 * m, dtype=torch.float64, device=dev)
    nat.check(lib.dbgsom_node_stats_weighted(t["idx"].data_ptr(), 2, t["dist"].data_ptr(), 2, n, t["pos"].data_ptr(), m,
                                             bw, t["w"].data_ptr(), out.data_ptr(), stream), "node_stats_weighted")
    o = out.cpu().numpy()
    sep = pos[idx[:, 0]] - pos[idx[:, 1]]
    far = (sep * sep).sum(axis=1) > 2
    d0 = dist[:, 0]
    assert o[0] == pytest.approx(w[far].sum(), rel=1e-12)
    assert o[1] == pytest.approx((w * d0).sum(), rel=1e-12)
    np.testing.assert_allclose(o[2 : 2 + m], np.bincount(idx[:, 0], weights=w, minlength=m), rtol=1e-12)
    kern = np.exp(-(d0 * d0) / (2 * bw * bw)) / (bw * np.sqrt(2 * np.pi))
    np.testing.assert_allclose(o[2 + m :], np.bincount(idx[:, 0], weights=w * kern, minlength=m), rtol=1e-12)

    ws = torch.empty(lib.dbgsom_label_hist_weighted_workspace_bytes(n, m), dtype=torch.uint8, device=dev)
    results = []
    for _ in range(2):
        counts = torch.empty((m, c), dtype=torch.float64, device=dev)
        first = torch.empty((m, c), dtype=torch.int64, device=dev)
        nat.check(lib.dbgsom_label_hist_weighted(t["idx0"].data_ptr(), t["labels"].data_ptr(), t["w"].data_ptr(), n, 10,
                                                 m, c, counts.data_ptr(), first.data_ptr(), ws.data_ptr(), ws.numel(),
                                                 stream), "label_hist_weighted")
        results.append((counts.cpu().numpy(), first.cpu().numpy()))
    flat = idx[:, 0].astype(np.int64) * c + labels
    np.testing.assert_allclose(results[0][0].ravel(), np.bincount(flat, weights=w, minlength=m * c), rtol=1e-12)
    ref_first = np.full(m * c, np.iinfo(np.int64).max)
    pos_rows = np.flatnonzero(w > 0)
    np.minimum.at(ref_first, flat[pos_rows], pos_rows + 10)
    np.testing.assert_array_equal(results[0][1].ravel(), ref_first)
    np.testing.assert_array_equal(results[0][0], results[1][0])  # per-winner sums in a fixed order


def _fit(cls, X, y=None, w=None, **kw):
    est = cls(random_state=0, n_iter=40, **kw)
    est.fit(X, y, sample_weight=w) if w is not None else est.fit(X, y)
    return est


@pytest.mark.parametrize("kind", ["vq", "clf_entropy"])
def test_whole_fits_ones_and_mask(kind):
    from dbgsom_b200 import SomClassifier, SomVQ

    X, y = _datasets.load("digits")
    cls, kw = (SomVQ, {}) if kind == "vq" else (SomClassifier, {"growth_criterion": "entropy"})
    yy = None if kind == "vq" else y
    base = _fit(cls, X, yy, **kw)
    ones = _fit(cls, X, yy, np.ones(len(X)), **kw)
    np.testing.assert_array_equal(ones.weights_, base.weights_)
    assert list(ones.neurons_) == list(base.neurons_) and ones.n_iter_ == base.n_iter_
    assert ones.topographic_error_ == base.topographic_error_
    np.testing.assert_array_equal(ones._extract_values_from_graph("hit_count"), base._extract_values_from_graph("hit_count"))
    assert ones.quantization_error_ == pytest.approx(base.quantization_error_, rel=1e-12)
    np.testing.assert_allclose(ones._extract_values_from_graph("density"), base._extract_values_from_graph("density"),
                               rtol=1e-12)
    if kind == "vq":
        np.testing.assert_array_equal(ones.labels_, base.labels_)
    else:
        np.testing.assert_array_equal(ones._extract_values_from_graph("label"), base._extract_values_from_graph("label"))

    keep = np.random.default_rng(4).random(len(X)) < 0.7
    masked = _fit(cls, X, yy, keep.astype(np.float64), **kw)
    sub = _fit(cls, X[keep], None if yy is None else yy[keep], **kw)
    assert len(masked.neurons_) == len(sub.neurons_) and masked.n_iter_ == sub.n_iter_
    np.testing.assert_allclose(masked.weights_, sub.weights_, rtol=1e-9, atol=1e-9)
    assert masked.quantization_error_ == pytest.approx(sub.quantization_error_, rel=1e-9)
    assert masked.topographic_error_ == pytest.approx(sub.topographic_error_, rel=1e-9, abs=1e-12)
    if kind == "vq":
        np.testing.assert_array_equal(masked.labels_[keep], sub.labels_)


def test_two_nccl_ranks_with_weighted_shards_equal_one_gpu(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import os
    import socket

    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_nccl_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    from dbgsom_b200 import SomVQ

    X, _ = _datasets.load("digits")
    w = _weights_for(len(X))
    one = _fit(SomVQ, X, None, w)
    r0 = np.load(os.path.join(tmp_path, "rank0.npz"))
    np.testing.assert_array_equal(r0["neurons"], np.array(one.neurons_))
    np.testing.assert_allclose(r0["weights"], one.weights_, rtol=1e-9, atol=1e-9)
    assert float(r0["qe"]) == pytest.approx(one.quantization_error_, rel=1e-9)


def _weights_for(n):
    w = np.random.default_rng(8).uniform(0.0, 2.0, n)
    w[::7] = 0.0
    return w


def _nccl_worker(rank, world, port, out_dir):
    import os
    import sys

    here = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(here), here]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch
    import torch.distributed as dist

    import _datasets as ds
    from dbgsom_b200 import SomVQ

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        X, _ = ds.load("digits")
        w = _weights_for(len(X))
        lo, hi = rank * len(X) // world, (rank + 1) * len(X) // world
        est = SomVQ(random_state=0, n_iter=40, distributed=True, device=f"cuda:{rank}")
        est.fit(X[lo:hi], sample_weight=w[lo:hi])
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), neurons=np.array(est.neurons_), weights=est.weights_,
                 qe=est.quantization_error_)
    finally:
        dist.destroy_process_group()
