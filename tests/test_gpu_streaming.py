"""Streamed fits: samples pass through the device in row chunks every epoch (dbgsom_b200/streaming.py).

Streamed sums are taken per chunk and added in chunk order, so they agree with the resident fit to summation order
and repeat bit for bit with the same chunking; winners are the float64 winners outside the 1e-6 near-tie gate
either way."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _datasets
import test_gpu_parity as P
from conftest import golden_files
from oracle import som_oracle as O

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
TRAJ_FILES = golden_files("traj")


def engine(stream_rows=0, **kw):
    from dbgsom_b200.engine import DeviceEngine

    e = DeviceEngine(**kw)
    e.stream_rows = stream_rows
    return e


@pytest.fixture
def record_engines(monkeypatch):
    """(streaming, number of chunks) of every engine a fit closes."""
    from dbgsom_b200.engine import DeviceEngine

    seen = []
    close = DeviceEngine.close

    def rec(self):
        if getattr(self, "N", 0):
            seen.append((self.streaming, len(self.chunks) if self.chunks else 1))
        close(self)

    monkeypatch.setattr(DeviceEngine, "close", rec)
    return seen


# ------------------------------------------------------------------------------------------ (1) oracle trajectory
@pytest.mark.parametrize("shape,chunk", [((200_000, 256, 64), 76_800), ((19_200, 4096, 64), 5_120)],
                         ids=["c3-shape-3-chunks", "c5-width-4-chunks"])
def test_streamed_epochs_match_the_oracle_over_a_trajectory(shape, chunk):
    from bench import sigma_at
    from dbgsom_b200.topology import MapTopology

    n, d, side = shape
    m = side * side
    X = _datasets.gmm(n, d, 64, 3)
    W0 = X[np.random.default_rng(0).choice(n, m, replace=False)].astype(np.float64)
    hop = O.hop_matrix_grid(side, side)
    e = engine(chunk, bmu_backend="tensor")
    stats = e.load_data(X, None, 0)
    assert e.streaming and len(e.chunks) == -(-n // chunk)
    e.set_map(W0)
    e.set_hops_from_topology(MapTopology.full_grid(side, side))
    n_epochs, compared = 6, 0
    for epoch in range(n_epochs):
        W = e.weights()
        sigma = sigma_at(epoch, m)
        r = e.epoch(sigma, True, False)
        r["winners"] = e.last_winners_host()
        n_strict, _, _ = P.assert_epoch_parity(r, e.weights(), X, W, hop, sigma, stats["total_variance"],
                                               min_strict=0.85 if d <= 256 else 0.2)
        compared += n_strict
        if epoch == 0 and d <= 256:
            st = e.bmu_stats_host()
            assert st["classic_searches"] == len(e.chunks) and st["selective_searches"] == 0
    st = e.bmu_stats_host()
    assert st["fp32_reruns"] == 0
    if d <= 256:
        # every chunk's search is selective once the chunk's samples are sorted by winner
        assert st["selective_searches"] == len(e.chunks) * (n_epochs - 1) and st["classic_searches"] == 0
    e.close()
    assert compared > (0.9 if d <= 256 else 0.3) * n_epochs * n


# ------------------------------------------------------------------------------------------ (2) streamed == resident
@pytest.mark.parametrize("mode", ["unweighted", "weighted", "entropy"])
def test_streamed_epoch_equals_resident_epoch(mode):
    from dbgsom_b200.topology import MapTopology

    n, d, side = 90_000, 64, 24
    X, y = _datasets.gmm(n, d, 12, 8, return_labels=True)
    y = y % 5
    w = np.random.default_rng(2).integers(0, 4, n).astype(np.float64) if mode == "weighted" else None
    W0 = X[np.random.default_rng(1).choice(n, side * side, replace=False)].astype(np.float64)
    out = []
    for rows in (0, 20_000):
        e = engine(rows, bmu_backend="tensor")
        if mode == "weighted":
            e.load_data(X, None, 0, sample_weight=w)
        else:
            e.load_data(X, y if mode == "entropy" else None, 5 if mode == "entropy" else 0)
        assert e.streaming == (rows > 0)
        e.set_map(W0)
        e.set_hops_from_topology(MapTopology.full_grid(side, side))
        r = e.epoch(2.0, True, mode == "entropy")
        out.append((r, e.last_winners_host(), e.weights(), e.total_variance))
        e.close()
    (ra, wa, Wa, va), (rb, wb, Wb, vb) = out
    assert va == pytest.approx(vb, rel=1e-12)
    _, _, gap = O.bmu_with_gap(X.astype(np.float64), W0)
    strict = gap >= P.GAP
    np.testing.assert_array_equal(wa[strict], wb[strict])
    np.testing.assert_array_equal(ra["counts"], rb["counts"])
    np.testing.assert_allclose(rb["error"], ra["error"], rtol=1e-12, atol=0 if mode != "entropy" else 1e-15)
    np.testing.assert_allclose(Wb, Wa, rtol=1e-12, atol=1e-12 * np.abs(Wa).max())
    assert rb["change"] == pytest.approx(ra["change"], rel=1e-12)


# ------------------------------------------------------------------------------------------ (3) repeatability
@pytest.mark.parametrize("n,d,gx,gy,chunk", [(150_000, 64, 16, 16, 51_200), (20_000, 768, 8, 8, 6_144)],
                         ids=["selective", "wide_teams"])
def test_streamed_epochs_repeat_bit_for_bit(n, d, gx, gy, chunk):
    from dbgsom_b200.topology import MapTopology

    X = _datasets.gmm(n, d, 16, 7)
    m = gx * gy
    runs = []
    for _ in range(2):
        e = engine(chunk, bmu_backend="tensor")
        stats = e.load_data(X, None, 0)
        e.init_map_from_rows(np.random.default_rng(3).choice(n, m, replace=n < m), capacity=m)
        e.set_hops_from_topology(MapTopology.full_grid(gx, gy))
        outs = []
        for ep in range(4):
            r = e.epoch(max(2.0, 0.1 * gx) - 0.3 * ep, True, False)
            outs.append((e.weights(), r["error"], r["counts"], r["change"]))
        win = e.last_winners_host()
        assert (win >= 0).all()
        # every chunk's saved order lists its samples grouped by winner, ascending sample index within a winner
        perm = e.row_perm.cpu().numpy()
        for c0, c1 in e.chunks:
            np.testing.assert_array_equal(perm[c0:c1], np.argsort(win[c0:c1], kind="stable"))
        runs.append((stats["total_variance"], outs))
        e.close()
    assert runs[0][0] == runs[1][0]
    for a, b in zip(runs[0][1], runs[1][1]):
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)


# ------------------------------------------------------------------------------------------ (4) whole fits
@pytest.mark.parametrize("path", TRAJ_FILES, ids=[os.path.basename(p)[5:-4] for p in TRAJ_FILES])
def test_streamed_fit_matches_reference_fixture(path, monkeypatch, record_engines):
    monkeypatch.setenv("DBGSOM_STREAM_ROWS", "512")
    P.test_fit_matches_reference_fixture(path)
    fit = record_engines[0]
    assert fit[0] and fit[1] >= 2, fit  # the fit streamed, in several chunks


# ------------------------------------------------------------------------------------------ (5) weighted classifier
@pytest.mark.parametrize("data", ["rings3d", "blobs2d"])
def test_weighted_classifier_streamed_equals_resident(data, monkeypatch):
    from dbgsom_b200 import SomClassifier

    X, y = _datasets.load(data)
    w = np.random.default_rng(4).integers(1, 4, X.shape[0]).astype(np.float64)
    fits = []
    for rows in ("0", "256"):
        monkeypatch.setenv("DBGSOM_STREAM_ROWS", rows)
        est = SomClassifier(random_state=2, n_iter=40, max_neurons=30).fit(X, y, sample_weight=w)
        fits.append(est)
    a, b = fits
    np.testing.assert_array_equal(a.classes_, b.classes_)
    assert a.neurons_ == b.neurons_ and a.n_iter_ == b.n_iter_
    _, _, gap = O.bmu_with_gap(X, a.weights_)
    near = int((gap < 1e-9).sum())
    # the class counts per neuron: its majority label and class probabilities
    la, lb = a._extract_values_from_graph("label"), b._extract_values_from_graph("label")
    pa, pb = np.stack(a._extract_values_from_graph("probabilities")), np.stack(b._extract_values_from_graph("probabilities"))
    if near == 0:
        np.testing.assert_array_equal(la, lb)
        np.testing.assert_allclose(pb, pa, rtol=1e-9, atol=1e-12)
    else:
        assert (la != lb).sum() <= near
    ha, hb = a._extract_values_from_graph("hit_count"), b._extract_values_from_graph("hit_count")
    assert np.abs(ha - hb).sum() <= 2 * near * w.max()
    if near == 0:
        np.testing.assert_array_equal(ha, hb)
    np.testing.assert_allclose(b.weights_, a.weights_, rtol=1e-9, atol=1e-9 * np.abs(a.weights_).max())
    assert b.quantization_error_ == pytest.approx(a.quantization_error_, rel=1e-9)
    assert b.topographic_error_ == pytest.approx(a.topographic_error_, rel=1e-9, abs=1e-12)
    for attr in ("density", "average_distance"):
        np.testing.assert_allclose(b._extract_values_from_graph(attr), a._extract_values_from_graph(attr), rtol=1e-9,
                                   atol=1e-12)
    np.testing.assert_array_equal(a.predict(X), b.predict(X))


# ------------------------------------------------------------------------------------------ (6) chunked predict
@pytest.mark.parametrize("n,d,m,backend", [(100_000, 128, 400, "auto"), (5_000, 20, 30, "auto"),
                                           (30_000, 64, 256, "tensor")])
def test_predict_in_chunks_is_bit_identical(n, d, m, backend):
    X = _datasets.gmm(n, d, 16, 9)
    W = X[np.random.default_rng(5).choice(n, m, replace=False)].astype(np.float64) + 0.01
    out = []
    for rows in (0, 3_000):
        e = engine(rows, bmu_backend=backend)
        out.append(e.bmu(X, W, 1))
        e.close()
    np.testing.assert_array_equal(out[0][1], out[1][1])
    np.testing.assert_array_equal(out[0][0], out[1][0])


# ------------------------------------------------------------------------------------------ (7) automatic choice
def test_fit_streams_when_device_memory_is_short(monkeypatch, record_engines):
    import torch

    from dbgsom_b200 import SomVQ, streaming
    from dbgsom_b200 import _native as nat

    path = [p for p in TRAJ_FILES if "digits_vq" in p][0]
    P.test_fit_matches_reference_fixture(path)
    assert record_engines[0] == (False, 1)  # real free memory: resident
    record_engines.clear()

    g = np.load(path, allow_pickle=False)
    meta = json.loads(str(g["meta"]))
    X, _ = _datasets.load(meta["data"])
    lib = nat.load()
    need = streaming.resident_bytes(X.shape[0], X.shape[1], SomVQ(**meta["params"])._capacity_hint(), 0, False,
                                    lib.dbgsom_accumulate_workspace_bytes, lib.dbgsom_bmu_workspace_bytes)
    torch.cuda.empty_cache()
    total = torch.cuda.mem_get_info()[1]
    cached = torch.cuda.memory_reserved() - torch.cuda.memory_allocated()
    short = streaming.free_margin(total) + need - cached - 4096
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (short, total))
    P.test_fit_matches_reference_fixture(path)
    assert record_engines[0][0], record_engines[0]


# ------------------------------------------------------------------------------------------ (8) two ranks
def test_two_streaming_ranks_equal_one_resident_gpu():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29741", os.path.join(HERE, "_multirank_stream_worker.py")]
    res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MULTIRANK_STREAM_OK" in res.stdout
