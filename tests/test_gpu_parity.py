"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the reference fixtures.

All tests need a B200 (`-m gpu`).  Tolerances follow BASELINE.json's north star:
  * BMU indices bit-equal to the float64 oracle wherever the oracle's relative gap between best
    and second-best squared distance is >= 1e-6;
  * prototypes within 1e-5 relative (max|dW| / max|W|) per epoch; counts exact; E within 1e-5.
"""
import json
import os

import numpy as np
import pytest

import _datasets
from conftest import golden_files
from oracle import som_oracle as O

pytestmark = pytest.mark.gpu

STEP_FILES = golden_files("step")
TRAJ_FILES = golden_files("traj")
GAP = 1e-6


def engine(**kw):
    from dbgsom_b200.engine import DeviceEngine

    return DeviceEngine(**kw)


def hop_u16(hop):
    out = np.full(hop.shape, 0xFFFF, dtype=np.uint16)
    fin = np.isfinite(hop)
    out[fin] = hop[fin].astype(np.uint16)
    return out


def load_step(path):
    g = np.load(path, allow_pickle=False)
    meta = json.loads(str(g["meta"]))
    X, _ = _datasets.load(meta["data"])
    X = np.ascontiguousarray(X.astype(meta["cast"]))
    return g, meta, X


def assert_bmu_parity(idx, X, W, ref_idx=None):
    """idx [N] from the device; exact match required outside the oracle's near-tie set."""
    gap = O.relative_gap(X, W)
    if ref_idx is None:
        _, ref_idx = O.bmu_expansion(X, W, 1)
    strict = gap >= GAP
    bad = np.flatnonzero((idx != ref_idx) & strict)
    assert bad.size == 0, f"{bad.size} BMU mismatches outside near-ties, first rows {bad[:5]}"
    # inside the near-tie set the device winner must still be (numerically) as close
    loose = np.flatnonzero(idx != ref_idx)
    if loose.size:
        d_dev = np.linalg.norm(X[loose].astype(np.float64) - W[idx[loose]], axis=1)
        d_ref = np.linalg.norm(X[loose].astype(np.float64) - W[ref_idx[loose]], axis=1)
        np.testing.assert_allclose(d_dev, d_ref, rtol=2e-6)
    return int(strict.sum()), int(loose.size)


# ------------------------------------------------------------------------------------------ K4
def test_column_statistics():
    X = _datasets.gmm(30000, 100, 8, 3) * 3.0 + 50.0  # large mean: cancellation check
    e = engine()
    stats = e.load_data(X, None, 0)
    X64 = X.astype(np.float64)
    assert stats["n_samples"] == X.shape[0]
    assert stats["total_variance"] == pytest.approx(np.var(X64, axis=0).sum(), rel=1e-12)
    assert stats["std_norm"] == pytest.approx(np.linalg.norm(np.std(X64, axis=0, ddof=1)), rel=1e-12)
    np.testing.assert_allclose(e.shift.cpu().numpy()[:100], X64.mean(axis=0), rtol=1e-6)
    e.close()


def test_large_offset_data_warns_about_float32_storage():
    """float64 input is rounded to float32 once on upload: data whose offset dwarfs its spread loses digits of the
    spread, and `load_data` says so instead of silently training on quantised samples (ADVICE r1)."""
    X = _datasets.gmm(5000, 16, 4, 3).astype(np.float64) * 1e-2 + 1e4
    e = engine()
    with pytest.warns(RuntimeWarning, match="float32"):
        e.load_data(X, None, 0)
    e.close()


# ------------------------------------------------------------------------------------------ K1
@pytest.mark.parametrize("path", STEP_FILES, ids=[os.path.basename(p)[5:-4] for p in STEP_FILES])
@pytest.mark.parametrize("backend", ["simt", "tensor", "tensor1"])
def test_bmu_matches_reference_fixture(path, backend):
    g, meta, X = load_step(path)
    W = g["W"]
    e = engine(bmu_backend=backend)
    dist, idx = e.bmu(X, W, 1)
    assert idx.shape == (X.shape[0], 1) and idx.dtype == np.int64
    assert_bmu_parity(idx[:, 0], X, W, g["winners"])
    # the reference's GEMM expansion carries ~1e-6 absolute noise on zero distances (sample == prototype)
    np.testing.assert_allclose(dist[:, 0], g["dist"], rtol=1e-6, atol=5e-6)
    dist2, idx2 = e.bmu(X, W, 2)
    gap = O.relative_gap(X, W)
    ok = gap >= GAP
    np.testing.assert_array_equal(idx2[ok, 0], g["winners2"][ok, 0])
    np.testing.assert_allclose(dist2, g["dist2"], rtol=1e-6, atol=5e-6)
    assert (dist2[:, 0] <= dist2[:, 1]).all()
    e.close()


@pytest.mark.parametrize("backend,n_pass_name", [("simt", "fp32"), ("tensor", "3 pass"), ("tensor1", "1 pass")])
@pytest.mark.parametrize("shape", [(20000, 256, 1024), (9000, 128, 4096), (5000, 784, 400), (3000, 1000, 300)])
def test_bmu_large_maps(backend, n_pass_name, shape):
    """Random-row prototypes (benign) and a smooth sheet (many near-ties) at bench-like shapes."""
    n, d, m = shape
    X = _datasets.gmm(n, d, 32, 11)
    rng = np.random.default_rng(5)
    W_rows = X[rng.choice(n, m, replace=False)].astype(np.float64)
    # smooth sheet: heavily smoothed prototypes as after a large-sigma epoch
    side = int(np.sqrt(m))
    H = O.neighborhood(O.hop_matrix_grid(side, side), 4.0)
    W_sheet = (H @ W_rows[: side * side]) / H.sum(axis=1)[:, None]
    e = engine(bmu_backend=backend)
    for name, W in (("rows", W_rows), ("sheet", W_sheet)):
        dist, idx = e.bmu(X, W, 1)
        n_strict, n_loose = assert_bmu_parity(idx[:, 0], X, W)
        assert n_strict > 0.5 * n, name
        d_ref = np.sqrt(np.maximum(O.sqdist_exact(X[:500], W)[np.arange(500), idx[:500, 0]], 0))
        np.testing.assert_allclose(dist[:500, 0], d_ref, rtol=1e-9, atol=1e-9)
    e.close()


def test_bmu_duplicate_prototypes_lowest_index_wins():
    """Exact ties go to the lowest index, like sklearn's heap (sklearn/utils/_heap.pyx:46)."""
    X = _datasets.gmm(4000, 64, 4, 2)
    W = X[:40].astype(np.float64)
    W = np.concatenate([W, W[:20], W[:10]])  # rows 40..59 duplicate 0..19, rows 60..69 duplicate 0..9
    for backend in ("simt", "tensor", "tensor1"):
        e = engine(bmu_backend=backend)
        _, idx = e.bmu(X, W, 1)
        assert idx.max() < 40, backend
        _, ref = O.bmu_expansion(X, W[:40], 1)
        gap = O.relative_gap(X, W[:40])
        np.testing.assert_array_equal(idx[gap >= GAP, 0], ref[gap >= GAP])
        e.close()


def test_bmu_collapsed_cluster_of_near_identical_prototypes():
    """Late in a fit large dead regions of the map collapse onto one centre: thousands of prototypes that
    agree to ~1e-7 (identical fp16 shadows, distinct float64 rows) plus exact copies.  For the samples of that
    centre every one of them lies inside the error bound, which drives the epilogue's gate / eviction paths,
    the flagged-row policy and the float64 re-scan; winners must still equal the oracle's outside the 1e-6
    near-tie set, with and without strict ties, for one and two winners."""
    n, d, m = 20000, 128, 2048
    X = _datasets.gmm(n, d, 16, 4)
    rng = np.random.default_rng(9)
    W = X[rng.choice(n, m, replace=False)].astype(np.float64)
    centre = X[X.shape[0] // 2].astype(np.float64) + 0.01
    blob = np.arange(300, 1500)
    W[blob] = centre * (1.0 + 1e-7 * rng.standard_normal((blob.size, 1))) + 1e-7 * rng.standard_normal((blob.size, d))
    W[1500:1540] = W[310]  # exact copies of a blob member
    W[40:50] = W[7]        # and of an ordinary prototype
    ref_gap = O.relative_gap(X, W)
    _, ref = O.bmu_expansion(X, W, 1)
    ok = ref_gap >= GAP
    flagged_seen = 0
    for kw in (dict(), dict(strict_ties=True)):
        e = engine(bmu_backend="tensor", **kw)
        _, idx = e.bmu(X, W, 1)
        st = e.bmu_stats_host()
        flagged_seen += st["flagged"]
        np.testing.assert_array_equal(idx[ok, 0], ref[ok])
        assert_bmu_parity(idx[:, 0], X, W, ref)
        # the lowest index among exact copies wins
        assert not np.isin(idx[:, 0], np.arange(1500, 1540)).any() and not np.isin(idx[:, 0], np.arange(40, 50)).any()
        dist2, idx2 = e.bmu(X, W, 2)
        np.testing.assert_array_equal(idx2[ok, 0], ref[ok])
        assert (dist2[:, 0] <= dist2[:, 1]).all() and (idx2[:, 0] != idx2[:, 1]).all()
        e.close()
    assert flagged_seen > 0, "the collapsed cluster should overflow the candidate tables of its samples"


def test_exclude_duplicates_marks_only_later_copies():
    """dbgsom_exclude_duplicates: wnorm = +inf exactly for prototypes equal to a lower-indexed one."""
    import torch

    from dbgsom_b200 import _native as nat

    lib = nat.load()
    rng = np.random.default_rng(0)
    m, d = 700, 64
    W = rng.normal(size=(m, d))
    W[300] = W[5]
    W[650] = W[5]
    W[12] = W[11]
    W[400, 3] = -0.0
    W[401] = W[400]
    W[401, 3] = 0.0  # -0.0 == +0.0: still a copy
    W[500] = W[499]
    W[500, 17] += 1e-12  # not a copy
    dev = torch.device("cuda", 0)
    dW = torch.from_numpy(W).to(dev)
    col = torch.from_numpy(rng.permutation(768).astype(np.int32)).to(dev)
    wnorm = torch.zeros(768, dtype=torch.float32, device=dev)
    scratch = torch.empty(m, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    nat.check(lib.dbgsom_exclude_duplicates(dW.data_ptr(), m, d, col.data_ptr(), wnorm.data_ptr(), scratch.data_ptr(), stream), "x")
    torch.cuda.synchronize(dev)
    marked = np.flatnonzero(np.isinf(wnorm.cpu().numpy()))
    expect = np.sort(col.cpu().numpy()[[300, 650, 12, 401]])
    np.testing.assert_array_equal(marked, expect)


def test_bmu_ragged_and_tiny_shapes():
    rng = np.random.default_rng(0)
    for n, d, m in [(4, 3, 4), (1, 5, 2), (129, 17, 5), (1000, 65, 257), (257, 2, 300)]:
        X = rng.normal(size=(n, d)).astype(np.float32)
        W = rng.normal(size=(m, d))
        for backend in ("simt", "tensor"):
            e = engine(bmu_backend=backend)
            dist, idx = e.bmu(X, W, min(2, m))
            _, ref = O.bmu_expansion(X, W, min(2, m))
            gap = O.relative_gap(X, W)
            np.testing.assert_array_equal(idx[gap >= GAP, 0], ref.reshape(n, -1)[gap >= GAP, 0])
            e.close()


def test_selective_search_matches_classic_and_oracle_on_a_grown_map():
    """The selective search (FLAG pass with the one-pass bound, REFINE pass over the flagged column tiles, samples in
    sorted order, shadow columns in map-patch order) on an IRREGULAR map grown by the reference's rules, with exact
    duplicates and a collapsed cluster of near-identical prototypes: winners equal the oracle's outside the 1e-6
    near-tie set, for both mask granules, and the refined share stays below the classic search's full sweep."""
    import torch

    from dbgsom_b200 import _native as nat
    from dbgsom_b200.topology import MapTopology

    rng = np.random.default_rng(11)
    topo = MapTopology.initial_square()
    for ep in range(200):
        topo.error[:] = rng.random(len(topo)) * 10
        topo.distribute_errors(6.0)
        topo.grow(6.0, ep)
        if len(topo) >= 1100:
            break
    m = len(topo)
    n, d = 60000, 192
    X = _datasets.gmm(n, d, 24, 17)
    # a smooth sheet over the grown map (prototype = blend of data rows by grid position), then the awkward cases
    pos = topo.positions().astype(np.float64)
    pos = (pos - pos.min(axis=0)) / np.ptp(pos, axis=0).max()
    anchors = X[rng.choice(n, 4, replace=False)].astype(np.float64)
    W = ((1 - pos[:, :1]) * (1 - pos[:, 1:]) * anchors[0] + pos[:, :1] * (1 - pos[:, 1:]) * anchors[1]
         + (1 - pos[:, :1]) * pos[:, 1:] * anchors[2] + pos[:, :1] * pos[:, 1:] * anchors[3])
    W += 0.05 * rng.standard_normal(W.shape)
    W[100:130] = W[40]                                                        # exact copies
    W[300:420] = W[250] * (1 + 1e-7 * rng.standard_normal((120, 1)))          # collapsed cluster
    _, ref, gap = O.bmu_with_gap(X, W)
    ok = gap >= GAP
    assert ok.mean() > 0.9
    for granule in (64, 128):
        e = engine(bmu_backend="tensor")
        e.select_granule = granule
        e.load_data(X, None, 0)
        e.set_map(W)
        e.set_hops_from_topology(topo)
        assert e._select_eligible(n, m, (nat.BMU_TENSOR, 3))
        # sorted order from a previous epoch's winners: here a perturbed copy of the map
        e.set_map(W + 0.02 * rng.standard_normal(W.shape))
        e.epoch(3.0, True, False)
        assert e.row_perm is not None
        e.set_map(W)
        x16 = (e.X16_hi, e.X16_lo, e.xnorm16)
        got = torch.full((n, 1), -7, dtype=torch.int32, device=e.dev)
        cls = torch.full((n, 1), -7, dtype=torch.int32, device=e.dev)
        e.bmu_stats_host(reset=True)
        e._run_bmu(e.X, n, e.ldx, x16, e.W[e.cur], m, 1, False, got, None, backend=(nat.BMU_TENSOR, 3), row_perm=e.row_perm,
                   selective=True)
        st = e.bmu_stats_host()
        e._run_bmu(e.X, n, e.ldx, x16, e.W[e.cur], m, 1, False, cls, None, backend=(nat.BMU_TENSOR, 3), row_perm=e.row_perm)
        got, cls = got[:, 0].cpu().numpy().astype(np.int64), cls[:, 0].cpu().numpy().astype(np.int64)
        e.close()
        assert st["selective_searches"] == 1 and 0 < st["refined_share"] < 0.8
        np.testing.assert_array_equal(got[ok], ref[ok])
        np.testing.assert_array_equal(cls[ok], ref[ok])
        assert_bmu_parity(got, X, W, ref)
        assert not np.isin(got, np.arange(100, 130)).any()  # the lowest index among exact copies wins


# ------------------------------------------------------------------------------------------ one epoch
def run_epoch(X, W, hop, sigma, pack, backend="auto", y=None, n_classes=0, entropy=False):
    e = engine(bmu_backend=backend)
    stats = e.load_data(X, y, n_classes)
    e.set_map(W)
    e.set_hops(hop_u16(hop))
    r = e.epoch(sigma, pack, entropy)
    r["winners"] = e.last_winners_host()
    W_new = e.weights()
    e.close()
    return stats, r, W_new


def assert_epoch_parity(r, W_new, X, W, hop, sigma, total_var, pack=True, min_strict=0.99, ref_winners=None):
    """Every output of one device epoch against the oracle -- never skipped.

    The parity gate (BASELINE.json) exempts the BMU of samples whose two best float64 distances agree to 1e-6
    relative.  Outside that set the device winners must equal the oracle's (or the reference fixture's); inside it
    the device's choice must be (numerically) as close.  The oracle update is then TEACHER-FORCED with the device's
    winners -- which differ from its own only on exempt samples -- so counts (exact), E (1e-5), prototypes (1e-5
    of max|W|) and the convergence scalar are compared for every neuron.  Returns the number of samples compared
    strictly and the number where the device used the exemption.
    """
    X64 = np.asarray(X, dtype=np.float64)
    n = X64.shape[0]
    _, own, gap = O.bmu_with_gap(X64, W)
    if ref_winners is None:
        ref_winners = own
    strict = gap >= GAP
    assert strict.mean() >= min_strict, f"only {strict.mean():.4f} of the samples are outside the near-tie set"
    win = r["winners"]
    bad = np.flatnonzero((win != ref_winners) & strict)
    assert bad.size == 0, f"{bad.size} BMU mismatches outside near-ties, first rows {bad[:5]}"
    loose = np.flatnonzero(win != ref_winners)
    if loose.size:
        d_dev = O.expansion_distance(X64[loose], W, win[loose])
        d_ref = O.expansion_distance(X64[loose], W, ref_winners[loose])
        np.testing.assert_allclose(d_dev, d_ref, rtol=2e-6, atol=1e-9)
    ref = O.epoch_step(X64, W, hop, sigma, total_var, pack=pack, winners=win)
    np.testing.assert_array_equal(r["counts"], ref["n"])
    assert r["counts"].sum() == n
    np.testing.assert_allclose(r["error"], ref["E"], rtol=1e-5, atol=1e-6)
    scale = np.abs(ref["W_new"][np.isfinite(ref["W_new"])]).max()
    assert np.array_equal(np.isfinite(W_new), np.isfinite(ref["W_new"]))
    fin = np.isfinite(ref["W_new"])
    assert np.abs(W_new[fin] - ref["W_new"][fin]).max() / scale < 1e-5
    assert r["change"] == pytest.approx(ref["change"], rel=1e-5)
    return int(strict.sum()), loose, ref


@pytest.mark.parametrize("path", STEP_FILES, ids=[os.path.basename(p)[5:-4] for p in STEP_FILES])
@pytest.mark.parametrize("backend", ["simt", "tensor"])
def test_epoch_matches_reference_fixture(path, backend):
    g, meta, X = load_step(path)
    stats, r, W_new = run_epoch(X, g["W"], g["hop"], float(g["sigma"]), True, backend)
    assert stats["total_variance"] == pytest.approx(float(g["total_var"]), rel=1e-6)
    n_strict, loose, _ = assert_epoch_parity(r, W_new, X, g["W"], g["hop"], float(g["sigma"]), float(g["total_var"]),
                                             ref_winners=g["winners"])
    assert n_strict > 0.99 * X.shape[0]
    # and against what the reference itself produced: directly for every neuron no exempt sample moved to or from
    m = g["W"].shape[0]
    untouched = np.ones(m, dtype=bool)
    untouched[r["winners"][loose]] = False
    untouched[g["winners"][loose]] = False
    assert untouched.mean() > 0.9
    np.testing.assert_array_equal(r["counts"][untouched], np.bincount(g["winners"], minlength=m)[untouched])
    np.testing.assert_allclose(r["error"][untouched], g["E"][untouched], rtol=1e-5, atol=1e-6)
    if loose.size == 0:
        scale = np.abs(g["W_new"]).max()
        assert np.abs(W_new - g["W_new"]).max() / scale < 1e-5


def test_epoch_aligned_rows_mode():
    g, meta, X = load_step([p for p in STEP_FILES if "gmm64_6x6_dead" in p][0])
    _, r, W_new = run_epoch(X, g["W"], g["hop"], float(g["sigma"]), False)
    assert_epoch_parity(r, W_new, X, g["W"], g["hop"], float(g["sigma"]), float(g["total_var"]), pack=False)
    packed = O.epoch_step(X, g["W"], g["hop"], float(g["sigma"]), float(g["total_var"]), pack=True)
    assert np.abs(W_new - packed["W_new"]).max() / np.abs(packed["W_new"]).max() > 1e-2


@pytest.mark.parametrize("shape", [(40000, 256, 32), (20000, 784, 20), (6000, 2048, 12), (3000, 4096, 8)])
def test_epoch_wide_rows_and_large_maps(shape):
    """Every accumulate kernel configuration (D up to 4096) and a map with dead neurons."""
    n, d, side = shape
    X = _datasets.gmm(n, d, 16, 21)
    m = side * side
    rng = np.random.default_rng(1)
    W = X[rng.choice(n, m, replace=False)].astype(np.float64)
    W[3] += 1e3
    W[m // 2] -= 1e3
    hop = O.hop_matrix_grid(side, side)
    sigma = 0.2 * side
    stats, r, W_new = run_epoch(X, W, hop, sigma, True)
    n_strict, _, _ = assert_epoch_parity(r, W_new, X, W, hop, sigma, stats["total_variance"])
    assert n_strict > 0.99 * n
    assert r["counts"][3] == 0 and r["counts"][m // 2] == 0


@pytest.mark.parametrize("shape,backend", [((200_000, 256, 64), "tensor"), ((70_000, 784, 20), "auto"),
                                            ((120_000, 128, 64), "tensor"), ((19_200, 4096, 64), "tensor")],
                         ids=["c3-shape-200k-x256-m4096", "c2-shape-70k-x784-m400", "c4-shape-120k-x128-m4096",
                              "c5-width-19k-x4096-m4096"])
def test_epoch_parity_over_a_trajectory_at_baseline_shapes(shape, backend):
    """Oracle parity of EVERY epoch output at the BASELINE feature widths and map sizes (configs 3, 2 and 4 at a row
    count the float64 oracle finishes in seconds), over six consecutive epochs of the real training trajectory:
    random-row prototypes first, then the smooth, partly dead maps of the large-sigma phase, where the packed-row
    quirk (Q1) is active.  Each epoch starts from the DEVICE's prototypes, so errors cannot hide by accumulating
    in the oracle's favour, and the oracle update is teacher-forced only on the exempt near-tie samples.
    The config-5 width (D = 4096, 150 row tiles: the streamed CTA-pair search with segmented accumulation in tensor
    memory and per-tile error bounds) runs on a 64 x 64 map; its half-trained maps are the flat sheets on which
    thousands of prototypes tie."""
    from bench import sigma_at

    n, d, side = shape
    m = side * side
    X = _datasets.gmm(n, d, 64 if d != 784 else 10, 3)
    rng = np.random.default_rng(0)
    W0 = X[rng.choice(n, m, replace=False)].astype(np.float64)
    hop = O.hop_matrix_grid(side, side)
    from dbgsom_b200.topology import MapTopology

    e = engine(bmu_backend=backend)
    e.resort_every = 2
    stats = e.load_data(X, None, 0)
    e.set_map(W0)
    # with the map topology the engine knows the patch order of the shadow columns: from the second epoch on (once the
    # samples are sorted by winner) the tensor search for D <= 256 is the SELECTIVE one (FLAG + REFINE passes)
    e.set_hops_from_topology(MapTopology.full_grid(side, side))
    np.testing.assert_array_equal(e.hops_host(), hop_u16(hop))
    dead_below_live = 0
    compared = 0
    n_epochs = 6
    for epoch in range(n_epochs):
        W = e.weights()
        sigma = sigma_at(epoch, m)
        r = e.epoch(sigma, True, False)
        r["winners"] = e.last_winners_host()
        # on the collapsed maps of this trajectory several per cent of the samples sit between prototypes that agree to
        # 1e-6 (the gate's exempt set): for those the device's choice is verified to be equally close instead, and the
        # update is compared for ALL samples through the teacher-forced oracle
        # (the ten-component config-2 mixture on a 400-neuron map collapses much further: most samples there sit
        # between prototypes that agree to 1e-6)
        n_strict, _, ref = assert_epoch_parity(r, e.weights(), X, W, hop, sigma, stats["total_variance"],
                                               min_strict=0.85 if d not in (784, 4096) else 0.2)
        compared += n_strict
        live = np.flatnonzero(ref["n"] > 0)
        dead = np.flatnonzero(ref["n"] == 0)
        dead_below_live += int(dead.size > 0 and live.max() > dead.min())
        if backend == "tensor":
            from dbgsom_b200 import _native as nat

            assert e.last_backend[0] == nat.BMU_TENSOR
    st = e.bmu_stats_host()
    assert st["fp32_reruns"] == 0
    if d <= 256:
        assert st["selective_searches"] == n_epochs - 1 and st["classic_searches"] == 1
        assert 0.0 < st["refined_share"] < 0.9
    e.close()
    assert compared > (0.9 if d not in (784, 4096) else 0.3) * n_epochs * n
    assert dead_below_live >= 1, "the trajectory should exercise the packed-row quirk"


def test_epoch_from_host_equals_resident_epoch():
    """The streamed-upload epoch (chunked H2D overlapped with the BMU search) gives the same result."""
    import torch

    X = _datasets.gmm(30000, 128, 16, 4)
    W = X[:400].astype(np.float64)
    hop = O.hop_matrix_grid(20, 20)
    out = []
    for streamed in (False, True):
        e = engine(bmu_backend="tensor")
        e.load_data(X, None, 0)
        e.set_map(W)
        e.set_hops(hop_u16(hop))
        if streamed:
            host = torch.from_numpy(X).pin_memory()
            e.X.zero_()
            r = e.epoch_from_host(host, 2.0, True, False, chunk_rows=7000)
        else:
            r = e.epoch(2.0, True, False)
        out.append((r, e.weights()))
        e.close()
    np.testing.assert_array_equal(out[0][0]["counts"], out[1][0]["counts"])
    np.testing.assert_allclose(out[0][0]["error"], out[1][0]["error"], rtol=1e-12)
    np.testing.assert_allclose(out[0][1], out[1][1], rtol=1e-12, atol=1e-12)


def test_epoch_entropy_error():
    X, lab = _datasets.gmm(5000, 32, 6, 3, return_labels=True)
    W = X[:25].astype(np.float64)
    hop = O.hop_matrix_grid(5, 5)
    _, r, _ = run_epoch(X, W, hop, 1.0, True, y=lab.astype(np.int64), n_classes=6, entropy=True)
    _, win = O.bmu_expansion(X, W, 1)
    import scipy.stats

    ref = np.array([scipy.stats.entropy(np.bincount(lab[win == j]), base=2) for j in range(25)])
    np.testing.assert_allclose(r["error"], ref, rtol=1e-12, atol=1e-12)


def test_full_size_properties_10m_rows():
    """BASELINE.json config 3 at full size (10M x 256, 64 x 64 map; the oracle would need hours):
    size-independent properties + oracle parity of a row sub-sample, over three consecutive epochs of the
    real trajectory (random-row prototypes, then smooth / collapsed maps)."""
    import torch

    n, d, side = 10_000_000, 256, 64
    m = side * side
    g = torch.Generator(device="cuda").manual_seed(0)
    centers = torch.randn(64, d, device="cuda", generator=g) * 2
    X = torch.empty((n, d), dtype=torch.float32, device="cuda")
    for s0 in range(0, n, 1 << 20):
        s1 = min(n, s0 + (1 << 20))
        lab = torch.randint(0, 64, (s1 - s0,), device="cuda", generator=g)
        X[s0:s1] = centers[lab] + torch.randn(s1 - s0, d, device="cuda", generator=g)
    e = engine(bmu_backend="tensor")
    stats = e.load_device_data(X)
    assert stats["n_samples"] == n
    e.init_map_from_rows(np.random.default_rng(0).choice(n, m, replace=False), capacity=m)
    e.set_hops(hop_u16(O.hop_matrix_grid(side, side)))
    sub = torch.from_numpy(np.sort(np.random.default_rng(1).choice(n, 2000, replace=False))).cuda()
    Xs = X[sub].cpu().numpy()
    for epoch, sigma in enumerate((12.8, 12.4, 12.1)):
        W = e.weights()
        r = e.epoch(sigma, True, False)
        part = e.part[: m * d + 3 * m]
        Sk, sk = part[: m * d].view(m, d), part[m * d : m * d + m]
        cnt, E = r["counts"], r["error"]
        # every sample is counted once; weights in (0, 1]; errors are sums of distances
        assert cnt.sum() == n and (cnt >= 0).all()
        skh = sk.cpu().numpy()
        assert (skh[cnt > 0] > 0).all() and (skh <= cnt + 1e-6).all() and (E >= 0).all() and (E[cnt == 0] == 0).all()
        assert bool(torch.isfinite(Sk).all())
        # winners of the sub-sample against the float64 oracle (exact outside the 1e-6 near-tie set)
        idx = e.idx.view(-1)[:n][sub].cpu().numpy().astype(np.int64)
        n_strict, n_loose = assert_bmu_parity(idx, Xs, W)
        assert n_strict > 1000
        # linearity: sum_j E_j = sum_i d_i, checked on the sub-sample's share via exact distances
        d_sub = np.linalg.norm(Xs.astype(np.float64) - W[idx], axis=1)
        assert E.sum() / n == pytest.approx(d_sub.mean(), rel=0.05)
        assert np.isfinite(r["change"]) and r["change"] > 0
    # repeatability: the same state gives the same counts and (to float64 round-off) the same sums
    W = e.weights()
    e.set_map(W)
    r1 = e.epoch(11.0, True, False)
    e.set_map(W)
    r2 = e.epoch(11.0, True, False)
    np.testing.assert_array_equal(r1["counts"], r2["counts"])
    np.testing.assert_allclose(r1["error"], r2["error"], rtol=1e-12)
    assert r1["change"] == pytest.approx(r2["change"], rel=1e-12)
    e.close()


def test_strict_ties_and_worst_case_bound_agree_with_default():
    """`strict_ties` (flagged samples always re-scored against all prototypes) and bound_scale = 1
    (Cauchy-Schwarz worst case) must give the oracle's winners too; the default may only differ inside
    the 1e-6 near-tie set."""
    n, d, side = 30000, 128, 32
    X = _datasets.gmm(n, d, 16, 8)
    rng = np.random.default_rng(3)
    W_rows = X[rng.choice(n, side * side, replace=False)].astype(np.float64)
    H = O.neighborhood(O.hop_matrix_grid(side, side), 6.0)
    W = (H @ W_rows) / H.sum(axis=1)[:, None]  # smooth sheet: many near-ties
    W[100:140] = W[60]  # and a block of exact duplicates
    ref_gap = O.relative_gap(X, W)
    _, ref = O.bmu_expansion(X, W, 1)
    for kw in (dict(), dict(strict_ties=True), dict(bound_scale=1.0), dict(bmu_backend="tensor1", strict_ties=True)):
        e = engine(**{"bmu_backend": "tensor", **kw})
        _, idx = e.bmu(X, W, 1)
        st = e.bmu_stats_host()
        e.close()
        ok = ref_gap >= GAP
        np.testing.assert_array_equal(idx[ok, 0], ref[ok])
        assert idx[:, 0].min() >= 0 and not np.isin(idx[:, 0], np.arange(100, 140)).any()  # lowest duplicate wins
        if kw.get("strict_ties"):
            assert st["flagged"] == st["full_rescans"]


# ------------------------------------------------------------------------------------------ full fits
@pytest.mark.parametrize("path", TRAJ_FILES, ids=[os.path.basename(p)[5:-4] for p in TRAJ_FILES])
def test_fit_matches_reference_fixture(path):
    from dbgsom_b200 import SomClassifier, SomVQ

    g = np.load(path, allow_pickle=False)
    meta = json.loads(str(g["meta"]))
    X, y = _datasets.load(meta["data"])
    X = np.ascontiguousarray(X.astype(meta["cast"]))
    is_vq = meta["est"] == "vq"
    est = (SomVQ if is_vq else SomClassifier)(**meta["params"])
    est.fit(X) if is_vq else est.fit(X, y)
    # growth decisions are discrete: the same map must come out
    np.testing.assert_array_equal(np.array(est.neurons_), g["neurons"])
    assert est.n_iter_ == int(g["n_iter_"])
    assert est.growing_threshold_ == pytest.approx(float(g["growing_threshold"]), rel=1e-9)
    scale = np.abs(g["weights"]).max()
    assert np.abs(est.weights_ - g["weights"]).max() / scale < 1e-4
    assert est.quantization_error_ == pytest.approx(float(g["quantization_error"]), rel=1e-5)
    assert est.topographic_error_ == pytest.approx(float(g["topographic_error"]), abs=2.0 / X.shape[0])
    if is_vq:
        assert np.mean(est.labels_ == g["labels"]) > 0.999
        assert np.mean(est.predict(X[:200]) == g["predict_head"]) > 0.99
    else:
        np.testing.assert_array_equal(est.classes_, g["classes"])
        assert est.score(X, y) == pytest.approx(float(g["score"]), abs=2e-3)


# ------------------------------------------------------------------------------------------ config 2 (70000 x 784)
FITSTEP_FILES = golden_files("fitstep")


def load_fitstep(path):
    g = np.load(path, allow_pickle=False)
    meta = json.loads(str(g["meta"]))
    X, y = _datasets.load(meta["data"])
    return g, meta, np.ascontiguousarray(X.astype(meta["cast"])), y


@pytest.mark.parametrize("backend", ["auto", "simt"])
@pytest.mark.parametrize("path", FITSTEP_FILES, ids=[os.path.basename(p)[8:-4] for p in FITSTEP_FILES])
def test_config2_epochs_teacher_forced_from_reference_states(path, backend):
    """BASELINE.json configs[1]: the prototypes, hop matrix and sigma the REFERENCE had at epochs 5 .. 30 of its own
    `SomClassifier.fit` on the 70000 x 784 mixture go into one device epoch; winners must equal the reference's
    outside the near-tie set, per-neuron error and the updated prototypes must be the reference's (1e-5)."""
    g, meta, X, _ = load_fitstep(path)
    e = engine(bmu_backend=backend)
    stats = e.load_data(X, None, 0)
    assert stats["total_variance"] == pytest.approx(float(g["total_var"]), rel=1e-5)
    for ep in g["captured"]:
        W, h16, sigma = g[f"e{ep}_W"], g[f"e{ep}_hop"], float(g[f"e{ep}_sigma"])
        hop = h16.astype(np.float64)
        hop[h16 == 0xFFFF] = np.inf
        e.set_map(W)
        e.set_hops(h16)
        r = e.epoch(sigma, True, False)
        r["winners"] = e.last_winners_host()
        W_new = e.weights()
        ref_win = g[f"e{ep}_winners"].astype(np.int64)
        n_strict, loose, _ = assert_epoch_parity(r, W_new, X, W, hop, sigma, float(g["total_var"]), ref_winners=ref_win,
                                                 min_strict=0.9)
        assert n_strict > 0.9 * X.shape[0]
        m = W.shape[0]
        untouched = np.ones(m, dtype=bool)
        untouched[r["winners"][loose]] = False
        untouched[ref_win[loose]] = False
        np.testing.assert_allclose(r["error"][untouched], g[f"e{ep}_E"][untouched], rtol=1e-5, atol=1e-6)
        if loose.size == 0:
            scale = np.abs(g[f"e{ep}_W_new"]).max()
            assert np.abs(W_new - g[f"e{ep}_W_new"]).max() / scale < 1e-5
    e.close()


@pytest.mark.parametrize("backend", ["auto", "simt"])
@pytest.mark.parametrize("path", FITSTEP_FILES, ids=[os.path.basename(p)[8:-4] for p in FITSTEP_FILES])
def test_config2_fit_follows_the_reference_trajectory(path, backend):
    """The whole config-2 fit through the estimator API against the reference's own fit, epoch by epoch.

    Through the entire growth phase (epochs 0-19: the map grows from 4 to 64 neurons) the device reproduces the
    reference EXACTLY: the same map size every epoch, identical per-neuron sample counts and per-neuron errors to
    1e-9.  In the fine phase (sigma = 0.7) the packed-row quirk leaves prototypes that agree to ~1e-16; which of two
    such prototypes wins a sample is decided by the rounding of scikit-learn's GEMM expansion in the reference and by
    exact float64 differences here, so from epoch 20 on a few hundred samples per epoch are assigned differently and
    the two (chaotic) trajectories drift apart.  Past that point only the statistics are compared."""
    from dbgsom_b200 import SomClassifier
    from dbgsom_b200.engine import DeviceEngine

    g, meta, X, y = load_fitstep(path)
    log = dict(M=[], E=[], n=[])

    class Rec(DeviceEngine):
        def epoch(self, sigma, pack_rows, entropy_error, **kw):
            log["M"].append(self.M)
            r = super().epoch(sigma, pack_rows, entropy_error, **kw)
            log["E"].append(np.array(r["error"]))
            log["n"].append(np.array(r["counts"]))
            return r

    class Est(SomClassifier):
        def _make_engine(self, distributed=None):
            return Rec(device=self.device, bmu_backend=self.bmu_backend, strict_ties=self.strict_ties)

    est = Est(**meta["params"], strict_ties=True, bmu_backend=backend)
    est.fit(X, y)
    ref_m = g["epoch_M"]
    np.testing.assert_array_equal(log["M"], ref_m)            # every growth decision of the fit
    off = 0
    exact_epochs = 0
    for e_, m in enumerate(ref_m):
        E_ref, n_ref = g["E_flat"][off:off + m], g["n_flat"][off:off + m]
        off += m
        if e_ < 20:
            np.testing.assert_array_equal(log["n"][e_], n_ref)
            np.testing.assert_allclose(log["E"][e_], E_ref, rtol=1e-9, atol=1e-9)
            exact_epochs += 1
        else:
            assert log["n"][e_].sum() == n_ref.sum() == X.shape[0]
    assert exact_epochs == 20
    assert est.n_iter_ == int(g["n_iter_"])
    assert abs(len(est.neurons_) - len(g["neurons"])) <= 4
    assert est.quantization_error_ == pytest.approx(float(g["quantization_error"]), rel=0.1)
    np.testing.assert_array_equal(est.classes_, g["classes"])
    assert est.score(X[:5000], y[:5000]) >= 0.0  # the sparse-coding inference path runs at this shape


@pytest.mark.parametrize("n", [3, 4])
@pytest.mark.parametrize("backend", ["simt", "tensor"])
def test_one_prototype_wins_every_sample_of_a_tiny_set(n, backend):
    """Fewer samples than K2 has teams of warps: most teams have an empty range, and the teams that continue the one
    segment sit between empty ones.  Counts, errors and prototypes must still be the oracle's."""
    rng = np.random.default_rng(n)
    X = rng.normal(size=(n, 8)).astype(np.float32).astype(np.float64)
    W = np.concatenate([X.mean(axis=0, keepdims=True), 50.0 + rng.normal(size=(3, 8))])
    hop = O.hop_matrix_grid(2, 2).astype(np.float64)
    stats, r, W_new = run_epoch(X, W, hop, 1.0, True, backend)
    assert np.array_equal(r["winners"], np.zeros(n, dtype=np.int64))
    ref = O.epoch_step(X, W, hop, 1.0, stats["total_variance"], pack=True)
    np.testing.assert_array_equal(r["counts"], ref["n"])
    np.testing.assert_allclose(r["error"], ref["E"], rtol=1e-12, atol=1e-12)
    assert np.abs(W_new - ref["W_new"]).max() / np.abs(ref["W_new"]).max() < 1e-12


@pytest.mark.parametrize("n,d,gx,gy", [
    (300_000, 64, 16, 16),    # the sorted sample order feeds the selective search from the second epoch on
    (20_000, 768, 8, 8),      # D > 512: teams of several warps in K2
    (60_000, 16, 100, 100),   # M > 8192: one warp per CTA in the stable scatter
    (5, 8, 2, 2),             # fewer samples than K2 has teams
], ids=["selective", "wide_teams", "large_map", "tiny"])
def test_epochs_repeat_bit_for_bit(n, d, gx, gy):
    """Two engines on the same data and start produce the same prototypes, errors and counts, bit for bit, epoch after
    epoch: every sum is taken in a fixed order, and K2's permutation lists the samples of each winner in ascending
    sample index (maps of up to 24576 neurons)."""
    import torch

    from dbgsom_b200.topology import MapTopology

    X = _datasets.gmm(n, d, 16, 7)
    m = gx * gy
    runs = []
    for _ in range(2):
        e = engine(bmu_backend="tensor")
        stats = e.load_data(X, None, 0)
        e.init_map_from_rows(np.random.default_rng(3).choice(n, m, replace=n < m), capacity=m)
        e.set_hops_from_topology(MapTopology.full_grid(gx, gy))
        outs = []
        for ep in range(4):
            # sigma grows with the map, as in a fit: too narrow a neighbourhood leaves far rows with no weight (NaN)
            r = e.epoch(max(2.0, 0.1 * gx) - 0.3 * ep, True, False)
            outs.append((e.weights(), r["error"], r["counts"], r["change"]))
        win = e.last_winners_host()
        assert (win >= 0).all()
        off = int(e.lib.dbgsom_accumulate_perm_offset(e.N, e.M))
        perm = e._ws["acc"][off : off + 4 * e.N].view(torch.int32).cpu().numpy()
        np.testing.assert_array_equal(perm, np.argsort(win, kind="stable"))
        runs.append((stats["total_variance"], outs))
        e.close()
    assert runs[0][0] == runs[1][0]
    for a, b in zip(runs[0][1], runs[1][1]):
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)


def test_tile_bounds_are_the_column_tile_maxima():
    """dbgsom_tile_bounds: max ||u_j|| and max |wnorm_j| per 128 shadow columns, in the column order of the search,
    without padding columns and without prototypes taken out of the search (wnorm = +inf)."""
    import torch

    rng = np.random.default_rng(5)
    m, d = 700, 320
    X = rng.normal(size=(4000, d)).astype(np.float32)
    from dbgsom_b200.topology import MapTopology

    eng = engine(bmu_backend="tensor")
    eng.load_data(X, None, 0)
    W0 = rng.normal(size=(m, d)) * np.linspace(0.1, 3.0, m)[:, None]
    W0[13] = W0[7]  # an exact copy: leaves a top-1 search
    eng.set_map(W0)
    eng.set_hops_from_topology(MapTopology.full_grid(28, 25))
    W = eng.W[eng.cur]
    mpad = eng._prepare_w(W, m, True, True, top1=True)
    assert eng._tile_ready and mpad == 768
    torch.cuda.synchronize()
    tb = eng.tile_bound[: mpad // 64].cpu().numpy().reshape(-1, 2)
    poc = eng.proto_of_col[:mpad].cpu().numpy()
    wn = eng.wnorm[:mpad].cpu().numpy()
    Wd = W[:m, :d].cpu().numpy()
    u = (Wd - Wd.mean(axis=0)) * eng.scale
    un = np.sqrt((u * u).sum(axis=1))
    for t in range(mpad // 128):
        cols = np.arange(128 * t, 128 * t + 128)
        ok = (poc[cols] < m) & np.isfinite(wn[cols])
        assert not ok[poc[cols] == 13].any()  # the copy does not count
        exp_u = un[poc[cols][ok]].max() if ok.any() else 0.0
        exp_w = np.abs(wn[cols][ok]).max() if ok.any() else 0.0
        assert tb[t, 0] == pytest.approx(exp_u, rel=1e-6) and tb[t, 0] >= exp_u * (1 - 1e-7)
        assert tb[t, 1] == pytest.approx(exp_w, rel=1e-6)
    eng.close()


@pytest.mark.parametrize("env,shape", [
    ({"DBGSOM_TC_PAIR": "0"}, ("60000", "256", "1024", "4")),
    ({"DBGSOM_TC_PAIR": "0", "DBGSOM_TC_CLUSTER": "1"}, ("60000", "256", "1024", "4")),
    ({"DBGSOM_TC_PAIR": "1"}, ("60000", "256", "1024", "4")),
    ({"DBGSOM_TC_PAIR": "1", "DBGSOM_TC_BIAS": "1"}, ("60000", "128", "1024", "4")),
    ({"DBGSOM_TC_PAIR": "1"}, ("60000", "512", "1024", "3")),
    ({"DBGSOM_TC_PAIR": "1", "DBGSOM_TC_SEGM": "0"}, ("60000", "512", "1024", "3")),
    ({"DBGSOM_TC_SEGM": "1"}, ("60000", "512", "1024", "3")),
    ({"DBGSOM_TC_SEGM": "2"}, ("40000", "2048", "4096", "4")),
    ({"DBGSOM_TC_PAIR": "0"}, ("60000", "512", "1024", "3")),
    # 768 accumulation steps per score at D = 4096: wrong winners with exact relative gaps up to 8e-6 with the bound of
    # D = 256; now the chain is cut into partial accumulators (segmented form), or the bound follows the chain
    ({}, ("150000", "4096", "1024", "1")),
    # per-tile error bounds of the streamed forms (default on): the same search with the map-wide bound, and a large
    # half-trained map -- a flat sheet of small-norm prototypes far from the samples plus a few unfolded ones -- where
    # thousands of prototypes tie to 1e-8 and the tile bounds decide which rows can be proven near-ties
    ({"DBGSOM_TILE_BOUND": "0"}, ("60000", "512", "1024", "3")),
    ({}, ("40000", "2048", "4096", "6")),
    ({"DBGSOM_TC_SEGM": "0"}, ("40000", "2048", "4096", "6")),
], ids=["multicast-cluster", "single-cta", "cta-pair", "cta-pair-bias-kstep", "cta-pair-streamed-segmented",
        "cta-pair-streamed-one-chain", "cta-pair-streamed-segmented-register-sums", "cta-pair-streamed-segmented-8-kblocks",
        "multicast-streamed", "long-accumulation-chain", "streamed-map-wide-bound",
        "tile-bounds-flat-sheet-segmented", "tile-bounds-flat-sheet-one-chain"])
def test_tensor_kernel_variants_agree_with_simt(env, shape):
    """The forms of the tcgen05 candidate kernel (CTA pairs with cta_group::2 -- the default; sample tile in tensor
    memory for D <= 256, both operands streamed beyond, there with segmented accumulation whose running sums live in
    tensor memory -- the default -- or in registers, or with one accumulation chain; optionally wnorm as a bias k-step --, clusters with TMA
    multicast, single CTAs) are selected by environment switches read once per process, so each runs in its own
    interpreter: winners on a four-epoch bench-like trajectory must equal the fp32 SIMT back end's
    (both followed by the exact float64 re-score) outside a 1e-7 relative float64 gap."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "check_backends.py"), *shape],
                         env={**os.environ, **env}, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip().endswith("OK"), out.stdout[-2000:]
