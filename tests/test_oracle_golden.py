"""Pin the CPU oracle against outputs of the reference itself (tests/golden/step_*.npz)."""
import json
import os

import numpy as np
import pytest

import _datasets
from conftest import golden_files
from oracle import som_oracle as O

STEP_FILES = golden_files("step")


def _load(path):
    g = np.load(path, allow_pickle=False)
    meta = json.loads(str(g["meta"]))
    X, _ = _datasets.load(meta["data"])
    X = np.ascontiguousarray(X.astype(meta["cast"]))
    return g, meta, X


def test_golden_files_present():
    assert len(STEP_FILES) >= 7
    assert len(golden_files("traj")) >= 7


@pytest.mark.parametrize("path", STEP_FILES, ids=[os.path.basename(p)[5:-4] for p in STEP_FILES])
def test_step_matches_reference(path):
    g, meta, X = _load(path)
    W, hop = g["W"], g["hop"]
    assert float(O.total_variance(X)) == pytest.approx(float(g["total_var"]), rel=1e-13)
    assert O.growing_threshold(X) == pytest.approx(float(g["growing_threshold"]), rel=1e-13)
    # float64 statistics (what the device computes) agree to float32 round-off at worst
    assert float(O.total_variance(X.astype(np.float64))) == pytest.approx(float(g["total_var"]), rel=1e-6)
    sigma = O.current_sigma(
        meta["epoch"], W.shape[0], n_iter=meta["n_iter"], phase=meta["phase"], **meta.get("params", {})
    )
    assert sigma == pytest.approx(float(g["sigma"]), rel=1e-15)
    out = O.epoch_step(X, W, hop, sigma, float(g["total_var"]), pack=True)
    # float32 X: the reference keeps gamma = 1/V as a float32 scalar (BaseSom.py:536) -> 1e-7 level
    tol = 1e-9 if meta["cast"] == "float64" else 2e-7
    np.testing.assert_array_equal(out["winners"], g["winners"])
    np.testing.assert_allclose(out["dist"], g["dist"], rtol=tol, atol=1e-9)
    np.testing.assert_allclose(out["k"], g["k"], rtol=tol, atol=1e-12)
    np.testing.assert_allclose(out["E"], g["E"], rtol=max(tol, 1e-10))
    np.testing.assert_allclose(out["W_new"], g["W_new"], rtol=tol, atol=tol)
    assert bool(out["change"] < 1e-5) == bool(g["converged"])


@pytest.mark.parametrize("path", STEP_FILES, ids=[os.path.basename(p)[5:-4] for p in STEP_FILES])
def test_restated_argkmin_matches_reference(path):
    """The numpy restatement of sklearn's ArgKmin64 gives the reference's BMUs (top-1 and top-2)."""
    g, meta, X = _load(path)
    d1, i1 = O.bmu_expansion(X, g["W"], 1)
    gap = O.relative_gap(X, g["W"])
    safe = gap > 1e-9
    np.testing.assert_array_equal(i1[safe], g["winners"][safe])
    np.testing.assert_allclose(d1, g["dist"], rtol=1e-6, atol=1e-6)
    d2, i2 = O.bmu_expansion(X, g["W"], 2)
    np.testing.assert_array_equal(i2[safe, 0], g["winners2"][safe, 0])
    np.testing.assert_allclose(d2, g["dist2"], rtol=1e-6, atol=1e-6)
    assert (d2[:, 0] <= d2[:, 1]).all()


def test_packing_quirk_is_required():
    """Q1: with dead neurons at low indices only the packed layout reproduces the reference."""
    path = [p for p in STEP_FILES if "gmm64_6x6_dead" in p][0]
    g, meta, X = _load(path)
    aligned = O.epoch_step(X, g["W"], g["hop"], float(g["sigma"]), float(g["total_var"]), pack=False)
    err = np.abs(aligned["W_new"] - g["W_new"]).max() / np.abs(g["W_new"]).max()
    assert err > 1e-2


def test_smooth_gemm_equals_broadcast_form():
    rng = np.random.default_rng(0)
    M, D = 30, 7
    C, n = rng.normal(size=(M, D)), rng.integers(0, 9, M).astype(float)
    H = O.neighborhood(O.hop_matrix_grid(5, 6), 1.3)
    np.testing.assert_allclose(O.smooth(C, n, H), O.smooth_broadcast(C, n, H), rtol=1e-12)


def test_initial_rows_equal_row_choice():
    X = np.arange(40.0).reshape(10, 4)
    rows = np.random.default_rng(seed=7).choice(a=X, size=4, replace=False)
    np.testing.assert_array_equal(X[O.initial_rows(10, 7)], rows)
    np.testing.assert_array_equal(O.initial_rows(1797, 0), [484, 918, 1526, 1143])


def test_hop_matrix_grid_equals_floyd_warshall():
    import networkx as nx

    g = nx.grid_2d_graph(4, 6)
    np.testing.assert_array_equal(O.hop_matrix_grid(4, 6), nx.floyd_warshall_numpy(g))


# ------------------------------------------------------------------ BASELINE.json configs[1] (70000 x 784, ten classes)
FITSTEP = golden_files("fitstep")


def load_fitstep(path):
    g = np.load(path, allow_pickle=False)
    meta = json.loads(str(g["meta"]))
    X, y = _datasets.load(meta["data"])
    return g, meta, np.ascontiguousarray(X.astype(meta["cast"])), y


def hop_float(h16):
    hop = h16.astype(np.float64)
    hop[h16 == 0xFFFF] = np.inf
    return hop


@pytest.mark.parametrize("path", FITSTEP, ids=[os.path.basename(p)[8:-4] for p in FITSTEP])
def test_fitstep_states_match_reference(path):
    """The oracle reproduces what the reference's epoch body computed INSIDE a config-2 fit, from the
    prototypes / hop matrix / sigma that fit had at the captured epochs (float32 samples: the reference runs
    sklearn's float32 -> float64 fallback path there)."""
    g, meta, X, _ = load_fitstep(path)
    # states of both phases: one of the growth phase and one at the fine phase's sigma (that of the last epoch)
    sig = g["epoch_sigma"][g["captured"]]
    assert sig.max() > sig.min() == g["epoch_sigma"][-1]
    for e in g["captured"]:
        W, hop, sigma = g[f"e{e}_W"], hop_float(g[f"e{e}_hop"]), float(g[f"e{e}_sigma"])
        assert W.shape[0] == int(g["epoch_M"][e]) and sigma == pytest.approx(float(g["epoch_sigma"][e]), rel=1e-15)
        out = O.epoch_step(X, W, hop, sigma, float(g["total_var"]), pack=True)
        gap = O.relative_gap(X, W)
        safe = gap > 1e-9
        ref_win = g[f"e{e}_winners"].astype(np.int64)
        np.testing.assert_array_equal(out["winners"][safe], ref_win[safe])
        assert safe.mean() > 0.99
        # Collapsed maps hold prototypes that agree to 1e-9 and closer; between those, sklearn's rounding decides.  The
        # update is therefore compared with the reference's OWN winners fed to the oracle (never skipped).
        if not safe.all():
            out = O.epoch_step(X, W, hop, sigma, float(g["total_var"]), pack=True, winners=ref_win)
        np.testing.assert_allclose(out["E"], g[f"e{e}_E"], rtol=2e-7, atol=1e-9)
        scale = np.abs(g[f"e{e}_W_new"]).max()
        assert np.abs(out["W_new"] - g[f"e{e}_W_new"]).max() / scale < 3e-7  # stored as float32
        # dead neurons below live ones: the packed-row quirk is active in these states
        n = out["n"]
        live = np.flatnonzero(n > 0)
        if e >= 11:
            assert (n == 0).any() and live.max() > np.flatnonzero(n == 0).min()
