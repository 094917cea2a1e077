"""kneighbors / the top-k BMU search (n_bmu > 2) on the device against exact float64 nearest neighbours."""
import numpy as np
import pytest

import _datasets
from _topk_reference import GAP, assert_topk_parity, bench_like_maps
from oracle import som_oracle as O

pytestmark = pytest.mark.gpu
KS = (3, 4, 5, 8, 16)


def engine(**kw):
    from dbgsom_b200.engine import DeviceEngine

    return DeviceEngine(**kw)


# "auto" picks the three-pass tensor search for every shape but the last (N * M * ldx >= 2^31, M >= 128).  The launch
# forms: D <= 256 with 157 row tiles -> CTA pairs with the sample tile in tensor memory; D > 256 with >= 148 row tiles
# -> streamed CTA pairs (segmented accumulation); fewer row tiles -> single-CTA forms.
@pytest.mark.parametrize("backend", ["auto", "simt"])
@pytest.mark.parametrize("shape", [(20000, 64, 2048), (20000, 256, 1024), (6000, 768, 512), (20000, 768, 512),
                                   (3000, 4096, 300), (20000, 4096, 256), (500, 32, 100)])
def test_topk_matches_exact(backend, shape):
    from dbgsom_b200 import _native as nat

    n, d, m = shape
    X, W = bench_like_maps(n, d, m)
    e = engine(bmu_backend=backend)
    tensor = backend == "auto" and m >= 128
    for k in KS:
        dist, idx = e.bmu(X, W, k)
        assert e.last_backend == ((nat.BMU_TENSOR, 3) if tensor else (nat.BMU_SIMT, 0))
        assert idx.dtype == np.int64 and dist.dtype == np.float64
        assert_topk_parity(dist, idx, X, W, k)
    e.close()


def test_one_pass_tensor_refuses_topk():
    X, W = bench_like_maps(2000, 64, 300)
    e = engine(bmu_backend="tensor1")
    with pytest.raises(ValueError, match="at most 2"):
        e.bmu(X, W, 3)
    e.close()


@pytest.mark.parametrize("backend", ["tensor", "simt"])
def test_exact_copies_are_consecutive_lowest_first(backend):
    X, W = bench_like_maps(4000, 64, 200)
    src = 17
    copies = [17, 40, 41, 150]
    for c in copies[1:]:
        W[c] = W[src]
    e = engine(bmu_backend=backend)
    for k in (4, 8, 16):
        dist, idx = e.bmu(X, W, k)
        assert_topk_parity(dist, idx, X, W, k)
        rows = np.flatnonzero(np.isin(idx, copies).any(axis=1))
        assert rows.size > 0
        for r in rows:
            pos = np.flatnonzero(np.isin(idx[r], copies))
            got = idx[r, pos]
            # the copies present form a run, in ascending index, starting at the lowest copy
            assert (np.diff(pos) == 1).all(), (r, idx[r])
            np.testing.assert_array_equal(got, copies[: len(got)])
            assert np.all(dist[r, pos] == dist[r, pos[0]])
    e.close()


@pytest.mark.parametrize("backend", ["tensor", "simt"])
def test_collapsed_map_overflows_and_rescans(backend):
    """Hundreds of near-identical prototypes: candidate tables overflow and rows go to the float64 re-scan."""
    rng = np.random.default_rng(2)
    X = _datasets.gmm(6000, 64, 8, 4)
    # ten clusters of 50 prototypes each, at samples 0..9 and equal in float32; plus 100 sample rows
    W = np.repeat(X[:10].astype(np.float64), 50, axis=0) + rng.normal(0.0, 1e-9, size=(500, 64))
    W = np.concatenate([W, X[rng.choice(np.arange(10, len(X)), 100, replace=False)]])
    e = engine(bmu_backend=backend)
    for k in (3, 8, 16):
        dist, idx = e.bmu(X, W, k)  # each call starts its statistics from zero
        st = e.bmu_stats_host()
        assert st["flagged"] > 0 and st["full_rescans"] == st["flagged"], st
        assert_topk_parity(dist, idx, X, W, k)
    e.close()


@pytest.mark.parametrize("d", [256, 768])
def test_strict_worst_case_bound_is_exact(d):
    """Tensor search with the Cauchy-Schwarz bound and the linear accumulation term: exact outside 1e-9."""
    from dbgsom_b200 import _native as nat

    X, W = bench_like_maps(20000, d, 1024)
    e = engine(strict_ties=True, bound_scale=1.0)
    for k in (3, 16):
        dist, idx = e.bmu(X, W, k)
        assert e.last_backend == (nat.BMU_TENSOR, 3)
        assert_topk_parity(dist, idx, X, W, k, gap=1e-9)
    e.close()


def test_small_k_unchanged_and_full_sort():
    from dbgsom_b200 import SomVQ

    X, W = bench_like_maps(30000, 64, 2048)
    som = SomVQ()
    som.weights_ = W
    for k in (1, 2):
        d_old, i_old = som._get_winning_neurons(X, k)
        d_new, i_new = som.kneighbors(X, k)
        np.testing.assert_array_equal(i_new.reshape(i_old.shape), i_old)
        np.testing.assert_array_equal(d_new.reshape(d_old.shape), d_old)
    # k = M: the whole map in order
    Ws = W[:12]
    som.weights_ = Ws
    dist, idx = som.kneighbors(X[:3000], 12)
    assert_topk_parity(dist, idx, X[:3000], Ws, 12)
    d2 = O.sqdist_exact(X[:3000], Ws)
    np.testing.assert_array_equal(np.sort(idx, axis=1), np.tile(np.arange(12), (3000, 1)))
    np.testing.assert_allclose(dist, np.sqrt(np.sort(d2, axis=1)), rtol=1e-12)


@pytest.mark.parametrize("k", [3, 16])
def test_chunked_is_bit_identical(k):
    """The chunks keep the shadow shift and scale of the whole X, so even the tensor search gives identical results."""
    X, W = bench_like_maps(20000, 256, 1024)
    e = engine()
    d_one, i_one = e.bmu(X, W, k)
    e.close()
    e = engine()
    e.stream_rows = 4096
    d_ch, i_ch = e.bmu(X, W, k)
    e.close()
    np.testing.assert_array_equal(i_ch, i_one)
    np.testing.assert_array_equal(d_ch, d_one)


def test_repeatable():
    X, W = bench_like_maps(20000, 256, 1024)
    out = []
    for _ in range(2):
        e = engine()
        out.append(e.bmu(X, W, 8))
        e.close()
    np.testing.assert_array_equal(out[0][1], out[1][1])
    np.testing.assert_array_equal(out[0][0], out[1][0])


def test_estimators_on_digits():
    from sklearn.neighbors import NearestNeighbors

    from dbgsom_b200 import SomClassifier, SomVQ

    X, y = _datasets.load("digits")
    som = SomVQ(random_state=0).fit(X)
    clf = SomClassifier(random_state=0, n_iter=40).fit(X, y)
    for est in (som, clf):
        W = est.weights_
        for k in (1, 5, 16):
            dist, idx = est.kneighbors(X, k)
            assert_topk_parity(dist, idx, X.astype(np.float32), W, k)
            ref_d, ref_i = NearestNeighbors(n_neighbors=k).fit(W).kneighbors(X)
            ok = O.relative_gap(X, W) >= GAP
            np.testing.assert_array_equal(idx[ok, 0], ref_i[ok, 0])
            np.testing.assert_allclose(dist, ref_d, rtol=1e-6, atol=1e-6)
    np.testing.assert_array_equal(som.kneighbors(X, 1)[1][:, 0], som.predict(X))
    only = som.kneighbors(X, 4, return_distance=False)
    np.testing.assert_array_equal(only, som.kneighbors(X, 4)[1])
