"""`fit(X, y, sample_weight)`: frequency weights through the estimator layer, driven by the CPU oracle engine."""
import os
import socket
import sys

import numpy as np
import pytest

import _datasets
import _weighted_oracle as WO
from _weighted_oracle import WeightedOracleEngine as OracleEngine
from dbgsom_b200 import SomClassifier, SomVQ
from oracle import som_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))


def oracle_cls(cls, **attrs):
    return type(cls.__name__, (cls,), {"_make_engine": lambda self, distributed=None: OracleEngine(), **attrs})


def fit(cls, X, y=None, w=None, **kw):
    kw.setdefault("random_state", 0)
    kw.setdefault("n_iter", 20)
    est = oracle_cls(cls)(**kw)
    return est.fit(X, y, sample_weight=w) if w is not None else est.fit(X, y)


def assert_same_fit(a, b, exact=True):
    assert list(a.neurons_) == list(b.neurons_) and a.n_iter_ == b.n_iter_
    if exact:
        np.testing.assert_array_equal(a.weights_, b.weights_)
        assert a.quantization_error_ == b.quantization_error_ and a.topographic_error_ == b.topographic_error_
    else:
        np.testing.assert_allclose(a.weights_, b.weights_, rtol=1e-9, atol=1e-9)
        assert a.quantization_error_ == pytest.approx(b.quantization_error_, rel=1e-9)
        assert a.topographic_error_ == pytest.approx(b.topographic_error_, rel=1e-9, abs=1e-12)


@pytest.fixture(scope="module")
def blobs():
    X = _datasets.gmm(600, 6, 5, 3).astype(np.float64)
    y = np.arange(len(X)) % 3
    return X, y


@pytest.mark.parametrize("bad,match", [
    (lambda n: -np.ones(n), "(?i)negative"),
    (lambda n: np.where(np.arange(n) == 3, np.nan, 1.0), "NaN|finite"),
    (lambda n: np.where(np.arange(n) == 3, np.inf, 1.0), "infinity|finite"),
    (lambda n: np.ones(n - 1), "shape|length|samples"),
    (lambda n: (np.arange(n) < 3).astype(float), "at least 4"),
], ids=["negative", "nan", "inf", "length", "three_positive"])
def test_bad_weights_raise(blobs, bad, match):
    X, y = blobs
    with pytest.raises(ValueError, match=match):
        fit(SomVQ, X, w=bad(len(X)))
    with pytest.raises(ValueError, match=match):
        fit(SomClassifier, X, y, w=bad(len(X)))


@pytest.mark.parametrize("cls", [SomVQ, SomClassifier])
def test_unit_weights_are_the_unweighted_fit(blobs, cls):
    X, y = blobs
    yy = y if cls is SomClassifier else None
    a, b = fit(cls, X, yy), fit(cls, X, yy, np.ones(len(X)))
    # the oracle's weighted sums take another order than its unweighted ones (the device kernels agree bit for bit)
    assert_same_fit(a, b, exact=False)
    np.testing.assert_array_equal(a._extract_values_from_graph("hit_count"), b._extract_values_from_graph("hit_count"))
    if cls is SomVQ:
        np.testing.assert_array_equal(a.labels_, b.labels_)
    else:
        np.testing.assert_array_equal(a._extract_values_from_graph("label"), b._extract_values_from_graph("label"))


@pytest.mark.parametrize("cls,criterion", [(SomVQ, "quantization_error"), (SomClassifier, "entropy")])
def test_zero_one_weights_are_the_subset_fit(blobs, cls, criterion):
    X, y = blobs
    keep = np.random.default_rng(1).random(len(X)) < 0.6
    yy = y if cls is SomClassifier else None
    a = fit(cls, X, yy, keep.astype(float), growth_criterion=criterion)
    b = fit(cls, X[keep], None if yy is None else yy[keep], growth_criterion=criterion)
    assert_same_fit(a, b, exact=False)
    if cls is SomVQ:
        np.testing.assert_array_equal(a.labels_[keep], b.labels_)
        assert a.labels_.shape == (len(X),)  # zero-weight rows still get their winner
    else:
        np.testing.assert_array_equal(a._extract_values_from_graph("label"), b._extract_values_from_graph("label"))
        np.testing.assert_allclose(a._extract_values_from_graph("probabilities"),
                                   b._extract_values_from_graph("probabilities"), rtol=1e-12)


@pytest.mark.parametrize("cls", [SomVQ, SomClassifier])
def test_integer_weights_are_repeated_rows(blobs, cls):
    X, y = blobs
    w = np.random.default_rng(2).integers(1, 4, len(X))
    rep = np.repeat(np.arange(len(X)), w)
    # the two fits draw their start rows from different row counts: start both from the same four samples
    start = np.array([5, 100, 333, 599])

    def weighted_rows(self, n_samples, sample_weight, engine):
        return start

    def repeated_rows(self, n_samples, sample_weight, engine):
        return (np.cumsum(w) - w)[start]  # first copy of each start sample

    yy = y if cls is SomClassifier else None
    a = oracle_cls(cls, _start_rows=weighted_rows)(random_state=0, n_iter=20).fit(X, yy, sample_weight=w)
    b = oracle_cls(cls, _start_rows=repeated_rows)(random_state=0, n_iter=20).fit(
        X[rep], None if yy is None else yy[rep])
    assert_same_fit(a, b, exact=False)
    np.testing.assert_allclose(a._extract_values_from_graph("hit_count"), b._extract_values_from_graph("hit_count"))
    if cls is SomVQ:
        np.testing.assert_array_equal(a.labels_[rep], b.labels_)


def test_start_rows_skip_zero_weights_and_match_the_unweighted_draw(blobs):
    X, _ = blobs
    est = oracle_cls(SomVQ)(random_state=4)
    est._comm = None
    eng = OracleEngine()
    n = len(X)
    drawn = est._start_rows(n, None, eng)
    np.testing.assert_array_equal(est._start_rows(n, np.full(n, 0.5), eng), drawn)
    w = np.zeros(n)
    w[::3] = 1.0
    rows = est._start_rows(n, w, eng)
    assert (w[rows] > 0).all()
    np.testing.assert_array_equal(rows, np.flatnonzero(w > 0)[np.random.default_rng(4).choice(w.astype(bool).sum(), 4,
                                                                                            replace=False)])


def test_fit_predict_fit_transform_and_pipeline_forward_the_weights(blobs):
    from sklearn.pipeline import make_pipeline
    from sklearn.preprocessing import StandardScaler

    X, y = blobs
    w = np.random.default_rng(3).uniform(0.0, 2.0, len(X))
    Est = oracle_cls(SomVQ)
    ref = Est(random_state=0, n_iter=15).fit(X, sample_weight=w)
    np.testing.assert_array_equal(Est(random_state=0, n_iter=15).fit_predict(X, sample_weight=w), ref.labels_)
    np.testing.assert_allclose(Est(random_state=0, n_iter=15).fit_transform(X, sample_weight=w), ref.transform(X))
    assert ref.calculate_quantization_error(X, sample_weight=np.ones(len(X))) == pytest.approx(
        ref.calculate_quantization_error(X), rel=1e-12)
    dist = np.linalg.norm(X - ref.weights_[ref.predict(X)], axis=1)
    assert ref.calculate_quantization_error(X, sample_weight=w) == pytest.approx(np.average(dist, weights=w), rel=1e-9)

    Clf = oracle_cls(SomClassifier)
    pipe = make_pipeline(StandardScaler(), Clf(random_state=0, n_iter=15))
    pipe.fit(X, y, somclassifier__sample_weight=w)
    direct = Clf(random_state=0, n_iter=15).fit(StandardScaler().fit_transform(X), y, sample_weight=w)
    np.testing.assert_array_equal(pipe[-1].weights_, direct.weights_)


def test_weighted_oracle_pieces_equal_repeated_rows(blobs):
    X, _ = blobs
    w = np.random.default_rng(6).integers(0, 4, len(X)).astype(np.float64)
    rep = np.repeat(X, w.astype(np.int64), axis=0)
    assert WO.total_variance(X, w) == pytest.approx(O.total_variance(rep), rel=1e-12)
    assert WO.growing_threshold(X, freq_weight=w) == pytest.approx(O.growing_threshold(rep), rel=1e-12)
    W = X[:9]
    hop = O.hop_matrix_grid(3, 3)
    a = WO.epoch_step(X, W, hop, 1.5, WO.total_variance(X, w), freq_weight=w)
    b = O.epoch_step(rep, W, hop, 1.5, WO.total_variance(X, w))
    for key in ("Sk", "sk", "n", "E", "W_new"):
        np.testing.assert_allclose(a[key], b[key], rtol=1e-12, atol=1e-12)
    # default None: the unweighted oracle, bit for bit
    assert WO.total_variance(X, None) == O.total_variance(X)
    np.testing.assert_array_equal(O.epoch_step(X, W, hop, 1.5, 2.0)["W_new"],
                                  WO.epoch_step(X, W, hop, 1.5, 2.0, freq_weight=None)["W_new"])


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _weights(n):
    w = np.random.default_rng(8).uniform(0.0, 2.0, n)
    w[::5] = 0.0
    return w


def _gloo_worker(rank, world, port, kind, out_dir):
    sys.path[:0] = [os.path.dirname(HERE), HERE]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist

    import _datasets as ds
    from _weighted_oracle import WeightedOracleEngine as OE
    from _weighted_oracle import WeightedShardedOracleEngine as ShardedOracleEngine
    from dbgsom_b200 import SomClassifier as Clf
    from dbgsom_b200 import SomVQ as VQ
    from dbgsom_b200.engine import Comm

    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        comm = Comm(True)
        X, y = ds.load("digits")
        w = _weights(len(X))
        lo, hi = rank * len(X) // world, (rank + 1) * len(X) // world

        def factory(self, distributed=None):
            return ShardedOracleEngine(comm) if distributed is not False else OE()

        cls = VQ if kind == "vq" else Clf
        est = type(cls.__name__, (cls,), {"_make_engine": factory})(random_state=0, n_iter=20, distributed=True)
        est.fit(X[lo:hi], None if kind == "vq" else y[lo:hi], sample_weight=w[lo:hi])
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), neurons=np.array(est.neurons_), weights=est.weights_,
                 qe=est.quantization_error_, te=est.topographic_error_, hits=est._extract_values_from_graph("hit_count"),
                 labels=est._extract_values_from_graph("label"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("kind", ["vq", "clf"])
def test_two_gloo_ranks_with_weighted_shards_equal_one_process(tmp_path, kind):
    import torch.multiprocessing as mp

    mp.spawn(_gloo_worker, args=(2, _free_port(), kind, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    for key in ("neurons", "weights", "qe", "te", "hits", "labels"):
        np.testing.assert_array_equal(r0[key], r1[key])
    X, y = _datasets.load("digits")
    one = fit(SomVQ if kind == "vq" else SomClassifier, X, None if kind == "vq" else y, _weights(len(X)))
    np.testing.assert_array_equal(r0["neurons"], np.array(one.neurons_))
    np.testing.assert_allclose(r0["weights"], one.weights_, rtol=1e-9, atol=1e-9)
    assert float(r0["qe"]) == pytest.approx(one.quantization_error_, rel=1e-9)
    assert float(r0["te"]) == pytest.approx(one.topographic_error_, rel=1e-9, abs=1e-12)
    np.testing.assert_allclose(r0["hits"], one._extract_values_from_graph("hit_count"), rtol=1e-12)
    np.testing.assert_array_equal(r0["labels"], one._extract_values_from_graph("label"))
