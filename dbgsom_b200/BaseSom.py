"""Host driver of the B200 batch-SOM: same estimator surface as the reference's `BaseSom`.

Mirrors `dbgsom/BaseSom.py` of SandroMartens/DBGSOM at the API level (constructor
keywords :42-80, `fit` :88-131, fitted attributes, `transform`, metrics) while the numeric
epoch (:394-407) runs on the GPU through `dbgsom_b200.engine.DeviceEngine` (ctypes ->
`libdbgsom_b200.so`, hand-written sm_100a kernels).  There is no CPU fallback: without the
CUDA library and a device, `fit` raises.

What stays on the host, as in the reference: the growing-map logic (`topology.py`), the
sigma schedule, thresholds, early stopping, and the fitted NetworkX graph `som_`.
"""

from __future__ import annotations

import os
import time
from math import exp, log, sqrt
from typing import Any

import numpy as np
from sklearn.base import BaseEstimator
from sklearn.utils import check_array, check_random_state
from sklearn.utils.validation import _check_sample_weight, check_is_fitted

from .topology import MapTopology

__all__ = ["BaseSom", "sigma_linear", "sigma_exponential"]


def sigma_linear(sigma_start, sigma_end, max_iter, current_iter, learning_rate=None):
    """Same contract as `linear_decay`, dbgsom/BaseSom.py:1001-1012."""
    frac = current_iter / max_iter
    return sigma_start * (1 - frac) + sigma_end * frac


def sigma_exponential(sigma_start, sigma_end, max_iter, current_iter, learning_rate):
    """Same contract as `exponential_decay`, dbgsom/BaseSom.py:1015-1025."""
    return sigma_end + (sigma_start - sigma_end) * exp(-learning_rate * current_iter)


class BaseSom(BaseEstimator):
    """Shared training driver of `SomVQ` and `SomClassifier`.

    Hyper-parameters are those of the reference (same names, defaults and meaning,
    including the spelling `convergence_treshold`); the trailing ones are additions:

    device : str, default "cuda"
        CUDA device the epoch kernels run on.
    compat_pack_rows : bool, default True
        Reproduce the reference's packed centre rows (SURVEY.md quirk Q1).  False gives
        the index-aligned batch update.
    bmu_backend : {"auto", "tensor", "simt"}, default "auto"
        "tensor" = tcgen05 fp16 candidate search + exact float64 re-score of the candidates,
        "simt" = fp32 CUDA-core candidate search (proven rounding bound) + the same re-score.
        The tensor search keeps every prototype inside an error bound around the best approximate
        score.  By default that bound is a CALIBRATED fraction of the Cauchy-Schwarz worst case
        (rounding errors of 2D products do not align; csrc/common.cuh, tools/calibrate_bound.py), and a
        sample with more candidates than the table holds is accepted without a full re-scan when
        its best two approximate scores are provably inside the 1e-6 near-tie gate.  Winners
        therefore equal the float64 reference outside that gate in every measured case, but only
        `bound_scale=1.0, strict_ties=True` makes it a guarantee.
    bound_scale : float, default 0.0
        Coefficient of the tensor search's rounding bound relative to the worst case; 0 selects the
        calibrated default, 1.0 the worst case (more samples re-scored, same winners).
    strict_ties : bool, default False
        Re-score samples whose candidate table overflowed against ALL prototypes in float64 instead of
        accepting provable near-ties.  The post-training passes (`labels_`, hit counts, errors)
        always run in this mode.
    distributed : bool, default False
        SPMD multi-GPU: every rank calls `fit` with its own shard of the samples; only the
        per-neuron partial sums are all-reduced each epoch (`torch.distributed`, NCCL).  The start
        rows are drawn on rank 0 and broadcast, and `classes_` is the union over all shards.

    `fit(X, y, sample_weight)` takes frequency weights like scikit-learn's `KMeans`: a sample of integer
    weight w counts like w copies of it (fractional weights extend the same sums), zero removes it from
    every sum of the fit while it still gets a winner in `labels_`.  The start prototypes are drawn among
    the samples with positive weight.
    """

    def __init__(
        self,
        n_iter: int = 200,
        convergence_iter: int = 1,
        spreading_factor: float = 0.5,
        sigma_start: float | None = None,
        sigma_end: float | None = None,
        vertical_growth: bool = False,
        decay_function: str = "exponential",
        learning_rate: float = 0.02,
        verbose: bool = False,
        coarse_training_frac: float = 0.5,
        random_state: Any = None,
        convergence_treshold: float = 10**-5,
        max_neurons: int = 100,
        metric: str = "euclidean",
        threshold_method: str = "se",
        growth_criterion: str = "quantization_error",
        min_samples_vertical_growth: int = 100,
        n_jobs: int = 1,
        device: str = "cuda",
        compat_pack_rows: bool = True,
        bmu_backend: str = "auto",
        distributed: bool = False,
        bound_scale: float = 0.0,
        strict_ties: bool = False,
    ) -> None:
        self.spreading_factor = spreading_factor
        self.n_iter = n_iter
        self.convergence_iter = convergence_iter
        self.sigma_start = sigma_start
        self.sigma_end = sigma_end
        self.decay_function = decay_function
        self.learning_rate = learning_rate
        self.verbose = verbose
        self.coarse_training_frac = coarse_training_frac
        self.random_state = random_state
        self.convergence_treshold = convergence_treshold
        self.max_neurons = max_neurons
        self.metric = metric
        self.threshold_method = threshold_method
        self.growth_criterion = growth_criterion
        self.min_samples_vertical_growth = min_samples_vertical_growth
        self.vertical_growth = vertical_growth
        self.n_jobs = n_jobs
        self.device = device
        self.compat_pack_rows = compat_pack_rows
        self.bmu_backend = bmu_backend
        self.distributed = distributed
        self.bound_scale = bound_scale
        self.strict_ties = strict_ties

    # ------------------------------------------------------------------ hooks for subclasses
    def _check_input_data(self, X, y):
        raise NotImplementedError

    def _label_prototypes(self, y, engine) -> None:
        raise NotImplementedError

    def _fit(self, engine) -> None:
        pass

    def predict(self, X):
        raise NotImplementedError

    # ------------------------------------------------------------------ engine plumbing
    def _make_engine(self, distributed: bool | None = None):
        """Create the device engine (the only place one is made).

        CPU-only unit tests of the host logic replace this factory with a checker; the
        product path has no alternative to the CUDA engine.
        """
        from .engine import DeviceEngine

        return DeviceEngine(
            device=self.device,
            bmu_backend=self.bmu_backend,
            distributed=self.distributed if distributed is None else distributed,
            bound_scale=self.bound_scale,
            strict_ties=self.strict_ties,
            capacity_hint=self._capacity_hint(),
        )

    def _check_arguments(self) -> None:
        # The reference declares these checks (dbgsom/BaseSom.py:143-155) but never calls
        # them; invalid values would fail later with obscure errors, so they are enforced.
        if self.decay_function not in ("linear", "exponential"):
            raise ValueError("Decay function not supported. Must be 'linear' or 'exponential'.")
        if self.threshold_method not in ("se", "classical"):
            raise ValueError("threshold_method not supported. Must be 'se' or 'classical'.")
        if self.growth_criterion not in ("quantization_error", "entropy"):
            raise ValueError("growth_criterion not supported. Must be 'quantization_error' or 'entropy'.")
        if self.vertical_growth:
            # The reference's vertical growth raises TypeError on every call (quirk Q11).
            raise NotImplementedError("vertical_growth is not supported (broken in the reference, out of scope)")

    # ------------------------------------------------------------------ fit
    def fit(self, X, y=None, sample_weight=None):
        """Train the map on X (and y).  Same contract as dbgsom/BaseSom.py:88-131.

        sample_weight : array of shape (n_samples,), default None
            Frequency weights (finite, >= 0, at least four positive); None weighs every sample 1.
        """
        self._check_arguments()
        X, y = self._check_input_data(X, y)
        if sample_weight is not None:
            sample_weight = self._check_sample_weight(sample_weight, X)
        if y is None and self.growth_criterion == "entropy":
            # the reference indexes `y[winners == j]` with y = None here (dbgsom/BaseSom.py:547-551) and dies with
            # a TypeError in the first epoch; say what is wrong instead of silently growing on another criterion
            raise ValueError("growth_criterion='entropy' needs class labels y (use SomClassifier)")
        self.random_state_ = check_random_state(self.random_state)
        engine = self._make_engine()
        comm = getattr(engine, "comm", None)
        self._comm = comm if comm is not None and getattr(comm, "enabled", False) and comm.world > 1 else None
        if y is not None:
            classes = np.unique(y)
            if self._comm is not None:
                # shards may hold different class sets: every rank must use the same index <-> class map (and the
                # same histogram width in the collectives)
                classes = self._comm.union_sorted(classes)
            y = np.searchsorted(classes, y)
            self.classes_ = np.array(classes)
        profile = os.environ.get("DBGSOM_PROFILE") == "1"  # wall time per stage + device time per kernel phase
        if profile and hasattr(engine, "enable_profiling"):
            engine.enable_profiling(True)
        self._host_growth_s = 0.0
        self._host_hops_s = 0.0
        try:
            t0 = time.perf_counter()
            self._initialize_som(engine, X, y, sample_weight)
            t1 = time.perf_counter()
            self._grow_som(engine)
            t2 = time.perf_counter()
            self._finalize(engine, y)
            t3 = time.perf_counter()
            if profile:
                self.fit_profile_ = {
                    "initialize_s": t1 - t0, "epochs_s": t2 - t1, "finalize_s": t3 - t2,
                    "host_growth_s": self._host_growth_s, "hops_s": self._host_hops_s,
                    "finalize": {k: float(v) for k, v in self._finalize_profile.items()},
                }
                if hasattr(engine, "phase_times_ms"):
                    self.fit_profile_["device_ms"] = {k: round(float(np.sum(v)), 2) for k, v in engine.phase_times_ms().items()}
        finally:
            engine.close()
            self._comm = None
        self.n_features_in_ = X.shape[1]
        self.n_iter_ = self._current_epoch
        return self

    @staticmethod
    def _check_sample_weight(sample_weight, X) -> np.ndarray:
        """float64 weights of the rows of X: the right length, finite and non-negative."""
        w = _check_sample_weight(sample_weight, X, dtype=np.float64, ensure_non_negative=True,
                                 allow_all_zero_weights=True)
        if not np.isfinite(w).all():
            raise ValueError("sample_weight must be finite")
        return np.ascontiguousarray(w, dtype=np.float64)

    def _initialize_som(self, engine, X: np.ndarray, y, sample_weight=None) -> None:
        """`_initialize_som` + `_create_som`, dbgsom/BaseSom.py:352-369, :419-444."""
        self._current_epoch = 0
        self.converged_ = False
        self._training_phase = "coarse"
        self._neurons_added = True
        n_classes = len(self.classes_) if y is not None else 0
        if sample_weight is None:
            stats = engine.load_data(X, y, n_classes)
        else:
            stats = engine.load_data(X, y, n_classes, sample_weight=sample_weight)
        # the amount of data the error means are taken over: the total weight of a weighted fit
        self._n_total = stats.get("total_weight")
        self._total_variance = stats["total_variance"]
        self.growing_threshold_ = self._growing_threshold(stats, X.shape[1])
        rows = self._start_rows(stats["n_samples"], sample_weight, engine)
        self._topology = MapTopology.initial_square()
        engine.init_map_from_rows(rows, capacity=self._capacity_hint())
        self._hops_dirty = True

    def _start_rows(self, n_samples: int, sample_weight, engine) -> np.ndarray:
        """Global sample indices of the four start prototypes (dbgsom/BaseSom.py:423-430).

        Unweighted: the draw of `rng.choice(a=data, size=4, replace=False)` (row choice).  Weighted: the same draw
        over the rows with positive weight (in global order), so zero-weight rows never become prototypes and
        all-positive weights give exactly the unweighted rows.  When sharded, rank 0 draws and every rank
        resolves the positions that fall into its own shard; the others are -1 (owned by another rank)."""
        rng = np.random.default_rng(seed=self.random_state)
        if sample_weight is None:
            rows = rng.choice(n_samples, size=4, replace=False)
            if self._comm is not None:
                # an unseeded (or per-rank different) generator would give every rank its own four rows
                rows = np.asarray(self._comm.broadcast_object(rows, src=0))
            return rows
        positive = np.flatnonzero(sample_weight > 0)
        pos_offset, n_pos = 0, positive.size
        if self._comm is not None:
            pos_offset, n_pos = self._comm.exclusive_offset(positive.size, getattr(self._comm, "device", None))
        if n_pos < 4:
            raise ValueError(f"sample_weight has {n_pos} positive entries; at least 4 are needed (one per start prototype)")
        pick = rng.choice(n_pos, size=4, replace=False)
        if self._comm is not None:
            pick = np.asarray(self._comm.broadcast_object(pick, src=0))
        local = pick - pos_offset
        own = (local >= 0) & (local < positive.size)
        return np.where(own, positive[np.where(own, local, 0)] + getattr(engine, "sample_offset", 0), -1)

    def _capacity_hint(self) -> int:
        # growth is only tested before a growth step (quirk Q8) so the map can overshoot
        # max_neurons by up to one boundary ring; the engine re-allocates if exceeded.
        return int(max(16, 2 * self.max_neurons + 64))

    def _growing_threshold(self, stats: dict, n_dim: int) -> float:
        """`_calculate_growing_threshold`, dbgsom/BaseSom.py:371-385."""
        if self.growth_criterion == "entropy":
            return self.spreading_factor
        if self.threshold_method == "classical":
            return -n_dim * log(self.spreading_factor)
        return float(150 * -log(self.spreading_factor) * stats["std_norm"])

    def _current_sigma(self) -> float:
        """`_calculate_current_sigma`, dbgsom/BaseSom.py:863-902."""
        m = len(self._topology)
        start = 0.2 * sqrt(m) if self.sigma_start is None else self.sigma_start
        end = max(0.7, 0.05 * sqrt(m)) if self.sigma_end is None else self.sigma_end
        if self._training_phase != "coarse":
            return end
        decay = sigma_linear if self.decay_function == "linear" else sigma_exponential
        return decay(
            sigma_start=start,
            sigma_end=end,
            max_iter=self.n_iter,
            current_iter=self._current_epoch / self.coarse_training_frac,
            learning_rate=self.learning_rate,
        )

    def _grow_som(self, engine) -> None:
        """Epoch loop -- dbgsom/BaseSom.py:387-417."""
        topo = self._topology
        epochs = range(self.n_iter)
        if self.verbose:
            from tqdm import tqdm

            epochs = tqdm(epochs, unit=" epochs")
        use_entropy = self.growth_criterion == "entropy"
        for epoch in epochs:
            self._current_epoch = epoch
            if epoch > self.coarse_training_frac * self.n_iter:
                self._training_phase = "fine"
            if self._hops_dirty:
                # the reference recomputes all-pairs hops every epoch (quirk Q3); they only
                # change when the map grew
                th = time.perf_counter()
                engine.set_hops_from_topology(topo)
                self._host_hops_s += time.perf_counter() - th
                self._hops_dirty = False
            result = engine.epoch(
                sigma=self._current_sigma(),
                pack_rows=self.compat_pack_rows,
                entropy_error=use_entropy,
            )
            topo.error[:] = result["error"]
            if not np.isfinite(result["change"]):
                # A neuron farther than ~38 sigma hops from every live one gets 0/0 prototypes (SURVEY.md
                # quirk Q10); the reference then fails in its next `kneighbors` call with the same error.
                raise ValueError("Input X contains NaN (a prototype became NaN during neighbourhood smoothing).")
            if result["change"] < self.convergence_treshold:
                self.converged_ = True  # a latch, like the reference (quirk Q7)
            if self.converged_ and self._training_phase == "fine":
                break
            if (
                self._training_phase == "coarse"
                and len(topo) < self.max_neurons
                and epoch % self.convergence_iter == self.convergence_iter - 1
            ):
                tg = time.perf_counter()
                topo.distribute_errors(self.growing_threshold_)
                ops = topo.grow(self.growing_threshold_, epoch)
                if ops:
                    engine.apply_row_ops(ops, n_rows=len(topo))
                    self._hops_dirty = True
                    self._max_map_size = max(getattr(self, "_max_map_size", 0), len(topo))  # before dead-neuron removal
                self._host_growth_s += time.perf_counter() - tg

    # ------------------------------------------------------------------ after the loop
    def _finalize(self, engine, y) -> None:
        """Everything `fit` does after `_grow_som` (dbgsom/BaseSom.py:116-127).

        The reference runs four to five separate BMU passes with Python loops over the samples here
        (topographic error, quantisation error, node statistics, classifier labelling, `labels_`).
        Two BMU searches on the device feed all of them (a top-2 pass on the pre-update prototypes,
        a top-1 pass on the final reduced map) and the per-sample reductions run on the device too
        (`engine.final_statistics`, `engine.label_histogram`); only per-neuron vectors come back.
        """
        topo = self._topology
        tf = [time.perf_counter()]
        # Quirk kept for parity: after the loop the reference's `weights_` / `neurons_` still
        # hold the state from the START of the last epoch (they are refreshed at the top of
        # the loop body, dbgsom/BaseSom.py:397-401), so topographic error, quantisation
        # error and node statistics are measured against the prototypes BEFORE the final
        # update, while the graph (and the final `weights_`) carry the updated ones.
        st = engine.final_statistics(topo.positions(), topo.degrees())
        n_total = engine.n_samples_global if self._n_total is None else self._n_total
        tf.append(time.perf_counter())
        # topographic error: grid distance of the two BMUs > 1.5 (dbgsom/BaseSom.py:924-953)
        self.topographic_error_ = st["te_count"] / n_total
        self.quantization_error_ = st["qe_sum"] / n_total

        # node statistics (dbgsom/BaseSom.py:181-221)
        m = len(topo)
        if st["n_rows"] != m:
            raise RuntimeError(
                "the map grew in the final epoch (coarse_training_frac >= 1); the reference "
                "fails in this configuration as well (hit_count missing on the new nodes)"
            )
        weights, avg_dist, hits = st["weights"], st["avg_dist"], st["hits"]
        with np.errstate(divide="ignore", invalid="ignore"):
            density = np.where(hits > 0, st["dens_sum"] / hits, 0.0)

        # neurons without samples leave the map (dbgsom/BaseSom.py:223-235)
        dead = np.flatnonzero(hits == 0)
        alive = np.flatnonzero(hits > 0)
        attrs = {
            "weight": list(weights),
            "density": list(density),
            "hit_count": list(hits),
            "average_distance": list(avg_dist),
        }
        graph = topo.to_networkx(attrs)
        graph.remove_nodes_from([topo.pos[i] for i in dead])
        self.som_ = graph
        self._topology = topo.without(dead)
        self.neurons_ = list(graph.nodes)
        self.weights_ = weights[alive]
        self._distance_matrix_cache = None  # all-pairs hops of the reduced map: built on first use (`_distance_matrix`)

        # prototype labels and `labels_` use the UPDATED, reduced map (dbgsom/BaseSom.py:121,
        # :127; SomVQ.py:150-152; SomClassifier.py:130-152): one more BMU pass, kept on the device
        tf.append(time.perf_counter())
        engine.keep_rows(alive)
        engine.final_winners()
        tf.append(time.perf_counter())
        self._label_prototypes(y, engine)
        self._fit(engine)
        tf.append(time.perf_counter())
        self._finalize_profile = dict(zip(("statistics_s", "graph_s", "final_winners_s", "labels_s"), np.diff(tf).round(4)))

    @property
    def _distance_matrix(self) -> np.ndarray:
        """All-pairs hop counts of the fitted map, float64 with inf between components -- the reference's
        `_distance_matrix` (dbgsom/BaseSom.py:235).  Nothing in `fit`/`predict`/`transform` reads it, and it
        is M x M float64 (2 GB at 16k neurons), so it is built on first access instead of inside `fit`."""
        if getattr(self, "_distance_matrix_cache", None) is None:
            self._distance_matrix_cache = self._topology.hop_matrix()
        return self._distance_matrix_cache

    @_distance_matrix.setter
    def _distance_matrix(self, value) -> None:
        self._distance_matrix_cache = value

    # ------------------------------------------------------------------ inference helpers
    def _get_winning_neurons(self, data, n_bmu: int):
        """Distances and indices of the `n_bmu` best matching prototypes per sample.

        Same return shapes as dbgsom/BaseSom.py:446-464; computed on the device.
        """
        engine = self._make_engine(distributed=False)
        try:
            dist, idx = engine.bmu(np.asarray(data), self.weights_, n_bmu)
        finally:
            engine.close()
        if n_bmu == 1:
            return dist.reshape(-1), idx.reshape(-1)
        return dist, idx

    def _extract_values_from_graph(self, attribute: str) -> np.ndarray:
        """Node attribute as an array in node order (dbgsom/BaseSom.py:237-239)."""
        return np.array([data[attribute] for _, data in self.som_.nodes.data()])

    def calculate_quantization_error(self, X, sample_weight=None) -> float:
        """Mean distance to the nearest prototype (dbgsom/BaseSom.py:904-922); weighted mean with `sample_weight`."""
        check_is_fitted(self)
        X = check_array(X)
        if sample_weight is not None:
            sample_weight = self._check_sample_weight(sample_weight, X)
        dist, _ = self._get_winning_neurons(X, n_bmu=1)
        if sample_weight is None:
            return float(np.mean(dist))
        return float(np.average(dist, weights=sample_weight))

    def transform(self, X, y=None) -> np.ndarray:
        """Non-negative sparse code of each sample over the normalised prototypes.

        Same result as dbgsom/BaseSom.py:241-268 (scikit-learn `SparseCoder`, `lasso_lars`, positive, alpha 0)
        computed on the device: the LARS-lasso path of every sample runs in `dbgsom_sparse_code`
        (csrc/lars_core.cuh restates scikit-learn's solver; SURVEY.md section 8(f) rank 3).

        The path is evaluated in float64 for float64 and float32 samples alike.  For float32 samples
        scikit-learn casts the Gram matrix to float32 and runs the Cholesky part of the path in float32
        (`_sparse_encode`), so on ill-conditioned maps the reference's own codes carry float32 noise (up to
        ~1e-3 on a smooth 400-neuron sheet); this implementation returns the float64 result there.
        """
        from sklearn.preprocessing import normalize

        check_is_fitted(self)
        X = check_array(X, dtype=[np.float64, np.float32])
        engine = self._make_engine(distributed=False)
        try:
            return engine.sparse_code(normalize(X), normalize(self.weights_))
        finally:
            engine.close()
