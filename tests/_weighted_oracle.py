"""TEST-ONLY: frequency weights (`sample_weight` of fit) on top of the CPU oracle.

`freq_weight` ([N] float64, >= 0) makes a sample of integer weight w count like w copies of it, so every result equals
the unweighted oracle on `np.repeat(X, w, axis=0)` up to summation order.  It is not the reference's `sample_weights`
(the per-sample similarity k_i, `oracle.som_oracle.sample_weights`).  The functions and engines here build on
`oracle.som_oracle` and `_oracle_engine` without changing them; with `freq_weight=None` / no weights they call the
unweighted code.
"""
import numpy as np

from _oracle_engine import OracleEngine, ShardedOracleEngine
from dbgsom_b200.hostmath import class_entropy
from oracle import som_oracle as O


def weighted_sq_dev(X, w) -> np.ndarray:
    """Per column sum_i w_i (x_id - mu_d)^2 about the weighted mean (float64)."""
    X = np.asarray(X, dtype=np.float64)
    w = np.asarray(w, dtype=np.float64)
    mu = (w @ X) / w.sum()
    return w @ ((X - mu) ** 2)


def total_variance(X, freq_weight=None) -> float:
    """dbgsom/BaseSom.py:363 weighted: sum_d sum_i w_i (x_id - mu_d)^2 / sum_i w_i."""
    if freq_weight is None:
        return O.total_variance(X)
    return float(weighted_sq_dev(X, freq_weight).sum() / np.sum(freq_weight))


def std_norm(X, freq_weight) -> float:
    """|| std(X, axis=0, ddof=1) ||_2 with the weighted std sqrt(sum_i w_i (x_id - mu_d)^2 / (sum_i w_i - 1))."""
    return float(np.linalg.norm(np.sqrt(weighted_sq_dev(X, freq_weight) / (np.sum(freq_weight) - 1))))


def growing_threshold(X, spreading_factor=0.5, threshold_method="se", growth_criterion="quantization_error",
                      freq_weight=None) -> float:
    """dbgsom/BaseSom.py:371-385 with the weighted std of the 'se' method."""
    if freq_weight is None or growth_criterion == "entropy" or threshold_method == "classical":
        return O.growing_threshold(X, spreading_factor, threshold_method, growth_criterion)
    return float(150 * -np.log(spreading_factor) * std_norm(X, freq_weight))


def voronoi_sums(k, X, winners, M, freq_weight=None):
    """Sk_j = sum w_i k_i x_i, sk_j = sum w_i k_i, n_j = sum w_i."""
    if freq_weight is None:
        return O.voronoi_sums(k, X, winners, M)
    Sk, sk, _ = O.voronoi_sums(np.asarray(k, dtype=np.float64) * freq_weight, X, winners, M)
    return Sk, sk, np.bincount(winners, weights=freq_weight, minlength=M).astype(np.float64)


def quantization_errors(winners, dist, M, freq_weight=None):
    """E_j = sum w_i d_i."""
    if freq_weight is None:
        return O.quantization_errors(winners, dist, M)
    return O.quantization_errors(winners, np.asarray(dist, dtype=np.float64) * freq_weight, M)


def epoch_step(X, W, hop, sigma, total_var, pack=True, winners=None, freq_weight=None) -> dict:
    """`oracle.som_oracle.epoch_step` with frequency weights (a neuron is live iff its weight sum is positive);
    `winners` teacher-forces the BMUs as there.  `k` is returned unweighted."""
    if freq_weight is None:
        return O.epoch_step(X, W, hop, sigma, total_var, pack=pack, winners=winners)
    W = np.asarray(W, dtype=np.float64)
    M = W.shape[0]
    if winners is None:
        dist, winners = O.bmu(X, W, 1)
    else:
        winners = np.asarray(winners, dtype=np.int64)
        dist = O.expansion_distance(X, W, winners)
    k = O.sample_weights(dist, total_var)
    Sk, sk, n = voronoi_sums(k, X, winners, M, freq_weight)
    live = np.flatnonzero(n > 0)
    C = np.zeros_like(Sk)
    with np.errstate(divide="ignore", invalid="ignore"):
        centres = Sk[live] / sk[live][:, None]
    if pack:
        C[: live.size] = centres
    else:
        C[live] = centres
    E = quantization_errors(winners, dist, M, freq_weight)
    W_new = O.smooth(C, n, O.neighborhood(hop, sigma))
    change = float(np.sum(np.linalg.norm(W - W_new, axis=1)))
    return dict(winners=winners, dist=dist, k=k, Sk=Sk, sk=sk, n=n, C=C, E=E, W_new=W_new, change=change)


class WeightedOracleEngine(OracleEngine):
    """`OracleEngine` that also takes `load_data(..., sample_weight=w)`; without weights it is `OracleEngine`."""

    w = None

    def load_data(self, X, y, n_classes, sample_weight=None):
        self.w = None
        if sample_weight is None:
            return super().load_data(X, y, n_classes)
        self.X, self.y, self.n_classes = X, y, n_classes
        self.n_samples_global = X.shape[0]
        self.w = np.asarray(sample_weight, dtype=np.float64)
        self.total_var = total_variance(X, self.w)
        return {"n_samples": X.shape[0], "total_variance": self.total_var, "std_norm": std_norm(X, self.w),
                "total_weight": float(self.w.sum())}

    def _hist(self, winners, y, m, n_classes):
        return np.bincount(winners * n_classes + y, weights=self.w, minlength=m * n_classes)

    def epoch(self, sigma, pack_rows, entropy_error):
        if self.w is None:
            return super().epoch(sigma, pack_rows, entropy_error)
        out = epoch_step(self.X, self.W, self.hop, sigma, self.total_var, pack=pack_rows, freq_weight=self.w)
        self.W_prev, self.W = self.W, out["W_new"]
        self.epochs += 1
        err = out["E"]
        if entropy_error:
            m = self.W.shape[0]
            err = class_entropy(self._hist(out["winners"], self.y, m, self.n_classes).reshape(m, self.n_classes))
        return {"error": err, "counts": out["n"], "change": out["change"]}

    def final_statistics(self, positions, degrees):
        if self.w is None:
            return super().final_statistics(positions, degrees)
        from scipy.spatial.distance import cdist

        dist2, idx2 = self.bmu_train(2, previous=True)
        m = self.W_prev.shape[0]
        pos = np.asarray(positions, dtype=np.float64)
        sep = pos[idx2[:, 0]] - pos[idx2[:, 1]]
        far = np.sqrt((sep * sep).sum(axis=1)) > 1.5
        winners, dist, w = idx2[:, 0], dist2[:, 0], self.w
        W = self.weights()
        total = degrees.sum()
        avg = (cdist(W, W) * degrees[None, :]).sum(axis=1) / total if total > 0 else np.full(len(W), np.nan)
        bw = avg.mean()
        kern = np.exp(-(dist**2) / (2 * bw**2)) / (bw * np.sqrt(2 * np.pi))
        hits = np.bincount(winners, weights=w, minlength=m)
        dens = np.bincount(winners, weights=kern * w, minlength=m)
        te, qe = self.allreduce_scalars([float(w[far].sum()), float((dist * w).sum())])
        hits, dens = self.allreduce_arrays([hits, dens])
        return {"te_count": te, "qe_sum": qe, "hits": hits, "dens_sum": dens, "avg_dist": avg, "weights": W, "n_rows": m}

    def label_histogram(self, n_classes):
        """Weighted class counts; `first` among the samples with positive weight."""
        if self.w is None:
            return super().label_histogram(n_classes)
        m = self.W.shape[0]
        y = self.y.astype(np.int64)
        flat = self._final * n_classes + y
        counts = self._hist(self._final, y, m, n_classes).astype(np.float64)
        first = np.full(m * n_classes, np.iinfo(np.int64).max, dtype=np.int64)
        present = np.flatnonzero(self.w > 0)
        np.minimum.at(first, flat[present], present.astype(np.int64) + self.sample_offset)
        (counts,) = self.allreduce_arrays([counts])
        (first,) = self.allreduce_arrays([first], op="min")
        return counts.reshape(m, n_classes), first.reshape(m, n_classes)


class WeightedShardedOracleEngine(WeightedOracleEngine, ShardedOracleEngine):
    """`ShardedOracleEngine` with weighted shards: the weighted sums are all-reduced like the unweighted ones."""

    def load_data(self, X, y, n_classes, sample_weight=None):
        if sample_weight is None:
            self.w = None
            return ShardedOracleEngine.load_data(self, X, y, n_classes)
        ShardedOracleEngine.load_data(self, X, y, n_classes)  # offsets and the global sample count
        self.w = np.asarray(sample_weight, dtype=np.float64)
        X64 = X.astype(np.float64)
        n = float(self._allreduce(np.array([self.w.sum()]))[0])
        mean = self._allreduce(self.w @ X64) / n
        ss = self._allreduce(self.w @ ((X64 - mean) ** 2))
        self.total_var = float((ss / n).sum())
        return {"n_samples": self.n_samples_global, "total_variance": self.total_var,
                "std_norm": float(np.sqrt((ss / (n - 1)).sum())), "total_weight": n}

    def epoch(self, sigma, pack_rows, entropy_error):
        if self.w is None:
            return ShardedOracleEngine.epoch(self, sigma, pack_rows, entropy_error)
        M, D = self.W.shape
        dist, win = O.bmu(self.X, self.W, 1)
        k = O.sample_weights(dist, self.total_var)
        Sk, sk, n = voronoi_sums(k, self.X, win, M, self.w)
        E = quantization_errors(win, dist, M, self.w)
        buf = self._allreduce(np.concatenate([Sk.ravel(), sk, n, E]))
        Sk, sk, n, E = buf[: M * D].reshape(M, D), buf[M * D : M * D + M], buf[M * D + M : M * D + 2 * M], buf[M * D + 2 * M :]
        live = np.flatnonzero(n > 0)
        C = np.zeros((M, D))
        if pack_rows:
            C[: live.size] = Sk[live] / sk[live][:, None]
        else:
            C[live] = Sk[live] / sk[live][:, None]
        W_new = O.smooth(C, n, O.neighborhood(self.hop, sigma))
        change = float(np.sum(np.linalg.norm(self.W - W_new, axis=1)))
        self.W_prev, self.W = self.W, W_new
        if entropy_error:
            E = class_entropy(self._allreduce(self._hist(win, self.y, M, self.n_classes)).reshape(M, self.n_classes))
        return {"error": E, "counts": n, "change": change}
