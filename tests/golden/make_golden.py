"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    NUMBA_NUM_THREADS=1 python tests/golden/make_golden.py

Two kinds of fixture, both produced by importing the reference through oracle/_refshim.py:

* step_*.npz  -- one epoch body on hand-set state (the step-level recipe of SURVEY.md
  section 8(c)): `_get_winning_neurons`, `_calculate_exp_similarity`, `_update_weights`,
  `_write_accumulative_error` of dbgsom/BaseSom.py called on a SomVQ whose graph, weights,
  hop matrix, epoch and phase were set by hand.  Inputs that are not regenerable from a
  seed (W, hop) are stored next to the outputs.
* traj_*.npz  -- a full `fit` with per-epoch records (map size, per-neuron error, sigma,
  weight change, weight checksums) and every fitted attribute.
* fitstep_*.npz -- states captured INSIDE a reference `fit` at chosen epochs (BASELINE.json configs[1]:
  SomClassifier on the 70000 x 784 ten-class mixture): the prototypes, hop matrix and sigma the epoch body
  saw (dbgsom/BaseSom.py:397-407) and what it produced (winners, E, updated prototypes), for
  teacher-forced per-epoch parity at the config-2 shape; plus the fitted attributes of that fit.

The fixtures depend on the installed numpy / scikit-learn / numba / networkx versions
(recorded in each file).
"""
import json
import os
import sys

os.environ["NUMBA_NUM_THREADS"] = "1"
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import networkx as nx  # noqa: E402
import numpy as np  # noqa: E402

import _datasets  # noqa: E402
from oracle import _refshim  # noqa: E402

SomVQ, SomClassifier, ref_base = _refshim.load()


def versions():
    import numba
    import sklearn

    return json.dumps(
        dict(numpy=np.__version__, sklearn=sklearn.__version__, numba=numba.__version__, networkx=nx.__version__)
    )


# ----------------------------------------------------------------------------- step level
STEP_CASES = [
    dict(name="digits_5x5", data="digits", cast="float64", grid=(5, 5), wseed=1, epoch=3, n_iter=200, phase="coarse"),
    dict(name="digits_2x2_start", data="digits", cast="float64", grid=(2, 2), wseed=0, epoch=0, n_iter=200, phase="coarse"),
    dict(name="gmm64_6x6_dead", data="gmm:3000:64:8:1:float32", cast="float64", grid=(6, 6), wseed=2, epoch=10,
         n_iter=100, phase="coarse", dead=[0, 3, 17]),
    dict(name="gmm32_8x4_fine", data="gmm:2500:32:6:4:float32", cast="float64", grid=(8, 4), wseed=3, epoch=150,
         n_iter=200, phase="fine", dead=[5]),
    dict(name="gmm48_f32_4x4", data="gmm:2000:48:5:7:float32", cast="float32", grid=(4, 4), wseed=4, epoch=20,
         n_iter=80, phase="coarse"),
    dict(name="rings3d_3x7_kdtree", data="rings3d", cast="float64", grid=(3, 7), wseed=5, epoch=7, n_iter=60,
         phase="coarse"),
    dict(name="gmm128_12x12_linear", data="gmm:4000:128:16:9:float32", cast="float64", grid=(12, 12), wseed=6,
         epoch=30, n_iter=100, phase="coarse", params=dict(decay_function="linear", sigma_start=3.0, sigma_end=0.5)),
]


def run_step(case):
    X, _ = _datasets.load(case["data"])
    X = np.ascontiguousarray(X.astype(case["cast"]))
    gx, gy = case["grid"]
    g = nx.grid_2d_graph(gx, gy)
    M = g.number_of_nodes()
    rng = np.random.default_rng(case["wseed"])
    W = X[rng.choice(X.shape[0], M, replace=False)].astype(np.float64)
    for j in case.get("dead", []):
        W[j] = X.mean(axis=0) + 1e3
    som = SomVQ(n_iter=case["n_iter"], **case.get("params", {}))
    for j, node in enumerate(g.nodes):
        g.nodes[node]["weight"] = W[j].copy()
        g.nodes[node]["epoch_created"] = 0
        g.nodes[node]["error"] = 0
    som.som_ = g
    som.neurons_ = list(g.nodes)
    som.weights_ = W.copy()
    som._distance_matrix = nx.floyd_warshall_numpy(g)
    som._current_epoch = case["epoch"]
    som._training_phase = case["phase"]
    som._total_variance = np.var(X, axis=0).sum()
    som.converged_ = False
    som.growing_threshold_ = som._calculate_growing_threshold(X)
    sigma = som._calculate_current_sigma()
    dist, win = som._get_winning_neurons(X, 1)
    dist2, win2 = som._get_winning_neurons(X, 2)
    k = som._calculate_exp_similarity(dist)
    som._update_weights(k, win, X)
    som._write_accumulative_error(win, None, dist)
    W_new = som._extract_values_from_graph("weight")
    E = som._extract_values_from_graph("error").astype(np.float64)
    out = dict(
        meta=json.dumps({k_: v for k_, v in case.items()}),
        versions=versions(),
        W=W,
        hop=som._distance_matrix,
        sigma=np.float64(sigma),
        total_var=np.float64(som._total_variance),
        winners=win.astype(np.int64),
        dist=dist,
        k=k,
        winners2=win2.astype(np.int64),
        dist2=dist2,
        E=E,
        W_new=W_new,
        converged=np.bool_(som.converged_),
        growing_threshold=np.float64(som.growing_threshold_),
    )
    path = os.path.join(HERE, f"step_{case['name']}.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "M", M, "live", int((np.bincount(win, minlength=M) > 0).sum()))


# ----------------------------------------------------------------------------- trajectories
TRAJ_CASES = [
    dict(name="digits_vq", est="vq", data="digits", cast="float64", params=dict(random_state=0)),
    dict(name="digits_clf", est="clf", data="digits", cast="float64", params=dict(random_state=0)),
    dict(name="gmm32_vq_dead", est="vq", data="gmm:3000:32:10:2:float32", cast="float64",
         params=dict(random_state=1, n_iter=40, max_neurons=60)),
    dict(name="rings_clf", est="clf", data="rings3d", cast="float64",
         params=dict(random_state=2, n_iter=60, max_neurons=40)),
    dict(name="blobs_vq_linear", est="vq", data="blobs2d", cast="float64",
         params=dict(random_state=3, n_iter=50, decay_function="linear", convergence_iter=2,
                     threshold_method="classical", spreading_factor=0.05, max_neurons=30)),
    dict(name="gmm16_clf_entropy", est="clf", data="gmm:1500:16:4:11:float32", cast="float64",
         params=dict(random_state=4, n_iter=30, growth_criterion="entropy", spreading_factor=0.3, max_neurons=40)),
    dict(name="gmm24_vq_sigma", est="vq", data="gmm:2000:24:6:13:float32", cast="float64",
         params=dict(random_state=5, n_iter=24, sigma_start=1.5, sigma_end=0.4, coarse_training_frac=0.75,
                     learning_rate=0.1, max_neurons=25)),
]

# BASELINE.json configs[1] (SURVEY.md section 8(d)): SomClassifier on the Fashion-MNIST-shaped 70000 x 784 mixture
# with ten classes.  n_iter is kept small enough for CI (the reference needs ~0.5 s per epoch here); the states of
# `capture` epochs are stored in full, everything else as per-epoch records like the traj_* files.  A captured state
# costs 0.2-0.6 MB (its float64 prototypes do not compress), so two are kept to hold the file under 1 MB: epoch 5 of
# the growth phase and epoch 30 of the fine phase (sigma 0.7, near-equal prototypes, dead neurons below live ones).
FITSTEP_CASES = [
    # cast float64 (float32-representable values, like the other fixtures): with float32 input the reference's
    # total variance is a float32 row-by-row accumulation over 70000 rows (np.var, dbgsom/BaseSom.py:363) whose ~1e-5
    # rounding noise this fit amplifies by flipping samples between near-equidistant prototypes -- from epoch 2 on the
    # trajectory then depends on numpy's summation order, which no other implementation can reproduce
    dict(name="c2_gmm784_clf", est="clf", data="gmm:70000:784:10:21:float32", cast="float64",
         params=dict(random_state=7, n_iter=36, max_neurons=400), capture=[5, 30]),
]


def recording(cls):
    class Rec(cls):
        def _update_weights(self, sample_weights, winners, data):
            old = self.weights_.copy()
            self._log["M"].append(len(self.neurons_))
            self._log["sigma"].append(self._calculate_current_sigma())
            super()._update_weights(sample_weights, winners, data)
            new = self._extract_values_from_graph("weight")
            self._log["change"].append(float(np.sum(np.linalg.norm(old - new, axis=1))))
            self._log["wsum"].append(float(new.sum()))
            self._log["wfro"].append(float(np.sqrt((new * new).sum())))
            self._log["n"].append(np.bincount(winners, minlength=len(self.neurons_)).astype(np.float64))

        def _write_accumulative_error(self, winners, y, distances):
            super()._write_accumulative_error(winners, y, distances)
            self._log["E"].append(self._extract_values_from_graph("error").astype(np.float64))
            self._log["phase"].append(self._training_phase == "fine")

        def _delete_dead_neurons_from_graph(self, X):
            self._log["nodes_pre"] = np.array(list(self.som_.nodes), dtype=np.int64)
            self._log["epoch_created_pre"] = np.array(
                [d["epoch_created"] for _, d in self.som_.nodes.data()], dtype=np.int64
            )
            self._log["weights_pre"] = self._extract_values_from_graph("weight")
            self._log["hit_count_pre"] = self._extract_values_from_graph("hit_count").astype(np.float64)
            self._log["density_pre"] = self._extract_values_from_graph("density").astype(np.float64)
            self._log["avgdist_pre"] = self._extract_values_from_graph("average_distance").astype(np.float64)
            super()._delete_dead_neurons_from_graph(X)

        def _get_winning_neurons(self, data, n_bmu):
            dist, win = super()._get_winning_neurons(data, n_bmu)
            cap = getattr(self, "_capture", None)
            # the search of the epoch body (dbgsom/BaseSom.py:403): n_bmu == 1 on the full training matrix
            if cap is not None and n_bmu == 1 and self._in_loop and self._current_epoch in cap["epochs"]:
                e = self._current_epoch
                cap[f"e{e}_W"] = self.weights_.copy()
                cap[f"e{e}_hop"] = np.asarray(self._distance_matrix).copy()
                cap[f"e{e}_sigma"] = np.float64(self._calculate_current_sigma())
                cap[f"e{e}_winners"] = win.astype(np.int32)
                cap[f"e{e}_dist"] = dist.copy()
            return dist, win

        def _grow_som(self, data, y):
            self._in_loop = True
            try:
                super()._grow_som(data, y)
            finally:
                self._in_loop = False

    Rec._in_loop = False
    Rec.__name__ = cls.__name__
    return Rec


def run_traj(case):
    X, y = _datasets.load(case["data"])
    X = np.ascontiguousarray(X.astype(case["cast"]))
    cls = recording(SomVQ if case["est"] == "vq" else SomClassifier)
    som = cls(**case["params"])
    som._log = dict(M=[], sigma=[], change=[], wsum=[], wfro=[], n=[], E=[], phase=[])
    if case["est"] == "vq":
        som.fit(X)
    else:
        som.fit(X, y)
    log = som._log
    E_flat = np.concatenate(log["E"])
    n_flat = np.concatenate(log["n"])
    out = dict(
        meta=json.dumps(case),
        versions=versions(),
        epoch_M=np.array(log["M"], dtype=np.int64),
        epoch_sigma=np.array(log["sigma"]),
        epoch_change=np.array(log["change"]),
        epoch_wsum=np.array(log["wsum"]),
        epoch_wfro=np.array(log["wfro"]),
        epoch_fine=np.array(log["phase"], dtype=np.bool_),
        E_flat=E_flat,
        n_flat=n_flat,
        nodes_pre=log["nodes_pre"],
        epoch_created_pre=log["epoch_created_pre"],
        weights_pre=log["weights_pre"],
        hit_count_pre=log["hit_count_pre"],
        density_pre=log["density_pre"],
        avgdist_pre=log["avgdist_pre"],
        neurons=np.array(som.neurons_, dtype=np.int64),
        weights=som.weights_,
        distance_matrix=som._distance_matrix,
        n_iter_=np.int64(som.n_iter_),
        converged=np.bool_(som.converged_),
        quantization_error=np.float64(som.quantization_error_),
        topographic_error=np.float64(som.topographic_error_),
        growing_threshold=np.float64(som.growing_threshold_),
        total_var=np.float64(som._total_variance),
        node_label=np.array([d["label"] for _, d in som.som_.nodes.data()], dtype=np.int64),
        node_error=som._extract_values_from_graph("error").astype(np.float64),
        edges=np.array(sorted(tuple(sorted(e)) for e in som.som_.edges), dtype=np.int64).reshape(-1, 2, 2),
    )
    if case["est"] == "vq":
        out["labels"] = som.labels_.astype(np.int64)
        out["predict_head"] = som.predict(X[:200]).astype(np.int64)
    else:
        out["classes"] = som.classes_
        out["probabilities"] = som._extract_values_from_graph("probabilities")
        out["predict_head"] = som.predict(X[:200])
        out["proba_head"] = som.predict_proba(X[:50])
        out["score"] = np.float64(som.score(X, y))
    out["transform_head"] = som.transform(X[:20])
    path = os.path.join(HERE, f"traj_{case['name']}.npz")
    np.savez_compressed(path, **out)
    print(
        "wrote", path, "epochs", len(log["M"]), "M", log["M"][0], "->", len(log["nodes_pre"]), "final", len(som.neurons_),
        "QE", som.quantization_error_, "TE", som.topographic_error_,
    )


def run_fitstep(case):
    """A reference fit at the config-2 shape with the epoch-body states of `capture` epochs stored."""
    X, y = _datasets.load(case["data"])
    X = np.ascontiguousarray(X.astype(case["cast"]))
    base = SomVQ if case["est"] == "vq" else SomClassifier

    class Cap(recording(base)):
        def _update_weights(self, sample_weights, winners, data):
            super()._update_weights(sample_weights, winners, data)
            e = self._current_epoch
            if e in self._capture["epochs"]:
                self._capture[f"e{e}_W_new"] = self._extract_values_from_graph("weight")

        def _write_accumulative_error(self, winners, y_, distances):
            super()._write_accumulative_error(winners, y_, distances)
            e = self._current_epoch
            if e in self._capture["epochs"]:
                self._capture[f"e{e}_E"] = self._extract_values_from_graph("error").astype(np.float64)

    Cap.__name__ = base.__name__
    som = Cap(**case["params"])
    som._log = dict(M=[], sigma=[], change=[], wsum=[], wfro=[], n=[], E=[], phase=[])
    som._capture = dict(epochs=set(case["capture"]))
    som.fit(X) if case["est"] == "vq" else som.fit(X, y)
    cap, log = som._capture, som._log
    out = dict(
        meta=json.dumps(case), versions=versions(), total_var=np.float64(som._total_variance),
        growing_threshold=np.float64(som.growing_threshold_),
        epoch_M=np.array(log["M"], dtype=np.int64), epoch_sigma=np.array(log["sigma"]),
        epoch_change=np.array(log["change"]), epoch_wfro=np.array(log["wfro"]),
        E_flat=np.concatenate(log["E"]), n_flat=np.concatenate(log["n"]),
        neurons=np.array(som.neurons_, dtype=np.int64), nodes_pre=log["nodes_pre"],
        weights=som.weights_.astype(np.float32),  # compared at 1e-4: float32 keeps the file small
        n_iter_=np.int64(som.n_iter_), quantization_error=np.float64(som.quantization_error_),
        topographic_error=np.float64(som.topographic_error_), converged=np.bool_(som.converged_),
    )
    if case["est"] != "vq":
        out["classes"] = som.classes_
        out["score"] = np.float64(som.score(X, y))
        out["node_label"] = np.array([d["label"] for _, d in som.som_.nodes.data()], dtype=np.int64)
    else:
        out["labels"] = som.labels_.astype(np.int32)
    for e in sorted(cap["epochs"]):
        if f"e{e}_W" not in cap:
            continue
        hop = cap[f"e{e}_hop"]
        h16 = np.full(hop.shape, 0xFFFF, dtype=np.uint16)
        h16[np.isfinite(hop)] = hop[np.isfinite(hop)].astype(np.uint16)
        m = cap[f"e{e}_W"].shape[0]
        out[f"e{e}_W"] = cap[f"e{e}_W"]                              # float64: the exact state the reference saw
        out[f"e{e}_hop"] = h16
        out[f"e{e}_sigma"] = cap[f"e{e}_sigma"]
        out[f"e{e}_winners"] = cap[f"e{e}_winners"].astype(np.uint8 if m <= 256 else np.uint16)
        out[f"e{e}_dist_sum"] = np.float64(cap[f"e{e}_dist"].sum())  # (the per-neuron sums of dist are E)
        out[f"e{e}_E"] = cap[f"e{e}_E"]
        out[f"e{e}_W_new"] = cap[f"e{e}_W_new"].astype(np.float32)   # compared at 1e-5
    out["captured"] = np.array(sorted(e for e in cap["epochs"] if f"e{e}_W" in cap), dtype=np.int64)
    path = os.path.join(HERE, f"fitstep_{case['name']}.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "epochs", len(log["M"]), "M per epoch", log["M"], "final", len(som.neurons_),
          "QE", som.quantization_error_, "size", os.path.getsize(path))


if __name__ == "__main__":
    only = sys.argv[1:]
    for c in FITSTEP_CASES:
        if not only or c["name"] in only:
            run_fitstep(c)
    for c in STEP_CASES:
        if not only or c["name"] in only:
            run_step(c)
    for c in TRAJ_CASES:
        if not only or c["name"] in only:
            run_traj(c)
