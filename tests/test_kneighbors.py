"""kneighbors on the host (no GPU): argument checks and the contract of scikit-learn's NearestNeighbors, with the
CPU oracle standing in for the device engine; the workspace size of the top-k search from the C ABI."""
import numpy as np
import pytest
from sklearn.neighbors import NearestNeighbors

from _oracle_engine import OracleEngine
from dbgsom_b200 import SomClassifier, SomVQ
from dbgsom_b200 import _native as nat


def _oracle(cls):
    return type(cls.__name__, (cls,), {"_make_engine": lambda self, distributed=None: OracleEngine()})


@pytest.fixture(scope="module")
def fitted():
    X = np.random.default_rng(3).uniform(0, 10, size=(400, 3))
    som = _oracle(SomVQ)(n_iter=30, spreading_factor=0.9, max_neurons=40, random_state=0).fit(X)
    assert len(som.weights_) >= 17  # room for the limit check below
    return som, X


def test_matches_nearest_neighbors(fitted):
    som, X = fitted
    Q = X[::7] + 0.05
    for k in (1, 2, 3, 5, 16):
        dist, ind = som.kneighbors(Q, k)
        ref_d, ref_i = NearestNeighbors(n_neighbors=k).fit(som.weights_).kneighbors(Q)
        assert dist.dtype == np.float64 and ind.dtype == np.int64
        assert dist.shape == ind.shape == (len(Q), k)
        np.testing.assert_array_equal(ind, ref_i)
        np.testing.assert_allclose(dist, ref_d, rtol=1e-12)
        assert np.all(np.diff(dist, axis=1) >= 0)


def test_default_and_return_distance(fitted):
    som, X = fitted
    dist, ind = som.kneighbors(X)
    assert ind.shape == (len(X), 5)
    only = som.kneighbors(X, 5, return_distance=False)
    assert isinstance(only, np.ndarray)
    np.testing.assert_array_equal(only, ind)


def test_one_neighbour_is_predict(fitted):
    som, X = fitted
    np.testing.assert_array_equal(som.kneighbors(X, 1)[1][:, 0], som.predict(X))


def test_classifier_has_it():
    rng = np.random.default_rng(5)
    X = np.concatenate([rng.normal(c, 0.3, size=(60, 2)) for c in (0.0, 3.0)])
    y = np.repeat([0, 1], 60)
    clf = _oracle(SomClassifier)(n_iter=10, max_neurons=12, random_state=0).fit(X, y)
    k = min(4, len(clf.weights_))
    dist, ind = clf.kneighbors(X, k)
    ref_d, ref_i = NearestNeighbors(n_neighbors=k).fit(clf.weights_).kneighbors(X)
    np.testing.assert_array_equal(ind, ref_i)
    np.testing.assert_allclose(dist, ref_d, rtol=1e-12)


def test_argument_checks(fitted):
    som, X = fitted
    m = len(som.weights_)
    with pytest.raises(ValueError, match="n_neighbors > 0"):
        som.kneighbors(X, 0)
    with pytest.raises(ValueError, match="n_neighbors > 0"):
        som.kneighbors(X, -3)
    with pytest.raises(ValueError, match=f"n_samples_fit = {m}"):
        som.kneighbors(X, m + 1)
    with pytest.raises(ValueError, match="limit of 16"):
        som.kneighbors(X, 17)
    with pytest.raises(TypeError):
        som.kneighbors(X, 2.5)
    with pytest.raises(ValueError, match="features"):
        som.kneighbors(X[:, :2], 3)


def test_not_fitted():
    from sklearn.exceptions import NotFittedError

    with pytest.raises(NotFittedError):
        _oracle(SomVQ)().kneighbors(np.zeros((3, 2)), 1)


def test_limit_matches_header():
    import os

    header = os.path.join(os.path.dirname(__file__), "..", "include", "dbgsom_b200.h")
    text = open(header).read()
    assert f"#define DBGSOM_MAX_NBMU {nat.MAX_NBMU}" in text


def test_workspace_bytes():
    """Size function only: the candidate table holds 8 slots per row for n_bmu <= 2 and 32 beyond."""
    from dbgsom_b200 import build as builder

    builder.build()
    lib = nat.load()
    for n in (1, 1000, 12345):
        base = lib.dbgsom_bmu_workspace_bytes(n, 1)
        assert lib.dbgsom_bmu_workspace_bytes(n, 2) == base
        assert base >= n * (4 * nat.MAX_CAND + 1 + 4)
        for k in (3, 8, 16):
            wide = lib.dbgsom_bmu_workspace_bytes(n, k)
            assert wide >= n * (4 * 32 + 1 + 4)
            assert wide - base >= n * 4 * (32 - nat.MAX_CAND) - 256  # tables are padded to 256 bytes


# Runs in a process without a visible device, so that an argument check that stops refusing cannot launch a kernel on
# fake pointers: the call then fails on the missing device instead.
_REFUSALS = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
from dbgsom_b200 import _native as nat

lib = nat.load()
N, D, M = 1000, 64, 100
cases = {}


def args(n_bmu, backend, **kw):
    a = nat.BmuArgs()
    fake = iter(range(0x100000, 0x10000000, 0x10000))  # 16-byte aligned, never dereferenced
    for name in ("d_X", "d_X16_hi", "d_X16_lo", "d_xnorm16", "d_W", "d_W32", "d_W16_hi", "d_W16_lo", "d_wnorm",
                 "d_wmax", "d_proto_of_col", "d_idx", "d_dist", "d_stats", "d_workspace"):
        setattr(a, name, next(fake))
    a.N, a.D, a.ldx, a.ld16, a.M, a.Mpad = N, D, D, 64, M, 256
    a.n_bmu, a.backend, a.n_pass, a.want_dist, a.select_granule = n_bmu, backend, 3, 1, 64
    a.workspace_bytes = lib.dbgsom_bmu_workspace_bytes(N, n_bmu)
    for name, value in kw.items():
        setattr(a, name, value)
    return a


def run(a):
    return [lib.dbgsom_bmu_candidates(a, None), lib.dbgsom_bmu_resolve(a, None), lib.dbgsom_bmu(a, None)]


for k in (3, 16):
    for be, be_name in ((nat.BMU_TENSOR, "tensor"), (nat.BMU_SIMT, "simt")):
        tag = f"{be_name}-{k}"
        cases[f"valid-{tag}"] = run(args(k, be))
        cases[f"select-flag-{tag}"] = run(args(k, be, select=nat.SELECT_FLAG, d_tile_mask=0x20000000))
        cases[f"select-refine-{tag}"] = run(args(k, be, select=nat.SELECT_REFINE, d_tile_mask=0x20000000))
        cases[f"ties_any-{tag}"] = run(args(k, be, ties_any=1))
        cases[f"tile_bound-{tag}"] = run(args(k, be, d_tile_bound=0x20000000))
        cases[f"row_perm-{tag}"] = run(args(k, be, d_row_perm=0x20000000))
        cases[f"more-than-M-{tag}"] = run(args(k, be, M=k - 1))
        cases[f"top2-workspace-{tag}"] = run(args(k, be, workspace_bytes=lib.dbgsom_bmu_workspace_bytes(N, 2)))
    cases[f"one-pass-tensor-{k}"] = run(args(k, nat.BMU_TENSOR, n_pass=1))
for be in (nat.BMU_TENSOR, nat.BMU_SIMT):
    cases[f"n_bmu-17-{be}"] = run(args(17, be, workspace_bytes=lib.dbgsom_bmu_workspace_bytes(N, 16)))
print(json.dumps(cases))
"""


def test_topk_abi_refusals():
    """The C ABI refuses what the top-k search (n_bmu > 2) does not support: the selective search, ties_any, tile
    bounds and a sorted sample order are top-1 tools, the tensor front end runs top-k in its three-pass form only, and
    the candidate table needs 32 slots per row."""
    import json
    import os
    import subprocess
    import sys

    from dbgsom_b200 import build as builder

    builder.build()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", _REFUSALS, root], env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                         capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr[-2000:]
    cases = json.loads(res.stdout.strip().splitlines()[-1])
    badarg, workspace, unsupported = -1, -2, -3  # DBGSOM_E_*
    expect = {"select-flag": badarg, "select-refine": badarg, "ties_any": badarg, "tile_bound": badarg,
              "row_perm": badarg, "more-than-M": badarg, "top2-workspace": workspace, "one-pass-tensor": unsupported,
              "n_bmu-17": badarg}
    assert len(cases) == 2 * 2 * 8 + 2 + 2
    for name, codes in cases.items():
        if name.startswith("valid"):
            # passes every argument check and fails only for want of a device: the refusals below are the checks'
            assert codes[0] not in (0, badarg, workspace, unsupported) and codes[1] not in (0, badarg, workspace,
                                                                                              unsupported), (name, codes)
            continue
        want = next(v for key, v in expect.items() if name.startswith(key + "-"))
        assert codes == [want] * 3, (name, codes)
