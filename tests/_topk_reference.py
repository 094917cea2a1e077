"""Exact float64 top-k references, the parity assertion and the seeded data sets of the top-k tests
(tests/test_gpu_kneighbors.py, tests/test_gpu_topk_forms.py and its worker tests/_topk_form_worker.py)."""
import numpy as np

import _datasets
from oracle import som_oracle as O

GAP = 1e-6
REF_RANKS = 17  # ranks the form tests keep: the largest k (16) and the rank behind it
OVERFLOW = 255  # DBGSOM_CAND_OVERFLOW: cand_count of a flagged row
SLOTS = 32      # DBGSOM_MAX_CAND_K: candidate slots per row of a top-k search


def exact_topk(X, W, k):
    """Indices (lowest index first on exact ties) and squared distances of the k + 1 nearest prototypes (all M when
    M <= k), by direct differences in float64.  The float64 expansion preselects k + 65 candidates; it cannot order
    prototypes whose distances differ by less than its cancellation error (samples sitting on a cluster of
    near-copies), so the candidates are ranked again by direct differences."""
    X64 = np.asarray(X, dtype=np.float64)
    W64 = np.asarray(W, dtype=np.float64)
    kk = min(k + 65, W.shape[0])
    _, cand = O.bmu_expansion(X64, W64, kk)
    cand = np.sort(cand.reshape(len(X), kk), axis=1)
    d2 = np.empty((len(X), kk))
    for s in range(0, len(X), 256):
        diff = X64[s : s + 256, None, :] - W64[cand[s : s + 256]]
        d2[s : s + 256] = np.einsum("nkd,nkd->nk", diff, diff)
    order = np.argsort(d2, axis=1, kind="stable")[:, : min(k + 1, kk)]
    return np.take_along_axis(cand, order, axis=1), np.take_along_axis(d2, order, axis=1)


def separated(d2, k, gap):
    """[N, k] bool: rank r's squared distance is more than `gap` (relative) away from those of ranks r - 1 and r + 1.
    `d2` holds at least k ranks; without a rank k + 1 (k == M) the last rank has nothing behind it."""
    scale = np.maximum(d2[:, :k], 1e-300)
    sep = np.ones((len(d2), k), dtype=bool)  # rank r is separated from rank r + 1
    m = min(d2.shape[1], k + 1)
    sep[:, : m - 1] = (d2[:, 1:m] - d2[:, : m - 1]) > gap * scale[:, : m - 1]
    ok = sep.copy()
    ok[:, 1:] &= sep[:, : k - 1]
    return ok


def assert_topk_parity(dist, idx, X, W, k, gap=GAP, ref=None):
    """Indices equal at every rank whose squared distance is more than `gap` (relative) away from its neighbours'
    ranks; distances equal to float64 rounding of the direct-difference sum.  `ref` = (indices, squared distances)
    of at least k + 1 ranks from `exact_topk` (computed here if None).  Returns the number of gated rows."""
    assert idx.shape == dist.shape == (len(X), k)
    ref_idx, d2 = exact_topk(X, W, k) if ref is None else (ref[0][:, : k + 1], ref[1][:, : k + 1])
    ok = separated(d2, k, gap)
    bad = np.argwhere((idx != ref_idx[:, :k]) & ok)
    assert bad.size == 0, f"{len(bad)} (row, rank) mismatches outside near-ties, first {bad[:5].tolist()}"
    # distances: exact where the index matches, within the gate elsewhere
    d2_k = d2[:, :k]
    same = idx == ref_idx[:, :k]
    np.testing.assert_allclose(dist[same], np.sqrt(d2_k[same]), rtol=1e-12, atol=1e-300)
    np.testing.assert_allclose(dist, np.sqrt(d2_k), rtol=gap)
    assert (np.diff(dist, axis=1) >= 0).all()
    # every returned index is a distinct prototype
    srt = np.sort(idx, axis=1)
    assert (srt[:, 1:] != srt[:, :-1]).all()
    return int((~ok).any(axis=1).sum())


def bench_like_maps(n, d, m, seed=11):
    X = _datasets.gmm(n, d, 32, seed)
    rng = np.random.default_rng(5)
    W = X[rng.choice(n, m, replace=False)].astype(np.float64)
    W += rng.normal(0.0, 0.01, size=W.shape) * np.abs(W).mean()
    return X, W


# ------------------------------------------------------------------------------------------------ form-test data sets
# Families: chosen sample rows, each with FAMILY prototypes at squared distances R^2 (1 + s q), q = 0 .. FAMILY - 1, in
# orthogonal directions.  At s = 1e-2 only the k nearest members lie inside the row's candidate bound; at s = 3e-9 all
# of them do, so the row has more in-bound prototypes than the table's 32 slots and must be flagged.
SPACINGS = (1e-2, 1e-5, 1e-7, 3e-9)
ROWS_PER_SPACING = 6
FAMILY = 36
N_COPIES = 17


def _nearest_sq(X, W):
    d, _ = O.bmu_expansion(X, W, 1)
    return d**2


def _pick_rows(X, W, count, rng):
    """`count` distinct sample rows whose nearest prototype is at about the median distance (not the sample rows the
    bench-like map was drawn from, which sit on a prototype)."""
    pool = rng.choice(len(X), min(len(X), 40 * count), replace=False)
    d2 = _nearest_sq(X[pool], W)
    return pool[np.argsort(np.abs(d2 - np.median(d2)))[:count]], np.median(d2)


def _directions(d, count, rng):
    q, _ = np.linalg.qr(rng.normal(size=(d, count)))
    return q.T  # [count, d] orthonormal rows


def families(n, d, m, seed):
    """Benign map of m - 24 * 36 prototypes plus one family of 36 per chosen row; the family members take scattered
    indices.  Returns X, W and {spacing: rows}."""
    n_fam = len(SPACINGS) * ROWS_PER_SPACING
    X, W0 = bench_like_maps(n, d, m - n_fam * FAMILY, seed)
    rng = np.random.default_rng(seed + 101)
    rows, _ = _pick_rows(X, W0, n_fam, rng)
    r2 = 0.25 * _nearest_sq(X[rows], W0)  # R = half the row's nearest-prototype distance
    members = []
    for i, row in enumerate(rows):
        s = SPACINGS[i // ROWS_PER_SPACING]
        radius = np.sqrt(r2[i] * (1.0 + s * np.arange(FAMILY)))
        members.append(X[row].astype(np.float64) + radius[:, None] * _directions(d, FAMILY, rng))
    W = np.concatenate([W0] + members)
    W = W[rng.permutation(len(W))]
    groups = {s: rows[i * ROWS_PER_SPACING : (i + 1) * ROWS_PER_SPACING] for i, s in enumerate(SPACINGS)}
    return X, W, groups


def copies(n, d, m, seed):
    """Benign map with two families written over scattered prototypes: 17 exact copies of one point near row a, and
    5 distinct members at 1e-2 spacing followed by 12 exact copies of one point near row b (rank k falls inside the
    run of copies for k = 6 .. 16).  Returns X, W and {row: member indices in rank order, lowest index first}."""
    X, W = bench_like_maps(n, d, m, seed)
    rng = np.random.default_rng(seed + 202)
    rows, _ = _pick_rows(X, W, 2, rng)
    r2 = 0.25 * _nearest_sq(X[rows], W)
    slots = rng.choice(m, 2 * N_COPIES, replace=False)
    a, b = slots[:N_COPIES], slots[N_COPIES:]
    u = _directions(d, 6, rng)
    W[a] = X[rows[0]] + np.sqrt(r2[0]) * u[0]
    for q in range(5):
        W[b[q]] = X[rows[1]] + np.sqrt(r2[1] * (1.0 + 1e-2 * q)) * u[1 + q]
    W[b[5:]] = X[rows[1]] + np.sqrt(r2[1] * (1.0 + 1e-2 * 5)) * u[5]
    order = {int(rows[0]): np.sort(a), int(rows[1]): np.concatenate([b[:5], np.sort(b[5:])])}
    return X, W, order


def make(name, n, d, m, seed=11):
    """X, W and the rows of interest of data set `name`: "benign", "families", "copies" or "mk<k>" (a map of exactly
    k prototypes)."""
    if name == "benign":
        X, W = bench_like_maps(n, d, m, seed)
        return X, W, None
    if name == "families":
        return families(n, d, m, seed)
    if name == "copies":
        return copies(n, d, m, seed)
    k = int(name[2:])
    X, W = bench_like_maps(n, d, m, seed)
    return X, W[:k].copy(), None


def row_bound_range(X, W, d):
    """(smallest, largest) of the tensor search's candidate window 2B over the kernel forms, bound scales and
    accumulation chains the form tests run, per row and in squared-distance units (csrc/common.cuh:
    tensor_score_bound with the coefficients of tensor_bound_coef and tensor_acc_coef_args; the shadow scale cancels).
    The shadows are centred on the prototypes' mean."""
    mu = W.mean(axis=0)
    xn = np.linalg.norm(np.asarray(X, np.float64) - mu, axis=1)
    wn = np.linalg.norm(W - mu, axis=1)
    umax, wnorm_max = wn.max(), (wn**2).max()
    ld16 = -(-d // 64) * 64
    steps = ld16 / 16 * 3
    grow = max(steps / 48, 1.0)
    coefs = (0.0625 * 1.9073486e-6, 1.9073486e-6)  # default and bound_scale = 1
    # accumulation: one chain (default / strict), chains of 4 and 8 k-blocks (default / strict)
    accs = (2.4e-7 * np.sqrt(grow), 2.4e-7 * grow, 2.4e-7 * 2.0, 2.4e-7 * 4.0, 2.4e-7 * 2.0 * np.sqrt(2.0), 2.4e-7 * 8.0)
    xw = xn * umax
    lo = 2.0 * (xw * min(coefs) + min(accs) * (xw + wnorm_max))
    hi = 2.0 * (xw * max(coefs) + max(accs) * (xw + wnorm_max))
    return lo, hi


def check_family_premises(X, W, groups, d):
    """The 1e-2 families have only their k nearest members inside every form's bound (a tenfold margin on the gap to
    member k + 1), the 3e-9 families all 36 (the spread of the family is under a tenth of the smallest bound).
    Returns a message per violated premise."""
    lo, hi = row_bound_range(X, W, d)
    msgs = []
    for s in (SPACINGS[0], SPACINGS[-1]):
        rows = groups[s]
        r2 = _nearest_sq(X[rows], W)  # the family's nearest member: R^2
        if s == SPACINGS[0] and not (s * r2 > 10.0 * hi[rows]).all():
            msgs.append(f"s={s}: member gap {s * r2} not 10x above the largest bound {hi[rows]}")
        if s == SPACINGS[-1] and not ((FAMILY - 1) * s * r2 < 0.1 * lo[rows]).all():
            msgs.append(f"s={s}: family spread {(FAMILY - 1) * s * r2} not under a tenth of the bound {lo[rows]}")
    return msgs
