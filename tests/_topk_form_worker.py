"""Worker of tests/test_gpu_topk_forms.py: one process per group of K1 launch switches (DBGSOM_TC_PAIR,
DBGSOM_TC_CLUSTER and DBGSOM_TC_SEGM are read once per process).

    python tests/_topk_form_worker.py GROUP REF_DIR

Runs every data set of the group's shapes through DeviceEngine.bmu for k = 1 .. 16, checks the results, the candidate
table the search left in the engine's workspace and the re-score counters against the float64 references in REF_DIR,
and prints one JSON line per (shape, backend, data set, run, k) that names the checks that failed."""
import json
import os
import sys
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import _topk_reference as T  # noqa: E402

LARGE = 19077  # 150 row tiles of 128: past the 148-SM threshold of the clustered forms, last tile has 5 rows
SMALL = 5000   # 40 row tiles: the single-CTA forms
KS = range(1, 17)
DATASETS = ["benign", "families", "copies"] + [f"mk{k}" for k in range(3, 17)]
STRICT_DATASETS = ("families", "copies")
STRICT_GAP = 1e-9


def m_of(dataset):
    return 1123 if dataset == "families" else 1100  # not multiples of 256: padding columns in the last tile


def form(bn, akb, cl, pair, sgt=0):
    return f"npass=3 nb=16 bn={bn} res_kb=0 akb={akb} cl={cl} pair={pair} sel=0 tb=0 sgt={sgt}"


# D = 64: one k-block (AKB = 2 forms); D = 200: ld16 = 256, four k-blocks with zero-padded columns (AKB = 4);
# D = 520: ld16 = 576, nine k-blocks (streamed forms; the segmented ones end on a short chain: 4 + 4 + 1 or 8 + 1)
GROUPS = {
    "default": {
        "env": {},
        "runs": [(LARGE, 64, "tensor"), (LARGE, 200, "tensor"), (LARGE, 520, "tensor"),
                 (SMALL, 64, "tensor"), (SMALL, 200, "tensor"), (SMALL, 520, "tensor"),
                 (SMALL, 64, "simt"), (SMALL, 200, "simt"), (SMALL, 520, "simt")],
        "forms": [form(128, 2, 2, 1), form(128, 4, 2, 1), form(256, 0, 2, 1, 4),
                  form(128, 2, 1, 0), form(128, 4, 1, 0), form(128, 0, 1, 0)],
    },
    "pair0": {
        "env": {"DBGSOM_TC_PAIR": "0"},
        "runs": [(LARGE, 64, "tensor"), (LARGE, 200, "tensor"), (LARGE, 520, "tensor")],
        "forms": [form(128, 2, 2, 0), form(128, 4, 2, 0), form(128, 0, 2, 0)],
    },
    "pair0-cluster4": {
        "env": {"DBGSOM_TC_PAIR": "0", "DBGSOM_TC_CLUSTER": "4"},
        "runs": [(LARGE, 64, "tensor"), (LARGE, 200, "tensor"), (LARGE, 520, "tensor")],
        "forms": [form(128, 2, 4, 0), form(128, 4, 4, 0), form(128, 0, 4, 0)],
    },
    "segm2-tmem-chains8": {
        "env": {"DBGSOM_TC_SEGM": "2"},
        "runs": [(LARGE, 520, "tensor")],
        "forms": [form(256, 0, 2, 1, 8)],
    },
    "segm1-register-sums": {
        "env": {"DBGSOM_TC_SEGM": "1"},
        "runs": [(LARGE, 520, "tensor")],
        "forms": [form(128, 0, 2, 1)],
    },
    "segm0-one-chain": {
        "env": {"DBGSOM_TC_SEGM": "0"},
        "runs": [(LARGE, 520, "tensor")],
        "forms": [form(256, 0, 2, 1)],
    },
}


def ref_name(n, d):
    return f"ref_{n}_{d}.npz"


def plan(group):
    """(n, d, backend, data set, run, k) of every search the group runs: the M == k maps (tensor only) at k = M, the
    others at every k, families and copies a second time with the strict worst-case bound."""
    out = []
    for n, d, backend in GROUPS[group]["runs"]:
        for ds in DATASETS:
            if ds.startswith("mk"):
                if backend == "tensor":
                    out.append((n, d, backend, ds, "default", int(ds[2:])))
                continue
            for run in ("default", "strict") if ds in STRICT_DATASETS else ("default",):
                out.extend((n, d, backend, ds, run, k) for k in KS)
    return out


def candidate_table(eng, lib, n, k):
    """cand_idx [n, 32] and cand_count [n] of the last search (BmuWorkspace in csrc/common.cuh)."""
    ws = eng._ws["bmu"]
    assert ws.numel() >= lib.dbgsom_bmu_workspace_bytes(n, k)
    idx_bytes = n * T.SLOTS * 4
    cidx = ws[:idx_bytes].view(eng.torch.int32).reshape(n, T.SLOTS).cpu().numpy()
    off = -(-idx_bytes // 256) * 256
    return cidx, ws[off : off + n].cpu().numpy()


def check_results(X, W, info, ds, run, k, dist, idx, ref_idx, ref_d2, flagged):
    """A: indices outside near-ties, distances, order; flagged rows exact to 1e-12; copies in index order."""
    gap = STRICT_GAP if run == "strict" else T.GAP
    gated = T.assert_topk_parity(dist, idx, X, W, k, gap=gap, ref=(ref_idx, ref_d2))
    fr = np.flatnonzero(flagged)  # these rows went through the float64 re-scan
    if fr.size:
        ok = T.separated(ref_d2[fr], k, 1e-12)
        bad = np.argwhere((idx[fr] != ref_idx[fr, :k]) & ok)
        assert bad.size == 0, f"flagged rows: {len(bad)} (row, rank) mismatches, first {fr[bad[:5, 0]].tolist()}"
    if ds == "copies":  # exact ties: lowest index first, nothing gated
        for row, members in info.items():
            np.testing.assert_array_equal(ref_idx[row, :k], members[:k])
            np.testing.assert_array_equal(idx[row], members[:k])
    return gated


def check_table(W, info, ds, run, k, cidx, ccnt, ref_idx, ref_d2):
    """B: the candidate table of every unflagged row is a duplicate-free superset of the exact top k within 32 slots;
    the families are flagged, or not, as their spacing dictates."""
    m = len(W)
    flagged = ccnt == T.OVERFLOW
    un = np.flatnonzero(~flagged)
    cnt = ccnt[un].astype(np.int64)
    assert (cnt >= min(k, m)).all() and (cnt <= T.SLOTS).all(), f"counts out of [k, 32]: {np.unique(cnt).tolist()}"
    live = np.arange(T.SLOTS)[None, :] < cnt[:, None]
    slots = cidx[un]
    assert ((slots >= 0) & (slots < m))[live].all(), "slot outside [0, M)"
    srt = np.sort(np.where(live, slots, -1 - np.arange(T.SLOTS)[None, :]), axis=1)
    assert (srt[:, 1:] != srt[:, :-1]).all(), "repeated prototype in a row's slots"
    # superset: every prototype whose exact distance is within the reference's k-th is a candidate
    r_idx, r_d2 = ref_idx[un], ref_d2[un]
    need = r_d2 <= r_d2[:, k - 1 : k]
    if run != "strict" and r_d2.shape[1] > k:  # the calibrated bound: only where rank k is separated from rank k + 1
        need &= ((r_d2[:, k] - r_d2[:, k - 1]) > T.GAP * np.maximum(r_d2[:, k - 1], 1e-300))[:, None]
    held = ((slots[:, None, :] == r_idx[:, :, None]) & live[:, None, :]).any(axis=2)
    miss = np.argwhere(need & ~held)
    assert miss.size == 0, f"{len(miss)} in-bound prototypes missing from the table, first rows {un[miss[:5, 0]].tolist()}"
    if ds == "families":
        rows = info[T.SPACINGS[-1]]
        assert flagged[rows].all(), f"s=3e-9 family rows not flagged: {rows[~flagged[rows]].tolist()}"
        rows = info[T.SPACINGS[0]]
        assert not flagged[rows].any(), f"s=1e-2 family rows flagged: {rows[flagged[rows]].tolist()}"
        sep = (ref_d2[rows, k] - ref_d2[rows, k - 1]) > 1e-4 * ref_d2[rows, k - 1]
        assert (ccnt[rows][sep] == k).all(), f"s=1e-2 family rows: counts {ccnt[rows].tolist()}, k = {k}"


def check_counters(ds, k, st, ccnt):
    """C: the re-score counters agree with the table; benign data flags almost nothing."""
    n = len(ccnt)
    flagged = ccnt == T.OVERFLOW
    cnt = ccnt[~flagged].astype(np.int64)
    n_flag = int(flagged.sum())
    assert st["flagged"] == st["full_rescans"] == n_flag, (st, n_flag)
    assert st["candidates"] == int(cnt.sum()), (st, int(cnt.sum()))
    assert st["ambiguous"] == int((cnt > k).sum()), (st, int((cnt > k).sum()))
    if ds == "benign":  # B200: at most 1 row (D = 520, k = 3) in every group, shape and k; a flag-all epilogue fails
        assert n_flag <= 10, f"{n_flag} of {n} benign rows flagged"


def check(eng, lib, X, W, info, ds, run, k, ref_idx, ref_d2):
    """Runs the search and checks A (results), B (candidate table, k >= 3; the one- and two-winner searches keep 8
    slots per row) and C (counters, k >= 3).  Returns the counters and {check: error} of the checks that failed."""
    n = len(X)
    dist, idx = eng.bmu(X, W, k)
    assert eng.N == n, "the search ran in row chunks"  # one call, so the workspace holds every row's table
    st = eng.bmu_stats_host()
    out, errors = {}, {}
    cidx, ccnt = candidate_table(eng, lib, n, k) if k >= 3 else (None, np.zeros(n, np.uint8))
    steps = [("A", lambda: out.update(gated_rows=check_results(X, W, info, ds, run, k, dist, idx, ref_idx, ref_d2,
                                                               ccnt == T.OVERFLOW)))]
    if k >= 3:
        steps += [("B", lambda: check_table(W, info, ds, run, k, cidx, ccnt, ref_idx, ref_d2)),
                  ("C", lambda: check_counters(ds, k, st, ccnt))]
        out.update(flagged=int((ccnt == T.OVERFLOW).sum()), candidates=st["candidates"], ambiguous=st["ambiguous"])
    for name, step in steps:
        try:
            step()
        except AssertionError:
            errors[name] = traceback.format_exc(limit=2)[-1000:]
    return out, errors


def main():
    group, ref_dir = sys.argv[1], sys.argv[2]
    from dbgsom_b200 import _native as nat
    from dbgsom_b200.engine import DeviceEngine

    lib = nat.load()
    data, refs, engines = {}, {}, {}
    for n, d, backend, ds, run, k in plan(group):
        if (n, d, ds) not in data:
            data = {(n, d, ds): T.make(ds, n, d, m_of(ds))}  # one data set at a time
        X, W, info = data[(n, d, ds)]
        if (n, d) not in refs:
            refs = {(n, d): np.load(os.path.join(ref_dir, ref_name(n, d)))}
        ref = refs[(n, d)]
        key = (n, d, backend, run)
        if key not in engines:
            for e in engines.values():
                e.close()
            strict = run == "strict"
            engines = {key: DeviceEngine(bmu_backend=backend, strict_ties=strict, bound_scale=1.0 if strict else 0.0)}
        rec = {"n": n, "d": d, "m": len(W), "backend": backend, "dataset": ds, "run": run, "k": k}
        counts, errors = check(engines[key], lib, X, W, info, ds, run, k, ref[f"{ds}_idx"], ref[f"{ds}_d2"])
        rec.update(counts, ok=not errors, failed=sorted(errors), errors=errors)
        print(json.dumps(rec), flush=True)
    for e in engines.values():
        e.close()


if __name__ == "__main__":
    main()
