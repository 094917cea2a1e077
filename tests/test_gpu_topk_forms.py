"""Every launch form of the top-k candidate search (the 15 `bmu_cand_tensor_kernel<3, 16, ...>` instantiations and the
SIMT top-k kernel) at k = 1 .. 16 against float64 references: results, the candidate tables behind them (superset of
the exact top k, flags) and the re-score counters.

The launch switches are read once per process, so every switch group runs in a worker process
(tests/_topk_form_worker.py).  The references are computed once here, by direct differences in float64, and handed to
the workers as files; the workers run the checks and report one JSON line per search.  With DBGSOM_TC_VERBOSE set the
launcher names each kernel form it launches, which proves that a group reached the forms it was written for."""
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import _topk_form_worker as FW
import _topk_reference as T

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def ref_dir(tmp_path_factory):
    """Top-17 indices and exact squared distances of every data set at every shape the groups run."""
    out = tmp_path_factory.mktemp("topk_ref")
    for n, d in sorted({(n, d) for g in FW.GROUPS.values() for n, d, _ in g["runs"]}):
        arrays = {}
        for ds in FW.DATASETS:
            X, W, info = T.make(ds, n, d, FW.m_of(ds))
            if ds == "families":
                # the flag assertions of the worker rest on these; if one fails, change R in T.families
                assert not T.check_family_premises(X, W, info, d), T.check_family_premises(X, W, info, d)
            arrays[f"{ds}_idx"], arrays[f"{ds}_d2"] = T.exact_topk(X, W, T.REF_RANKS - 1)
        np.savez(out / FW.ref_name(n, d), **arrays)
    return out


@pytest.mark.parametrize("group", list(FW.GROUPS))
def test_topk_forms_match_exact(group, ref_dir):
    env = {k: v for k, v in os.environ.items() if not k.startswith("DBGSOM_")}
    env.update(FW.GROUPS[group]["env"], DBGSOM_TC_VERBOSE="1")
    res = subprocess.run([sys.executable, os.path.join(HERE, "_topk_form_worker.py"), group, str(ref_dir)], env=env,
                         capture_output=True, text=True, timeout=1500)
    assert res.returncode == 0, res.stderr[-3000:]
    recs = [json.loads(line) for line in res.stdout.splitlines() if line.startswith("{")]
    assert len(recs) == len(FW.plan(group)), res.stdout[-2000:]
    failed = [r for r in recs if not r["ok"]]
    assert not failed, f"{len(failed)} of {len(recs)} searches failed, first:\n" + "\n".join(
        json.dumps(r) for r in failed[:3])
    # D. the group ran exactly the top-k forms it was written for: a switch that stops selecting its form fails here
    forms = set(re.findall(r"^dbgsom: K1 form (npass=3 nb=16 .*)$", res.stderr, flags=re.M))
    assert forms == set(FW.GROUPS[group]["forms"]), res.stderr[-3000:]
    for r in recs:
        if r["dataset"] == "benign" and r["k"] >= 3:
            print(f"{group} {r['backend']} N={r['n']} D={r['d']} k={r['k']}: flagged {r['flagged']}, "
                  f"ambiguous {r['ambiguous']}, candidates {r['candidates']}")
    print(res.stderr)
