"""Winners of the tensor back end against the fp32 SIMT back end (both followed by the exact float64 re-score) on
a bench-like problem; prints the number of differing rows and how many of those differ by more than a 1e-7 relative
float64 gap.  Used to validate kernel variants selected by environment switches (DBGSOM_TC_PAIR, DBGSOM_TC_CLUSTER).

    python tools/check_backends.py [rows] [d] [m] [epochs]
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bench import make_shard, sigma_at  # noqa: E402
from dbgsom_b200 import _native as nat  # noqa: E402
from dbgsom_b200.engine import DeviceEngine  # noqa: E402
from dbgsom_b200.topology import MapTopology  # noqa: E402


def main():
    rows = int(sys.argv[1]) if len(sys.argv) > 1 else 400_000
    d = int(sys.argv[2]) if len(sys.argv) > 2 else 256
    m = int(sys.argv[3]) if len(sys.argv) > 3 else 4096
    epochs = int(sys.argv[4]) if len(sys.argv) > 4 else 4
    side = int(round(m ** 0.5))
    dev = torch.device("cuda", 0)
    X = make_shard(torch, dev, rows, d, 64, 0)
    eng = DeviceEngine(device="cuda:0", bmu_backend="tensor")
    eng.load_device_data(X)
    eng.init_map_from_rows(np.random.default_rng(0).choice(rows, m, replace=False), capacity=m)
    # with a topology the streamed search (D > 256) lays its shadow columns out in map patches (per-tile bounds)
    eng.set_hops_from_topology(MapTopology.full_grid(side, side))
    total_bad = 0
    for e in range(epochs):
        W = eng.W[eng.cur]
        x16, _ = eng.samples.shadows(0, eng.X, (nat.BMU_TENSOR, 3), False)
        ref = torch.empty((rows, 1), dtype=torch.int32, device=dev)
        got = torch.empty((rows, 1), dtype=torch.int32, device=dev)
        eng.strict_ties = True
        eng._run_bmu(eng.X, rows, eng.ldx, None, W, m, 1, False, ref, None, backend=(nat.BMU_SIMT, 0))
        eng.strict_ties = False
        # (with a topology the engine may keep the shadows sorted by winner for its selective search: pass the order on)
        eng._run_bmu(eng.X, rows, eng.ldx, x16, W, m, 1, False, got, None, backend=(nat.BMU_TENSOR, 3),
                     row_perm=eng.row_perm)
        diff = torch.nonzero(got[:, 0] != ref[:, 0])[:, 0]
        bad = 0
        if diff.numel():
            xs = eng.X[diff][:, :d].double()
            Wd = W[:m, :d]
            da = ((xs - Wd[got[diff, 0].long()]) ** 2).sum(1)
            db = ((xs - Wd[ref[diff, 0].long()]) ** 2).sum(1)
            rel = (da - db).abs() / torch.minimum(da, db).clamp_min(1e-300)
            bad = int((rel > 1e-7).sum())
            if bad:  # who is right?  exact float64 scores of the differing rows against every prototype
                sel = diff[rel > 1e-7][:8]
                xs8 = eng.X[sel][:, :d].double()
                d2 = ((xs8[:, None, :] - Wd[None, :, :]) ** 2).sum(2)
                best = d2.argmin(1)
                two = torch.topk(d2, 2, dim=1, largest=False).values
                for q in range(sel.numel()):
                    print(f"   row {int(sel[q])}: exact {int(best[q])} tensor {int(got[sel[q], 0])} simt {int(ref[sel[q], 0])} "
                          f"exact rel gap {float((two[q, 1] - two[q, 0]) / two[q, 0]):.3e}", flush=True)
        total_bad += bad
        print(f"epoch {e}: {int(diff.numel())} rows differ, {bad} of them beyond a 1e-7 relative gap; min idx {int(got.min())}", flush=True)
        eng.epoch(sigma_at(e, m), True, False)
    print("OK" if total_bad == 0 else "MISMATCH")
    eng.close()


if __name__ == "__main__":
    main()
