"""Empirical check of the tensor back end's error-bound scale (run on a B200).

Trains a fixed map for a few epochs (real trajectory, reference semantics) and, at every epoch,
compares the winners of the tcgen05 search for several `bound_scale` values with the fp32 SIMT
search (whose candidate window is a proven worst-case bound) -- both followed by the same exact
float64 re-score.  A bound that is too small shows up as winners that differ although the exact
float64 gap between the two prototypes is far above rounding.

    python tools/calibrate_bound.py [--rows 1000000] [--d 256] [--side 64] [--epochs 10]
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bench import grid_hops, make_shard, sigma_at  # noqa: E402
from dbgsom_b200 import _native as nat  # noqa: E402
from dbgsom_b200.engine import DeviceEngine  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--d", type=int, default=256)
    ap.add_argument("--side", type=int, default=64)
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--scales", default="1,0.25,0.125,0.0625,0.03,0.015,0.004")
    ap.add_argument("--n-pass", type=int, default=3)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    m = args.side**2
    X = make_shard(torch, dev, args.rows, args.d, 64, 0)
    eng = DeviceEngine(device="cuda:0", bmu_backend="tensor" if args.n_pass == 3 else "tensor1")
    eng.load_device_data(X)
    eng.init_map_from_rows(np.random.default_rng(0).choice(args.rows, m, replace=False), capacity=m)
    eng.set_hops(grid_hops(args.side))
    scales = [float(s) for s in args.scales.split(",")]
    print("epoch  " + "  ".join(f"k={s:<7g}" for s in scales) + "   (mismatching winners with exact rel. gap > 1e-7 | flagged | ambiguous)")
    for e in range(args.epochs):
        W = eng.W[eng.cur]
        x16, _ = eng.samples.shadows(0, eng.X, (nat.BMU_TENSOR, 3), False)
        ref = torch.empty((eng.N, 1), dtype=torch.int32, device=dev)
        eng.strict_ties = True
        eng._run_bmu(eng.X, eng.N, eng.ldx, None, W, eng.M, 1, False, ref, None, backend=(nat.BMU_SIMT, 0))
        Wd = W[: eng.M]
        cells = []
        for s in scales:
            eng.bound_scale, eng.strict_ties = s, False
            eng.bmu_stats_host(reset=True)
            got = torch.empty((eng.N, 1), dtype=torch.int32, device=dev)
            eng._run_bmu(eng.X, eng.N, eng.ldx, x16, W, eng.M, 1, False, got, None, backend=(nat.BMU_TENSOR, args.n_pass))
            st = eng.bmu_stats_host(reset=True)
            diff = torch.nonzero(got[:, 0] != ref[:, 0])[:, 0]
            bad = 0
            if diff.numel():
                xs = eng.X[diff].double()
                da = ((xs - Wd[got[diff, 0].long()]) ** 2).sum(1)
                db = ((xs - Wd[ref[diff, 0].long()]) ** 2).sum(1)
                rel = (da - db).abs() / torch.minimum(da, db).clamp_min(1e-300)
                bad = int((rel > 1e-7).sum())
                worst = float(rel.max())
            cells.append(f"{bad}/{int(diff.numel())}|{st['flagged']}|{st['ambiguous']}")
        print(f"{e:5d}  " + "  ".join(f"{c:<9s}" for c in cells))
        eng.bound_scale, eng.strict_ties = 0.0, False
        eng.epoch(sigma_at(e, m), True, False)
    eng.close()


if __name__ == "__main__":
    main()
