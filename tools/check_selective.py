"""Winners of the SELECTIVE tensor search (one fp16 pass + split passes over the flagged column tiles, samples in sorted
order) against the classic three-pass search and the fp32 SIMT back end, epoch by epoch on a bench-like trajectory;
prints differing rows, how many differ by more than a 1e-7 relative float64 gap, the share of (row-tile pair, column
tile) products refined and the device time of every stage.

    python tools/check_selective.py [rows] [d] [m] [epochs]
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


def compare(eng, got, ref, d, m, W, tag):
    diff = torch.nonzero(got[:, 0] != ref[:, 0])[:, 0]
    bad = 0
    if diff.numel():
        xs = eng.X[diff][:, :d].double()
        Wd = W[:m, :d]
        da = ((xs - Wd[got[diff, 0].long().clamp_min(0)]) ** 2).sum(1)
        db = ((xs - Wd[ref[diff, 0].long()]) ** 2).sum(1)
        rel = (da - db).abs() / torch.minimum(da, db).clamp_min(1e-300)
        bad = int(((rel > 1e-7) | (got[diff, 0] < 0)).sum())
    print(f"   {tag}: {int(diff.numel())} rows differ, {bad} beyond a 1e-7 relative gap; min idx {int(got.min())}", flush=True)
    return bad


def main():
    rows = int(sys.argv[1]) if len(sys.argv) > 1 else 400_000
    d = int(sys.argv[2]) if len(sys.argv) > 2 else 256
    m = int(sys.argv[3]) if len(sys.argv) > 3 else 4096
    epochs = int(sys.argv[4]) if len(sys.argv) > 4 else 6
    side = int(round(m ** 0.5))
    dev = torch.device("cuda", 0)
    X = make_shard(torch, dev, rows, d, 64, 0)
    eng = DeviceEngine(device="cuda:0", bmu_backend="tensor")
    eng.load_device_data(X)
    eng.init_map_from_rows(np.random.default_rng(0).choice(rows, m, replace=False), capacity=m)
    eng.set_hops_from_topology(MapTopology.full_grid(side, side))
    eng.resort_every = int(os.environ.get("DBGSOM_RESORT_EVERY", "3"))
    total_bad = 0
    for e in range(epochs):
        W = eng.W[eng.cur]
        if eng.row_perm is not None:
            x16 = (eng.X16_hi, eng.X16_lo, eng.xnorm16)
            ref = torch.empty((rows, 1), dtype=torch.int32, device=dev)
            cls = torch.full((rows, 1), -7, dtype=torch.int32, device=dev)
            got = torch.full((rows, 1), -7, dtype=torch.int32, device=dev)
            eng.strict_ties = True
            eng._run_bmu(eng.X, rows, eng.ldx, None, W, m, 1, False, ref, None, backend=(nat.BMU_SIMT, 0))
            eng.strict_ties = False
            eng._run_bmu(eng.X, rows, eng.ldx, x16, W, m, 1, False, cls, None, backend=(nat.BMU_TENSOR, 3), row_perm=eng.row_perm)
            eng.enable_profiling(True)
            eng.bmu_stats_host(reset=True)
            eng._run_bmu(eng.X, rows, eng.ldx, x16, W, m, 1, False, got, None, backend=(nat.BMU_TENSOR, 3), row_perm=eng.row_perm,
                         selective=True)
            ph = {k: round(sum(v), 3) for k, v in eng.phase_times_ms().items()}
            st = eng.bmu_stats_host()
            eng.enable_profiling(False)
            print(f"epoch {e}: stages ms {ph}; refined share {st.get('refined_share', 0):.3f} -> {st.get('mma_passes', 0):.2f} passes;"
                  f" ambiguous {st['ambiguous']} flagged {st['flagged']} rescans {st['full_rescans']}", flush=True)
            total_bad += compare(eng, cls, ref, d, m, W, "classic tensor search on sorted shadows vs simt")
            total_bad += compare(eng, got, ref, d, m, W, "selective search vs simt")
        r = eng.epoch(sigma_at(e, m), True, False)
        print(f"epoch {e} done: live {int((r['counts'] > 0).sum())} sorted {eng.row_perm is not None} age {eng.samples.age}", flush=True)
    print("OK" if total_bad == 0 else "MISMATCH")
    eng.close()


if __name__ == "__main__":
    main()
