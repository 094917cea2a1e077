"""K1 candidate search alone: time per launch over a few map sizes (row-tile overhead vs. per-prototype cost).

    python tools/bench_k1.py [rows] [d] [m1,m2,...] [reps]

Prototypes are random sample rows (benign: one candidate per row), so the time is the MMA / epilogue pipeline
itself.  Prints ms per launch, algorithmic TFLOP/s (2 N M D) and cycles per 128-row tile at the sampled clock.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bench import make_shard  # noqa: E402
from dbgsom_b200 import _native as nat  # noqa: E402
from dbgsom_b200.engine import DeviceEngine  # noqa: E402


def main():
    rows = int(sys.argv[1]) if len(sys.argv) > 1 else 2_000_000
    d = int(sys.argv[2]) if len(sys.argv) > 2 else 256
    ms = [int(v) for v in (sys.argv[3] if len(sys.argv) > 3 else "1024,2048,4096,8192").split(",")]
    reps = int(sys.argv[4]) if len(sys.argv) > 4 else 5
    dev = torch.device("cuda", 0)
    X = make_shard(torch, dev, rows, d, 64, 0)
    for m in ms:
        eng = DeviceEngine(device="cuda:0", bmu_backend="tensor")
        eng.load_device_data(X)
        eng.init_map_from_rows(np.random.default_rng(0).choice(rows, m, replace=False), capacity=m)
        x16, _ = eng.samples.shadows(0, eng.X, (nat.BMU_TENSOR, 3), False)
        idx = torch.empty((rows, 1), dtype=torch.int32, device=dev)
        eng.enable_profiling(True)
        for _ in range(2):
            eng._run_bmu(eng.X, rows, eng.ldx, x16, eng.W[eng.cur], m, 1, False, idx, None, backend=(nat.BMU_TENSOR, 3))
        eng.phase_times_ms()
        for _ in range(reps):
            eng._run_bmu(eng.X, rows, eng.ldx, x16, eng.W[eng.cur], m, 1, False, idx, None, backend=(nat.BMU_TENSOR, 3))
        ph = eng.phase_times_ms()
        t = float(np.median(ph["bmu_candidates"]))
        tiles_per_sm = rows / 128 / 148
        print(f"M={m:6d}  {t:8.3f} ms  {2.0 * rows * m * d / t / 1e9:8.1f} TFLOP/s algorithmic  "
              f"{t * 1e-3 / tiles_per_sm * 1e6:8.2f} us per row tile  ({t * 1e-3 / tiles_per_sm / (m / 128) * 1e9:7.1f} ns per 128x128 tile)",
              flush=True)
        eng.close()


if __name__ == "__main__":
    main()
