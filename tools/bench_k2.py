"""Micro-benchmark of K2 (dbgsom_accumulate) alone: CUDA-event time per launch and achieved HBM GB/s.

    python tools/bench_k2.py [rows] [D] [M] [live]

`live` < M leaves M - live neurons without samples (the collapsed maps of a real trajectory).
"""
import sys, os, json
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dbgsom_b200 import _native as nat

n = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
d = int(sys.argv[2]) if len(sys.argv) > 2 else 256
m = int(sys.argv[3]) if len(sys.argv) > 3 else 4096
live = int(sys.argv[4]) if len(sys.argv) > 4 else m
lib = nat.load()
dev = torch.device("cuda", 0)
g = torch.Generator(device=dev).manual_seed(1)
X = torch.empty((n, d), dtype=torch.float32, device=dev)
for s in range(0, n, 1 << 20):
    X[s:s + (1 << 20)] = torch.randn(min(1 << 20, n - s), d, device=dev, generator=g)
bmu = (torch.randint(0, live, (n,), device=dev, generator=g) * (m // live)).to(torch.int32)
W = torch.randn(m, d, device=dev, generator=g, dtype=torch.float64)
part = torch.zeros(m * d + 3 * m, dtype=torch.float64, device=dev)
ws = torch.empty(lib.dbgsom_accumulate_workspace_bytes(n, m, d), dtype=torch.uint8, device=dev)
a = nat.AccumulateArgs()
a.d_X, a.N, a.D, a.ldx = X.data_ptr(), n, d, d
a.d_bmu, a.d_W, a.M = bmu.data_ptr(), W.data_ptr(), m
a.inv_total_variance = 1.0 / (2.0 * d)
a.d_part, a.d_labels, a.n_classes, a.d_class_hist = part.data_ptr(), None, 0, None
a.d_workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
stream = torch.cuda.current_stream().cuda_stream
for _ in range(3):
    nat.check(lib.dbgsom_accumulate(a, stream), "accumulate")
torch.cuda.synchronize()
ev = [torch.cuda.Event(enable_timing=True) for _ in range(11)]
ev[0].record()
for i in range(10):
    nat.check(lib.dbgsom_accumulate(a, stream), "accumulate")
    ev[i + 1].record()
torch.cuda.synchronize()
ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(10)]
bytes_ = n * (4.0 * d + 8) + 4.0 * (m * d + 3 * m)
# reference values (float64 torch) on a slice for a sanity check of the sums
nn = min(n, 200_000)
a.N = nn
nat.check(lib.dbgsom_accumulate(a, stream), "accumulate")
torch.cuda.synchronize()
Xs, bs = X[:nn].double(), bmu[:nn].long()
dist = (Xs - W[bs]).pow(2).sum(1).sqrt()
k = 1 - torch.sqrt(1 - torch.exp(-a.inv_total_variance * dist * dist))
Sk = torch.zeros(m, d, dtype=torch.float64, device=dev).index_add_(0, bs, Xs * k[:, None])
E = torch.zeros(m, dtype=torch.float64, device=dev).index_add_(0, bs, dist)
err_S = float((part[: m * d].view(m, d) - Sk).abs().max() / Sk.abs().max())
err_E = float((part[m * d + 2 * m:] - E).abs().max() / E.abs().max())
print(json.dumps({"rows": n, "D": d, "M": m, "live": live, "rows_env": os.environ.get("DBGSOM_ACC_ROWS"),
                  "ms_median": float(np.median(ms)), "ms_min": min(ms),
                  "GBps_median": bytes_ / (np.median(ms) * 1e-3) / 1e9, "relerr_Sk": err_S, "relerr_E": err_E}))
