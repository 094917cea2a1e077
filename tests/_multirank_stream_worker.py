"""Worker of tests/test_gpu_streaming.py::test_two_streaming_ranks_equal_one_resident_gpu, run under torchrun with one
rank per GPU: every rank streams its own contiguous shard in chunks; rank 0 repeats the epochs on one GPU with all
samples resident and compares (the sums differ in summation order only)."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import _datasets  # noqa: E402
from _multirank_worker import run  # noqa: E402
from dbgsom_b200.engine import DeviceEngine  # noqa: E402
from dbgsom_b200.topology import MapTopology  # noqa: E402


def main():
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    n, d, c = 80000, 96, 5
    X, y = _datasets.gmm(n, d, c, 7, return_labels=True)
    topo = MapTopology.full_grid(32, 32)
    rows = np.random.default_rng(0).choice(n, len(topo), replace=False)
    sigmas = [2.0, 1.6, 1.2]
    per = -(-n // world)
    sl = slice(rank * per, min(n, (rank + 1) * per))
    eng = DeviceEngine(device=f"cuda:{local}", distributed=True, bmu_backend="tensor")
    eng.stream_rows = 12_800
    outs, W, st, hist = run(eng, X[sl], y[sl], c, rows, topo, sigmas)
    streamed = eng.streaming and len(eng.chunks) > 1
    eng.close()
    if rank == 0:
        from oracle import som_oracle as O

        assert streamed
        ref = DeviceEngine(device="cuda:0", distributed=False, bmu_backend="tensor")
        r_outs, r_W, r_st, r_hist = run(ref, X, y, c, rows, topo, sigmas)
        assert not ref.streaming
        ref.close()
        for a, b in zip(outs, r_outs):
            np.testing.assert_array_equal(a["counts"], b["counts"])
            np.testing.assert_allclose(a["error"], b["error"], rtol=1e-10)
            assert abs(a["change"] - b["change"]) <= 1e-9 * abs(b["change"])
        np.testing.assert_allclose(W, r_W, rtol=1e-10, atol=1e-12)
        for k in ("te_count", "qe_sum"):
            assert abs(st[k] - r_st[k]) <= 1e-10 * max(1.0, abs(r_st[k])), k
        _, _, gap_final = O.bmu_with_gap(X.astype(np.float64), W)
        near = int((gap_final < 1e-9).sum())
        assert np.abs(hist[0] - r_hist[0]).sum() <= 2 * near
        assert hist[0].sum() == r_hist[0].sum() == n
        print("MULTIRANK_STREAM_OK world=%d" % world, flush=True)
    dist.barrier()
    dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
