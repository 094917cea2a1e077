"""Streamed against resident epochs (DESIGN.md, "Streaming fits").  Prints one JSON line.

    python tools/bench_stream.py [--epochs 10] [--warmup 2] [--beyond-hbm] [--out FILE]

  * raw H2D rate: a plain page-locked -> device copy of 4 GiB, the ceiling streaming can reach;
  * config 3 (10M x 256, 64 x 64 map) and the config-5 width on one GPU (625k x 4096, 128 x 128 map): resident and
    streamed epochs from the same start, timed alternately after warm-up; the streamed engine's effective H2D rate
    (float32 bytes of X per epoch over the epoch time), the staging threads' conversion rate, and the device time
    per phase of both (DBGSOM_PROFILE phases, from a separate profiled epoch);
  * --beyond-hbm: a 400M x 128 float32 X (205 GB of host RAM) that does not fit in device memory, planned
    automatically; reports epochs/s.  Skipped ("not measured") when the host lacks the RAM.

The samples are generated on the device (bench.make_shard) and copied to host memory once.  The card's name and
power limit and the host's free RAM are part of the record.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import bench  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def host_free_bytes():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


def raw_h2d(torch, nbytes=4 << 30, reps=5):
    host = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    host.fill_(1)
    dev = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dev.copy_(host, non_blocking=True)
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dev.copy_(host, non_blocking=True)
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    del host, dev
    torch.cuda.empty_cache()
    return {"bytes": nbytes, "ms": round(float(np.median(ts)), 2), "GBps": round(nbytes / np.median(ts) / 1e6, 2)}


def host_data(torch, n, d, k):
    X_dev = bench.make_shard(torch, torch.device("cuda"), n, d, k, 0)
    X = np.empty((n, d), dtype=np.float32)
    step = 1 << 20
    for s in range(0, n, step):
        X[s : s + step] = X_dev[s : s + step].cpu().numpy()
    del X_dev
    torch.cuda.empty_cache()
    return X


def make_engine(X, side, stream_rows):
    from dbgsom_b200.engine import DeviceEngine
    from dbgsom_b200.topology import MapTopology

    m = side * side
    eng = DeviceEngine(device="cuda", capacity_hint=m)
    eng.stream_rows = stream_rows
    eng.load_data(X, None, 0)
    eng.init_map_from_rows(np.random.default_rng(0).choice(X.shape[0], m, replace=False), capacity=m)
    eng.set_hops_from_topology(MapTopology.full_grid(side, side))
    return eng


def timed_epoch(torch, eng, epoch, m):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.epoch(bench.sigma_at(epoch, m), True, False)  # ends in the tail read-back (synchronises)
    return (time.perf_counter() - t0) * 1e3


def compare(torch, name, n, d, side, epochs, warmup, stream_rows):
    X = host_data(torch, n, d, 64)
    m = side * side
    res = make_engine(X, side, 0)
    st = make_engine(X, side, stream_rows)
    assert not res.streaming and st.streaming
    for e in range(warmup):
        timed_epoch(torch, res, e, m)
        timed_epoch(torch, st, e, m)
    t_res, t_st = [], []
    stager = st._stager
    b0, f0 = stager.bytes_staged, stager.fill_seconds
    for e in range(warmup, warmup + epochs):  # alternately, from the same epoch count
        t_res.append(timed_epoch(torch, res, e, m))
        t_st.append(timed_epoch(torch, st, e, m))
    staged, fill_s = stager.bytes_staged - b0, stager.fill_seconds - f0
    rescore = {}
    for label, eng in (("resident", res), ("streamed", st)):
        eng.bmu_stats_host(reset=True)
        timed_epoch(torch, eng, warmup + epochs, m)
        b = eng.bmu_stats_host(reset=True)
        rescore[label] = {k: b[k] for k in ("ambiguous", "flagged", "full_rescans", "selective_searches", "classic_searches")}
    phases = {}
    for label, eng in (("resident", res), ("streamed", st)):
        eng.enable_profiling(True)
        timed_epoch(torch, eng, warmup + epochs, m)
        phases[label] = {k: round(float(np.sum(v)), 3) for k, v in eng.phase_times_ms().items()}
        eng.enable_profiling(False)
    x_bytes = n * st.ldx * 4
    out = {
        "workload": name, "n": n, "d": d, "map": f"{side}x{side}", "chunk_rows": st.chunk_rows, "chunks": len(st.chunks),
        "epochs": epochs, "resident_ms": round(float(np.median(t_res)), 2), "streamed_ms": round(float(np.median(t_st)), 2),
        "resident_ms_all": [round(t, 2) for t in t_res], "streamed_ms_all": [round(t, 2) for t in t_st],
        "x_bytes_per_epoch": x_bytes,
        "effective_h2d_GBps": round(x_bytes / np.median(t_st) / 1e6, 2),
        "staging_workers": stager.workers,
        "staging_GBps_per_worker": round(staged / fill_s / 1e9, 2) if fill_s > 0 else None,
        "staging_GBps_aggregate_bound": round(staged / fill_s / 1e9 * stager.workers, 2) if fill_s > 0 else None,
        "device_ms_per_phase": phases,
        "rescore_one_epoch": rescore,
    }
    res.close()
    st.close()
    del X
    torch.cuda.empty_cache()
    return out


def beyond_hbm(torch, epochs):
    n, d, side = 400_000_000, 128, 64
    need = n * d * 4
    free = host_free_bytes()
    if free < 1.25 * need:
        return {"workload": "400M x 128", "status": "not measured", "reason": f"host has {free} free bytes, needs {need}"}
    X = host_data(torch, n, d, 64)
    eng = make_engine(X, side, 0)  # automatic plan: the resident fit does not fit
    m = side * side
    t = [timed_epoch(torch, eng, e, m) for e in range(epochs)]
    out = {"workload": "400M x 128", "streaming": eng.streaming, "chunk_rows": eng.chunk_rows, "chunks": len(eng.chunks),
           "epoch_ms_all": [round(x, 1) for x in t], "epochs_per_s": round(1e3 / float(np.median(t[1:] or t)), 3)}
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--only", choices=["c3", "c5w"], default=None)
    ap.add_argument("--beyond-hbm", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench_stream.py needs a CUDA device")
    rec = {"card": card(), "host_free_bytes": host_free_bytes(), "cpu_count": os.cpu_count(), "raw_h2d": raw_h2d(torch)}
    if args.only in (None, "c3"):
        rec["c3"] = compare(torch, "c3", 10_000_000, 256, 64, args.epochs, args.warmup, 1 << 19)
    if args.only in (None, "c5w"):
        rec["c5_width"] = compare(torch, "c5_width_1gpu", 625_000, 4096, 128, args.epochs, args.warmup, 1 << 15)
    rec["beyond_hbm"] = beyond_hbm(torch, 3) if args.beyond_hbm else {"status": "not measured", "reason": "not requested"}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
