#!/usr/bin/env python
"""Benchmark of the batch-SOM training epoch (BASELINE.json metric: training samples/s per epoch).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c4|c2|small] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one full training epoch (BMU search -> per-BMU accumulation -> [all-reduce] ->
neighbourhood smoothing -> read-back of per-neuron error/count/change) of a fixed side x side map on
synthetic Gaussian-mixture data, prototypes evolving from epoch to epoch exactly as in `fit`
(reference semantics incl. packed centre rows, sigma schedule of a 200-epoch fit).

Workloads (SURVEY.md section 8(d)); `c3` is the default at every GPU count (weak scaling: each GPU holds
10M x 256 samples, the only collective is the all-reduce of the M x D partial sums):
    c3     10M x 256 per GPU, 64 x 64 map           (BASELINE.json configs[2], the roofline config)
    c4     100M x 128 in total, sharded, 64 x 64    (configs[3], strong scaling)
    c2     70000 x 784, 20 x 20 map                 (configs[1]; latency-bound)
    c5     5M x 4096 in total, sharded, 128 x 128   (configs[4] at its final map size; needs 8 GPUs or --rows)
    small  200k x 64, 16 x 16 map                   (smoke-sized)

`--impl reference` times the CPU restatement of the reference's epoch (oracle/, numpy + the same
scikit-learn call the reference makes) on the host cores, on a bounded row sample of the workload.

`--dump-outputs DIR` writes what the last timed epoch computed to DIR/<name>.npy (float64): per-neuron `error`
and `counts`, `change`, the updated prototypes `weights` and the winners of the samples `winners` (rank 0's shard).
The inputs depend only on the arguments, so two builds can be compared output for output.  Outputs larger than
their share of 48 MB are a fixed, seeded row sample; the sampled row indices are written as `<name>_rows.npy`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to every rank.  The CPU legs of this script (the `--impl reference` arm, the
# cpu_baseline and the oracle parity check, all on rank 0) are meant to use the host's cores, and scikit-learn's
# OpenMP runtime reads the variable when it is first loaded -- so it is set here, before numpy / scikit-learn are
# imported.  Rank 0 takes every core in the reference arm (the other ranks exit at once); in our own arm the
# ranks share them.
_WORLD = max(1, int(os.environ.get("WORLD_SIZE", "1")))
_CORES = os.cpu_count() or 1
_THREADS = _CORES if "reference" in sys.argv else max(1, _CORES // _WORLD)
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_v] = str(_THREADS)

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # nothing is written into the tree the benchmark runs from (it may be read-only)

WORKLOADS = {
    #          rows per GPU (None = total/gpus), total rows, D, side, mixture components
    "c3": dict(per_gpu=10_000_000, total=None, d=256, side=64, k=64, name="SomVQ epoch, GMM 10M x 256 per GPU, fixed 64x64 map"),
    "c4": dict(per_gpu=None, total=100_000_000, d=128, side=64, k=64, name="SomVQ epoch, GMM 100M x 128 sharded, fixed 64x64 map"),
    "c2": dict(per_gpu=70_000, total=None, d=784, side=20, k=10, name="SomClassifier-shaped epoch, GMM 70000 x 784, 20x20 map"),
    "c5": dict(per_gpu=None, total=5_000_000, d=4096, side=128, k=64, name="SomVQ epoch, GMM 5M x 4096 sharded, fixed 128x128 map (16384 neurons)"),
    "small": dict(per_gpu=200_000, total=None, d=64, side=16, k=16, name="GMM 200k x 64, 16x16 map"),
}
N_ITER_SCHEDULE = 200  # sigma follows the coarse phase of a 200-epoch fit


def sigma_at(epoch: int, m: int) -> float:
    """dbgsom/BaseSom.py:863-902 with default hyper-parameters (exponential decay, coarse phase)."""
    from math import exp, sqrt

    s0, s1 = 0.2 * sqrt(m), max(0.7, 0.05 * sqrt(m))
    return s1 + (s0 - s1) * exp(-0.02 * (epoch / 0.5))


def grid_hops(side: int) -> np.ndarray:
    ii, jj = np.meshgrid(np.arange(side), np.arange(side), indexing="ij")
    p = np.stack([ii.ravel(), jj.ravel()], axis=1)
    return np.abs(p[:, None, :] - p[None, :, :]).sum(axis=2).astype(np.uint16)


def measured_peaks() -> dict:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        p["_source"] = "measured"
        return p
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


class ClockSampler:
    """nvidia-smi clock / throttle samples while the timed region runs."""

    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- data
def make_shard(torch, device, n, d, k, rank, chunk=1 << 20):
    """Synthetic Gaussian mixture shard generated on the device (centres N(0, 2^2), unit noise)."""
    gc = torch.Generator(device=device).manual_seed(20240)
    centers = torch.randn(k, d, device=device, generator=gc) * 2.0
    g = torch.Generator(device=device).manual_seed(1000 + rank)
    X = torch.empty((n, d), dtype=torch.float32, device=device)
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        lab = torch.randint(0, k, (e - s,), device=device, generator=g)
        X[s:e] = centers[lab]
        X[s:e] += torch.randn(e - s, d, device=device, generator=g)
    return X


def cpu_reference_epoch_rate(wl, n_sample, steps, warmup):
    """Oracle (CPU restatement of the reference epoch) on a bounded row sample; returns a dict."""
    from threadpoolctl import threadpool_limits

    from oracle import som_oracle as O

    # (the thread environment was set at the top of this file, before numpy / scikit-learn were loaded)
    threadpool_limits(limits=_THREADS)
    d, side, k = wl["d"], wl["side"], wl["k"]
    m = side * side
    X = O.gmm(n_sample, d, k, seed=0)
    rng = np.random.default_rng(0)
    W = X[rng.choice(n_sample, m, replace=False)].astype(np.float64)
    hop = grid_hops(side).astype(np.float64)
    V = float(O.total_variance(X.astype(np.float64)))
    X64 = X.astype(np.float64)  # same dtype as W: sklearn's ArgKmin64 path, like the reference on float64 input
    times, t_lin, t_const = [], [], []
    for e in range(warmup + steps):
        t0 = time.perf_counter()
        dist, win = O.bmu(X64, W, 1)
        kk = O.sample_weights(dist, V)
        C, n = O.voronoi_centers(kk, X64, win, m, pack=True)
        E = O.quantization_errors(win, dist, m)
        t1 = time.perf_counter()
        H = O.neighborhood(hop, sigma_at(e, m))
        W = O.smooth(C, n, H)
        t2 = time.perf_counter()
        if e >= warmup:
            times.append(t2 - t0)
            t_lin.append(t1 - t0)
            t_const.append(t2 - t1)
    return dict(t_step=float(np.mean(times)), t_linear=float(np.mean(t_lin)), t_smooth=float(np.mean(t_const)),
                n_sample=n_sample, E_checksum=float(E.sum()))


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_full = wl["per_gpu"] or wl["total"]
    n_sample = min(n_full, 100_000 if wl["side"] >= 32 else 70_000)
    r = cpu_reference_epoch_rate(wl, n_sample, args.steps, args.warmup)
    cores = os.cpu_count()
    # the CPU has ONE set of cores whatever --gpus says: its rate on the workload of one GPU is the rate on the
    # whole job.  BMU + update are linear in the rows (measured on the sample), the smoothing GEMM is not: the
    # value is rows / (linear part scaled to the full row count + smoothing), i.e. what the full workload would run at
    t_full = r["t_linear"] * n_full / n_sample + r["t_smooth"]
    value = n_full / t_full
    sample = (f"{n_sample} x {wl['d']} rows of the workload, full {wl['side']}x{wl['side']} map; numpy float64 + "
              f"sklearn NearestNeighbors (ArgKmin64), {_THREADS} threads; BMU+update {r['t_linear']:.3f}s (linear in rows, "
              f"scaled to {n_full} rows) + smoothing GEMM {r['t_smooth']:.3f}s (independent of rows) per epoch; "
              f"on the sample alone: {n_sample / r['t_step']:.4g} samples/s")
    line = {
        "impl": "reference", "metric": "training samples/sec/epoch", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["t_step"],
        "ms_per_step_note": "wall time of one step on the bounded row sample; `value` is the rate of the full workload "
                            "(row-linear part scaled, smoothing counted once)", "ms_per_step_full_workload": 1e3 * t_full,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"], "rows_timed": n_sample, "rows_scaled_to": n_full, "d": wl["d"],
                   "neurons": wl["side"] ** 2, "threads": _THREADS},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=args.out)


# ---------------------------------------------------------------------------------------------- ours
def bind_to_gpu_cpus(local: int) -> dict:
    """Pin this rank (and with it the first-touch placement of its pinned host buffers) to the CPU cores of the
    NUMA node its GPU hangs off, as NVML reports them.  torchrun does not bind ranks; with all eight staging buffers
    on one socket the per-step H2D of the end-to-end leg crosses the socket link for half of the GPUs."""
    info = {"bound": False}
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [w * 64 + b for w, bits in enumerate(mask) for b in range(64) if (bits >> b) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"bound": True, "cpus": f"{allowed[0]}-{allowed[-1]}", "n_cpus": len(allowed)}
        try:
            info["numa_node"] = int(open(f"/sys/bus/pci/devices/{pynvml.nvmlDeviceGetPciInfo(h).busId.lower()[4:]}/numa_node").read())
        except Exception:
            pass
    except Exception as exc:
        info["error"] = repr(exc)[:120]
    return info


def build_engine(torch, device, wl, n_local, rank, world, backend):
    from dbgsom_b200.engine import DeviceEngine
    from dbgsom_b200.topology import MapTopology

    d, side, k = wl["d"], wl["side"], wl["k"]
    m = side * side
    X = make_shard(torch, device, n_local, d, k, rank)
    eng = DeviceEngine(device=str(device), bmu_backend=backend, distributed=world > 1)
    eng.load_device_data(X)
    rows = np.random.default_rng(0).choice(eng.n_samples_global, m, replace=False)
    eng.init_map_from_rows(rows, capacity=m)
    # all-pairs hop counts of the side x side grid: BFS on the device from the adjacency table (dbgsom_hops)
    eng.set_hops_from_topology(MapTopology.full_grid(side, side))
    return eng, X


def timed_epochs(torch, eng, m, steps, warmup, device, world, epoch0=0, sampler=None):
    """W warm-up epochs, then K epochs between barrier + synchronize, CUDA events, max over ranks."""
    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(device)

    epoch = epoch0
    for _ in range(warmup):
        eng.epoch(sigma_at(epoch, m), True, False)
        epoch += 1
    eng.enable_profiling(True)
    eng.bmu_stats_host(reset=True)
    launches0 = eng.launches
    barrier()
    if sampler is not None:
        sampler.start()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    out = None
    for _ in range(steps):
        out = eng.epoch(sigma_at(epoch, m), True, False)
        epoch += 1
    t1.record()
    barrier()
    clocks = sampler.stop() if sampler is not None else None
    elapsed_ms = t0.elapsed_time(t1)
    res = {"launches": eng.launches - launches0, "bmu_stats": eng.bmu_stats_host(), "phases": eng.phase_times_ms(),
           "clocks": clocks, "out": out, "epoch": epoch}
    eng.enable_profiling(False)
    if world > 1:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device=device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    res["elapsed_ms"] = elapsed_ms
    return res


DUMP_WEIGHT_VALUES = 4 << 20   # 32 MB of float64 prototypes
DUMP_WINNER_ROWS = 1 << 20     # 8 MB of winners + 8 MB of their row indices


def dump_outputs(path, eng, out):
    """Write the result of the engine's last epoch (`out` is what `epoch` returned) to path/<name>.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = {"error": out["error"], "counts": out["counts"], "change": np.array([out["change"]])}
    W = eng.weights()
    if W.size > DUMP_WEIGHT_VALUES:
        arrays["weights_rows"] = np.sort(np.random.default_rng(1).choice(W.shape[0], DUMP_WEIGHT_VALUES // W.shape[1],
                                                                        replace=False))
        W = W[arrays["weights_rows"]]
    arrays["weights"] = W
    win = eng.idx.view(-1)[: eng.N]
    if eng.N > DUMP_WINNER_ROWS:
        arrays["winners_rows"] = np.sort(np.random.default_rng(2).choice(eng.N, DUMP_WINNER_ROWS, replace=False))
        win = win[eng.torch.from_numpy(arrays["winners_rows"]).to(win.device)]
    arrays["winners"] = win.cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def k1_time_ms(phases):
    """Whole BMU search per epoch: candidate kernel(s) + second stage + exact re-score (everything between the
    prototype shadows and the final winner indices)."""
    mean = lambda xs: float(np.mean(xs)) if xs else 0.0  # noqa: E731
    per_epoch = lambda name: float(np.sum(phases.get(name, []))) / max(1, len(phases.get("accumulate", [1])))  # noqa: E731
    return {"candidates": per_epoch("bmu_candidates"), "resolve": per_epoch("bmu_resolve"),
            "second_stage": per_epoch("bmu_second_stage"), "resort": per_epoch("resort"),
            "accumulate": mean(phases.get("accumulate"))}


def parity_check(torch, device, rank, world, backend="tensor"):
    """N >= 1 parity evidence in the bench line itself: a small sharded fit-like run (config-3 feature width and map,
    enough rows that every rank runs the CTA-pair tcgen05 kernel) -- two epochs through the distributed engine, the
    second one compared on rank 0 with the float64 oracle fed the device's prototypes of epoch 1: winners outside
    the 1e-6 near-tie gate, then (teacher-forced on the exempt samples) counts, E and the updated prototypes."""
    from dbgsom_b200.engine import DeviceEngine
    from dbgsom_b200.topology import MapTopology

    d, side = 256, 64
    m = side * side
    per = 19_200  # >= 148 row tiles of 128 per rank
    n = per * world
    from oracle import som_oracle as O

    X = O.gmm(n, d, 64, seed=5)
    sl = slice(rank * per, (rank + 1) * per)
    eng = DeviceEngine(device=str(device), bmu_backend=backend, distributed=world > 1)
    stats = eng.load_data(X[sl], None, 0)
    eng.init_map_from_rows(np.random.default_rng(2).choice(n, m, replace=False), capacity=m)
    eng.set_hops_from_topology(MapTopology.full_grid(side, side))
    eng.epoch(sigma_at(0, m), True, False)
    W1 = eng.weights()
    r = eng.epoch(sigma_at(1, m), True, False)
    W2 = eng.weights()
    win_local = eng.idx.view(-1)[:per].contiguous()
    if world > 1:
        parts = [torch.empty_like(win_local) for _ in range(world)]
        torch.distributed.all_gather(parts, win_local)
        win = torch.cat(parts).cpu().numpy().astype(np.int64)
    else:
        win = win_local.cpu().numpy().astype(np.int64)
    be = eng.last_backend
    eng.close()
    if rank != 0:
        return None
    X64 = X.astype(np.float64)
    _, ref_win, gap = O.bmu_with_gap(X64, W1)
    strict = gap >= 1e-6
    ref = O.epoch_step(X64, W1, grid_hops(side).astype(np.float64), sigma_at(1, m), stats["total_variance"], pack=True,
                       winners=win)
    scale = np.abs(ref["W_new"]).max()
    with np.errstate(divide="ignore", invalid="ignore"):
        rel_e = np.abs(r["error"] - ref["E"]) / np.maximum(np.abs(ref["E"]), 1e-6)
    return {"rows": int(n), "ranks": world, "d": d, "neurons": m, "backend": "tcgen05 x%d" % be[1] if be[0] == 1 else "simt",
            "rows_outside_gate": int(strict.sum()),
            "bmu_mismatch_outside_gate": int(np.count_nonzero((win != ref_win) & strict)),
            "bmu_differences_inside_gate": int(np.count_nonzero((win != ref_win) & ~strict)),
            "counts_equal": bool(np.array_equal(r["counts"], ref["n"])),
            "max_rel_W": float(np.abs(W2 - ref["W_new"]).max() / scale), "max_rel_E": float(rel_e.max()),
            "dead_neurons": int((ref["n"] == 0).sum())}


def fit_config2():
    """Fit-level wall time through the estimator API at BASELINE.json configs[1] (SomClassifier, 70000 x 784 ten-class
    mixture from host memory, growth towards 400 neurons): upload, every epoch, host growth, post-training passes."""
    from dbgsom_b200 import SomClassifier
    from oracle import som_oracle as O

    X, y = O.gmm(70_000, 784, 10, seed=21, return_labels=True)
    est = SomClassifier(max_neurons=400, n_iter=240, random_state=0)
    est.fit(X[:2000], y[:2000])  # untimed: library load, allocator warm-up
    t0 = time.perf_counter()
    est.fit(X, y)
    dt = time.perf_counter() - t0
    epochs = est.n_iter_ + 1
    return {"seconds": dt, "epochs": epochs, "neurons": len(est.neurons_), "epochs_per_s": epochs / dt,
            "samples_per_s_per_epoch": 70_000 * epochs / dt, "quantization_error": float(est.quantization_error_),
            "api": "SomClassifier(max_neurons=400, n_iter=240, random_state=0).fit(X, y), host numpy in, fitted attributes out"}


def run_ours(args, wl):
    import torch

    from dbgsom_b200 import _native as nat

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    affinity = bind_to_gpu_cpus(local) if world > 1 else {"bound": False}
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    device = torch.device("cuda", local)
    torch.cuda.set_device(device)
    n_gpus = world

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(device)

    d, side = wl["d"], wl["side"]
    m = side * side
    n_local = wl["per_gpu"] if wl["per_gpu"] else wl["total"] // n_gpus
    scaling = "weak" if wl["per_gpu"] else "strong"
    if args.rows:
        n_local = args.rows
    eng, X = build_engine(torch, device, wl, n_local, rank, world, args.backend)
    n_global = eng.n_samples_global

    # ------------------------------------------------------------------ timed region (device resident)
    res = timed_epochs(torch, eng, m, args.steps, args.warmup, device, world, sampler=ClockSampler(local))
    elapsed_ms, launches, bmu_stats, phases, clocks, out = (res[k_] for k_ in ("elapsed_ms", "launches", "bmu_stats", "phases", "clocks", "out"))
    epoch = res["epoch"]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, out)  # before the end-to-end leg trains the map further
    ms_per_step = elapsed_ms / args.steps
    value = n_global * args.steps / (elapsed_ms * 1e-3)

    peaks = measured_peaks()
    be, n_pass = eng.last_backend
    mean = lambda xs: float(np.mean(xs)) if xs else None  # noqa: E731
    k1 = k1_time_ms(phases)
    t_k1 = k1["candidates"] + k1["second_stage"] + k1["resolve"] + k1["resort"]
    t_acc = k1["accumulate"]
    flops = 2.0 * n_local * m * d
    passes = bmu_stats.get("mma_passes")
    roof = {
        "kernel": "bmu_cand_tensor_kernel" if be == nat.BMU_TENSOR else "bmu_cand_simt_kernel",
        "bound": "tensor", "unit": "TFLOP/s",
        "achieved": flops / (t_k1 * 1e-3) / 1e12 if t_k1 else None,
        "peak": peaks["bf16_tflops_sustained"], "peak_source": peaks["_source"] + " (sustained cuBLAS bf16)",
        "traffic": None, "ms_per_launch": t_k1, "ms_candidates": k1["candidates"], "ms_second_stage": k1["second_stage"],
        "ms_resolve": k1["resolve"], "ms_resort": k1["resort"], "algorithmic_flops_per_launch": flops,
        "time_basis": "whole BMU search per epoch: FLAG / candidate kernel + REFINE kernel + exact float64 re-score + the "
                      "amortised re-sort of the sample shadows",
        "refined_share": bmu_stats.get("refined_share"),
        "mma_passes": (passes if passes is not None else n_pass) if be == nat.BMU_TENSOR else 0,
    }
    roof["frac"] = roof["achieved"] / roof["peak"] if roof["achieved"] else None
    upd_bytes = n_local * (4.0 * d + 8.0) + 4.0 * (m * d + 3 * m)
    roof_upd = {
        "kernel": "dbgsom_accumulate (histogram + scan + scatter + segmented accumulate)", "bound": "hbm", "unit": "GB/s",
        "achieved": upd_bytes / (t_acc * 1e-3) / 1e9 if t_acc else None, "peak": peaks["hbm_gbs"],
        "peak_source": peaks["_source"] + " (copy)", "traffic": None, "ms_per_launch": t_acc,
        "algorithmic_bytes_per_launch": upd_bytes,
    }
    roof_upd["frac"] = roof_upd["achieved"] / roof_upd["peak"] if roof_upd["achieved"] else None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tr = json.load(f).get(args.workload, {})
        roof["traffic"] = tr.get(roof["kernel"])
        roof_upd["traffic"] = tr.get("accumulate_kernel")
        roof["traffic_source"] = roof_upd["traffic_source"] = tr.get("source", "profiles/ncu_traffic.json (one ncu --set full capture, scaled per launch)")
    except Exception:
        pass

    # ------------------------------------------------------------------ end to end (host buffers)
    e2e = None
    if not args.no_e2e:
        try:
            host = torch.empty((n_local, d), dtype=torch.float32, pin_memory=True)
            host.copy_(X)
            torch.cuda.synchronize(device)
            k_e2e = max(1, min(args.steps, 3))
            eng.epoch_from_host(host, sigma_at(epoch, m), True, False)  # untimed: one-off stream / workspace setup
            epoch += 1
            barrier()
            w0 = time.perf_counter()
            step_ms = []
            for _ in range(k_e2e):
                ws = time.perf_counter()
                # H2D of this step's samples in row chunks on a copy stream; the fp16 shadow and the BMU
                # search of a chunk run while the next one is in flight; reads back error/count/change
                r = eng.epoch_from_host(host, sigma_at(epoch, m), True, False)
                w_host = eng.weights()                 # D2H of the prototypes (the step's result)
                epoch += 1
                step_ms.append(round(1e3 * (time.perf_counter() - ws), 2))
            barrier()
            dt = time.perf_counter() - w0
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=device)
                torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
                dt = float(t.item())
            e2e = {"value": n_global * k_e2e / dt, "unit": "samples/s", "steps": k_e2e, "step_ms": step_ms,
                   "h2d_bytes_per_step": int(n_local * d * 4), "d2h_bytes_per_step": int(w_host.nbytes + 8 * (3 * m + 5)),
                   "h2d_gbs_per_gpu": n_local * d * 4 / (min(step_ms) * 1e-3) / 1e9, "cpu_affinity": affinity,
                   "note": "per step: H2D of all samples from pinned host memory (chunked, overlapped with the fp16 shadow rebuild and the BMU search), update, smoothing, D2H of prototypes and per-neuron error"}
            del host
        except Exception as exc:  # e.g. pinned allocation refused
            e2e = {"value": None, "unit": "samples/s", "error": repr(exc)[:200]}

    eng.close()
    del eng, X
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ north-star scaling record (config 4, strong)
    strong = None
    if args.workload == "c3" and not args.no_strong and not args.rows:
        try:
            wl4 = WORKLOADS["c4"]
            n4 = wl4["total"] // n_gpus
            eng4, X4 = build_engine(torch, device, wl4, n4, rank, world, args.backend)
            k4, w4 = max(3, min(args.steps, 5)), 3
            r4 = timed_epochs(torch, eng4, m, k4, w4, device, world)
            kk = k1_time_ms(r4["phases"])
            t4 = kk["candidates"] + kk["second_stage"] + kk["resolve"] + kk["resort"]
            f4 = 2.0 * n4 * 4096 * wl4["d"]
            b4 = n4 * (4.0 * wl4["d"] + 8.0) + 4.0 * (4096 * wl4["d"] + 3 * 4096)
            strong = {
                "workload": wl4["name"], "scaling": "strong", "rows_total": eng4.n_samples_global, "rows_per_gpu": n4,
                "d": wl4["d"], "neurons": 4096, "steps": k4, "warmup": w4, "ms_per_step": r4["elapsed_ms"] / k4,
                "value": eng4.n_samples_global * k4 / (r4["elapsed_ms"] * 1e-3), "unit": "samples/s",
                "phases_ms": {k_: float(np.sum(v)) / k4 for k_, v in r4["phases"].items()},
                "k1_frac_of_tensor_peak": f4 / (t4 * 1e-3) / 1e12 / peaks["bf16_tflops_sustained"] if t4 else None,
                "k2_frac_of_hbm_peak": b4 / (kk["accumulate"] * 1e-3) / 1e9 / peaks["hbm_gbs"] if kk["accumulate"] else None,
                "mma_passes": r4["bmu_stats"].get("mma_passes"), "refined_share": r4["bmu_stats"].get("refined_share"),
                "note": "fixed 100M x 128 rows split over the ranks (all of them on one GPU at N = 1); speed-up vs N = 1 "
                        "is this record's value at N over the N = 1 run's",
            }
            eng4.close()
            del eng4, X4
            torch.cuda.empty_cache()
        except Exception as exc:
            strong = {"error": repr(exc)[:300]}

    parity = None
    if not args.no_parity:
        try:
            parity = parity_check(torch, device, rank, world)
        except Exception as exc:
            parity = {"error": repr(exc)[:300]}

    cpu = fit2 = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu:
        n_sample = min(n_local, 100_000 if side >= 32 else 70_000)
        r = cpu_reference_epoch_rate(wl, n_sample, 2, 1)
        full = n_local / (r["t_linear"] * n_local / n_sample + r["t_smooth"])
        cpu = {"value": full, "unit": "samples/s", "cores": _THREADS, "kind": "port",
               "sample": (f"{n_sample} rows of the workload, full map; BMU+update {r['t_linear']:.3f}s scaled linearly to "
                          f"{n_local} rows + smoothing GEMM {r['t_smooth']:.3f}s; measured on the sample: "
                          f"{n_sample / r['t_step']:.4g} samples/s")}
    if rank == 0 and n_gpus == 1 and not args.no_fit:
        try:
            fit2 = fit_config2()
        except Exception as exc:
            fit2 = {"error": repr(exc)[:300]}

    if rank == 0:
        line = {
            "metric": "training samples/sec/epoch", "value": value, "unit": "samples/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f16 tensor cores (tcgen05) + f64 re-score / f64 update / f64 smoothing"
            if be == nat.BMU_TENSOR else "f32 search + f64 re-score / f64 update / f64 smoothing",
            "data": "synthetic",
            "config": {"workload": wl["name"], "rows_per_gpu": n_local, "rows_total": n_global, "d": d, "neurons": m,
                       "cache": "inputs (>= 10x L2) streamed from HBM every step, no flush needed"
                       if n_local * d * 4 > 1.2e9 else "inputs smaller than 10x L2",
                       "bmu_backend": {nat.BMU_TENSOR: f"tcgen05 fp16, n_pass mode {n_pass}", nat.BMU_SIMT: "fp32 CUDA cores"}[be],
                       "prototype_evolution": "real trajectory (reference semantics, packed rows), sigma schedule of a 200-epoch fit",
                       "parallelism": f"dp{n_gpus}"},
            "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
            "roofline": roof, "roofline_update": roof_upd, "cpu_baseline": cpu,
            "phases_ms": {k_: float(np.sum(v)) / args.steps for k_, v in phases.items()},
            "bmu_rescore_per_epoch": {k_: (v / args.steps if k_ not in ("mma_passes", "refined_share") else v)
                                      for k_, v in bmu_stats.items()}, "last_change": out["change"],
            "strong_c4": strong, "parity_check": parity, "fit_c2": fit2,
        }
        print(json.dumps(line), file=args.out)
    if world > 1:
        torch.distributed.destroy_process_group()


def _stdout_for_json_only():
    """Send everything libraries write to fd 1 (e.g. NCCL's version banner) to stderr; return a file for
    the one JSON line the driver parses."""
    sys.stdout.flush()
    keep = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(keep, "w")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--backend", default="auto", choices=["auto", "tensor", "tensor1", "simt"])
    ap.add_argument("--rows", type=int, default=0, help="override rows per GPU (debugging)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the config-4 strong-scaling sub-record")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity check of the sharded epoch")
    ap.add_argument("--no-fit", action="store_true", help="skip the config-2 fit-level record")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 0)
    wl = WORKLOADS[args.workload]
    args.out = _stdout_for_json_only()
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)
    args.out.flush()


if __name__ == "__main__":
    main()
