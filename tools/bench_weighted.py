"""Cost of frequency weights (`sample_weight`) in the training epoch, config 3 (10M x 256 per GPU, 64 x 64 map,
samples resident in HBM).

Three engines share one sample matrix: unweighted, random integer weights 1..4, and fractional weights with 10 %
zeros.  They run their epochs in alternating rounds in one process, with CUDA-event times per phase
(`enable_profiling`).  With --parent DIR (a checkout of the parent commit, library built), `bench.py` of this tree
and of DIR run alternately as separate processes, for the unweighted epoch of both.  One JSON document, with the
card's name and power limit, goes to --out.

    python tools/bench_weighted.py --out profiles/bench_weighted_b200.json [--parent DIR]
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


def card_info():
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [c.strip() for c in q.split(",")]
        info.update(name=name, power_limit=power, sm_clock_max=clock)
    except Exception as exc:  # the name from torch stays; the power limit is then unknown
        info["power_limit"] = f"unavailable ({exc!r:.80})"
    return info


def weighted_epochs(args):
    import torch

    import bench
    from dbgsom_b200.engine import DeviceEngine
    from dbgsom_b200.topology import MapTopology

    dev = torch.device("cuda", 0)
    n, d, side = args.rows, args.d, args.side
    m = side * side
    X = bench.make_shard(torch, dev, n, d, 64, 0)
    g = torch.Generator(device=dev).manual_seed(77)
    w_int = torch.randint(1, 5, (n,), device=dev, generator=g).to(torch.float64)
    w_frac = torch.rand(n, device=dev, generator=g, dtype=torch.float64) * 2.0
    w_frac[torch.rand(n, device=dev, generator=g) < 0.1] = 0.0
    positive = torch.nonzero(w_frac > 0).view(-1).cpu().numpy()
    rows = positive[np.random.default_rng(0).choice(positive.size, m, replace=False)]
    engines = {}
    for name, w in (("unweighted", None), ("int_1_4", w_int), ("frac_10pct_zero", w_frac)):
        eng = DeviceEngine(device="cuda:0", bmu_backend="auto")
        eng.load_device_data(X, weight_dev=w)
        eng.init_map_from_rows(rows, capacity=m)
        eng.set_hops_from_topology(MapTopology.full_grid(side, side))
        engines[name] = [eng, 0]
    for eng_ep in engines.values():  # warm-up: module loads, first selective search, resort
        for _ in range(args.warmup):
            eng_ep[0].epoch(bench.sigma_at(eng_ep[1], m), True, False)
            eng_ep[1] += 1
    rec = {name: {"epoch_ms": [], "k2_ms": [], "phases_ms": []} for name in engines}
    for _ in range(args.rounds):
        for name, eng_ep in engines.items():
            eng = eng_ep[0]
            torch.cuda.synchronize(dev)
            eng.enable_profiling(True)
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(args.epochs):
                eng.epoch(bench.sigma_at(eng_ep[1], m), True, False)
                eng_ep[1] += 1
            t1.record()
            torch.cuda.synchronize(dev)
            ph = eng.phase_times_ms()
            eng.enable_profiling(False)
            rec[name]["epoch_ms"].append(t0.elapsed_time(t1) / args.epochs)
            rec[name]["k2_ms"].append(float(np.mean(ph["accumulate"])))
            rec[name]["phases_ms"].append({k: round(float(np.mean(v)), 4) for k, v in ph.items()})
    for eng_ep in engines.values():
        eng_ep[0].close()
    med = {name: {"epoch_ms": float(np.median(r["epoch_ms"])), "k2_ms": float(np.median(r["k2_ms"]))}
           for name, r in rec.items()}
    u = med["unweighted"]
    targets = {}
    for name in ("int_1_4", "frac_10pct_zero"):
        k2 = med[name]["k2_ms"] / u["k2_ms"]
        ep = med[name]["epoch_ms"] / u["epoch_ms"]
        targets[name] = {"k2_ratio": round(k2, 4), "k2_target": 1.10, "k2_met": k2 <= 1.10,
                         "epoch_ratio": round(ep, 4), "epoch_target": 1.03, "epoch_met": ep <= 1.03}
    return {"rounds": rec, "median": med, "targets": targets}


def parent_comparison(args):
    """bench.py of this tree and of the parent tree, alternately, each its own process (unweighted epochs)."""
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.bench_steps), "--warmup", "3", "--no-strong",
           "--no-fit"]
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = {"this": [], "parent": []}
    for _ in range(args.parent_rounds):
        for who, tree in (("this", ROOT), ("parent", os.path.abspath(args.parent))):
            res = subprocess.run(cmd, cwd=tree, env=env, capture_output=True, text=True)
            line = next((ln for ln in res.stdout.splitlines()[::-1] if ln.startswith("{")), None)
            if res.returncode != 0 or line is None:
                out[who].append({"error": (res.stderr or res.stdout)[-400:]})
                continue
            r = json.loads(line)
            out[who].append({"ms_per_step": r.get("ms_per_step"), "value": r.get("value")})
    ms = {k: [x["ms_per_step"] for x in v if "ms_per_step" in x] for k, v in out.items()}
    summary = {k: {"median_ms": float(np.median(v)) if v else None, "min_ms": min(v) if v else None,
                   "max_ms": max(v) if v else None} for k, v in ms.items()}
    if ms["this"] and ms["parent"]:
        spread = max(ms["parent"]) - min(ms["parent"])
        diff = float(np.median(ms["this"]) - np.median(ms["parent"]))
        summary["this_minus_parent_ms"] = diff
        summary["parent_spread_ms"] = spread
        summary["within_parent_spread"] = abs(diff) <= spread
    return {"runs": out, "summary": summary}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--d", type=int, default=256)
    ap.add_argument("--side", type=int, default=64)
    ap.add_argument("--epochs", type=int, default=10, help="epochs per engine and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--parent", default=None, help="checkout of the parent commit with its library built")
    ap.add_argument("--parent-rounds", type=int, default=3)
    ap.add_argument("--bench-steps", type=int, default=20)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    doc = {"workload": {"rows": args.rows, "d": args.d, "neurons": args.side**2, "resident": True,
                        "epochs_per_round": args.epochs, "rounds": args.rounds},
           "card": card_info(), "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    doc["weighted"] = weighted_epochs(args)
    if args.parent:
        doc["parent"] = parent_comparison(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps({"card": doc["card"], "median": doc["weighted"]["median"], "targets": doc["weighted"]["targets"],
                      "parent": doc.get("parent", {}).get("summary")}))


if __name__ == "__main__":
    main()
