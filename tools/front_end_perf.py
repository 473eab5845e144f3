"""Front-end throughput: KinoAstar searches on host threads (ualm_front_end_batch) versus the GPU (ualm_front_end_batch_device).

For each terrain (the reference's when maps_built/<name>.umap exists, else its seeded stand-in) and B in {512, 4096}, on the
(start, goal) stream problems.generate_astar draws from (same Rng, bounds and min_dist, every pair kept):
  host      the host batch on all usable cores (os.sched_getaffinity), wall clock, best of `--reps`;
  kernel    the device search kernel alone, CUDA events, median of `--reps` after one warm-up call;
  device    the whole device entry, wall clock: H2D, search, D2H of the polylines and the host resample.
Prints pairs/s and writes profiles/front_end_perf_<tag>.json with the card's name and power limit.

    python tools/front_end_perf.py [--batches 512 4096] [--reps 3] [--tag b200]
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


def pairs(B, seed=0, lo=-4.5, hi=4.5, min_dist=1.5):
    """the first B (start, goal) candidates of problems.generate_astar's stream"""
    from uneven_planner_b200 import problems
    rng = problems.Rng(seed)
    s, e = [], []
    while len(s) < B:
        a = np.array([rng.uniform(lo, hi), rng.uniform(lo, hi), rng.uniform(-np.pi, np.pi)])
        b = np.array([rng.uniform(lo, hi), rng.uniform(lo, hi), rng.uniform(-np.pi, np.pi)])
        if np.hypot(*(a[:2] - b[:2])) < min_dist:
            continue
        s.append(a); e.append(b)
    return np.array(s), np.array(e)


def card():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        info["nvidia_smi"] = None
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 4096])
    ap.add_argument("--terrains", nargs="+", default=["hill", "desert", "volcano", "forest"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--tag", default="b200")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("front_end_perf: no CUDA device (the device timings need one)")
    from uneven_planner_b200 import api, configs, front_end, maps
    ncores = len(os.sched_getaffinity(0))
    opt = api.BatchALMTrajOpt()
    rows = []
    for name in args.terrains:
        m = maps.terrain_or_standin(name)
        standin = maps.get_terrain(name, build_if_missing=False) is None
        view = front_end.MapView(m, configs.TERRAINS[name]["min_cnormal"], configs.TERRAINS[name]["max_rho"])
        for B in args.batches:
            s, e = pairs(B)
            host = []
            for _ in range(args.reps):
                t0 = time.perf_counter(); pbh, packh, nexph = front_end.plan_batch(view, s, e, nthreads=ncores); host.append(time.perf_counter() - t0)
            front_end.plan_batch_device(opt, view, s, e)                       # warm-up: module load, map upload, workspaces
            kern, wall = [], []
            for _ in range(args.reps):
                t = {}
                t0 = time.perf_counter(); pbd, packd, nexpd = front_end.plan_batch_device(opt, view, s, e, timing=t); wall.append(time.perf_counter() - t0)
                kern.append(t["search_ms"] / 1e3)
            row = {"terrain": name, "standin": standin, "B": B, "host_threads": ncores,
                   "packed_host": int(pbh.B), "packed_device": int(pbd.B), "mean_closed_nodes": float(nexpd.mean()), "max_closed_nodes": int(nexpd.max()),
                   "host_s": min(host), "kernel_s": float(np.median(kern)), "device_entry_s": float(np.median(wall))}
            for k in ("host", "kernel", "device_entry"):
                row[k + "_pairs_per_s"] = B / row[k + "_s"]
            rows.append(row)
            print(f"{name:8s} B={B:5d}  host {row['host_pairs_per_s']:9.0f} pairs/s ({ncores} threads)   kernel {row['kernel_pairs_per_s']:9.0f} pairs/s"
                  f"   device entry {row['device_entry_pairs_per_s']:9.0f} pairs/s   packed {pbh.B}/{pbd.B}   mean closed {nexpd.mean():.0f}", flush=True)
    opt.close()
    out = {"card": card(), "host_cpu_threads": ncores, "reps": args.reps, "rows": rows,
           "note": "host = ualm_front_end_batch (libm trig) on all usable cores; kernel = CUDA-event time of the search kernel; device entry = "
                   "wall clock of ualm_front_end_batch_device incl. H2D, D2H and the host resample. Pairs: problems.generate_astar's stream, seed 0."}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, f"front_end_perf_{args.tag}.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
