"""SOR defence timing: functional.sor and SORDefense.forward against the reference's torch float64 formulation on the
same GPU, with the mask agreement of the same run, the card name and its power limit, written as one JSON file.

    python tools/sor_bench.py --out DIR [--reps 30] [--warmup 5]

The working set (a few MB of coordinates and outputs) stays in the 126 MB L2 after the first pass, and the sweep is
bound by the FP64 pipe, not by memory, so the L2 is not flushed between repetitions.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
from oracle import sor_oracle as R  # noqa: E402

F = pcd.functional
K, ALPHA = 2, 1.1
WORKLOADS = [(64, 1024), (32, 4096), (1, 4096)]       # configs[2]'s batch, configs[1], the reference's operating point


def event_median(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.median([a.elapsed_time(b) for a, b in ev]))


def host_median(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for sor_bench.json")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sor_bench needs a CUDA device")
    res = {"card": card(), "k": K, "alpha": ALPHA, "reps": args.reps, "statistic": "median", "workloads": []}
    for B, N in WORKLOADS:
        pc = synth.face_clouds(B, N, seed=11)
        pc = (pc + 0.01 * torch.randn(pc.shape, generator=torch.Generator().manual_seed(12))).cuda()
        defense = pcd.defense.SORDefense(k=K, alpha=ALPHA, npoint=1024)
        np.random.seed(0)
        t_sor = event_median(lambda: F.sor(pc, K, ALPHA), args.reps, args.warmup)
        t_fwd = host_median(lambda: defense(pc), args.reps, args.warmup)
        t_ref = event_median(lambda: R.sor_statistic(pc, K, ALPHA), args.reps, args.warmup)
        r = F.sor(pc, K, ALPHA)
        mask, value, thr = R.sor_statistic(pc, K, ALPHA)
        t = thr[:, None]
        band = (value - t).abs() <= 1e-9 * t.abs()
        differ = r.keep != mask
        pairs = B * N * N
        row = {"B": B, "N": N, "pairs": pairs,
               "sor_ms": t_sor, "sor_pairs_per_s": pairs / (t_sor * 1e-3),
               "defense_forward_ms": t_fwd,
               "torch_f64_statistic_ms": t_ref, "torch_f64_pairs_per_s": pairs / (t_ref * 1e-3),
               "speedup_vs_torch_f64": t_ref / t_sor,
               "mask_points": B * N, "mask_differ": int(differ.sum()), "mask_differ_outside_band": int((differ & ~band).sum()),
               "points_inside_band": int(band.sum()), "removed_fraction": float(1 - r.keep.float().mean()),
               "max_value_rel_diff_vs_torch_f64": float(((r.value - value).abs() / value.abs().clamp_min(1e-300)).max())}
        print(json.dumps(row))
        res["workloads"].append(row)
        del mask, value, thr, r
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "sor_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("card", res["card"], "->", path)


if __name__ == "__main__":
    main()
