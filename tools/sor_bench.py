"""SOR defence timing: functional.sor and SORDefense.forward against the reference's torch float64 formulation on the
same GPU, with the mask agreement of the same run, the card name and its power limit, written as one JSON file.
functional.sor runs pcd_sor_forward_len; the fixed-size entry pcd_sor_forward is timed next to it, and at B = 1 the
new entry also with its columns unsplit (col_split = 1).  A ragged batch (lengths drawn in [N/2, N]) is timed against
the torch formulation looped over its truncated samples, which is what the reference would have to do.

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
# configs[2]'s batch, configs[1], the reference's operating point (B = 1) at three sizes up to a raw face scan
WORKLOADS = [(64, 1024), (32, 4096), (1, 1024), (1, 4096), (1, 10000)]
RAGGED = (32, 4096)


def fixed_size_entry(pc):
    """pcd_sor_forward (two launches, one N for the batch) with outputs allocated once"""
    lib = pcd._lib.load()
    B, N, _ = pc.shape
    out = [torch.empty((B, N), dtype=torch.float64, device="cuda"), torch.empty((B,), dtype=torch.float64, device="cuda"),
           torch.empty((B, N), dtype=torch.uint8, device="cuda"), torch.empty((B, N), dtype=torch.int32, device="cuda"),
           torch.empty((B,), dtype=torch.int32, device="cuda")]

    def run():
        st = lib.pcd_sor_forward(pc.data_ptr(), pc.stride(0), pc.stride(1), pc.stride(2), B, N, K, ALPHA,
                                 *[t.data_ptr() for t in out], torch.cuda.current_stream().cuda_stream)
        pcd._lib.check(st, "pcd_sor_forward")
    return run, out


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
        old, old_out = fixed_size_entry(pc)
        t_old = event_median(old, args.reps, args.warmup)
        t_unsplit = event_median(lambda: F.sor(pc, K, ALPHA, col_split=1), args.reps, args.warmup) if B == 1 else None
        r = F.sor(pc, K, ALPHA)
        assert torch.equal(r.value, old_out[0]) and torch.equal(r.keep, old_out[2].bool())
        mask, value, thr = R.sor_statistic(pc, K, ALPHA)
        t = thr[:, None]
        band = (value - t).abs() <= 1e-9 * t.abs()
        differ = r.keep != mask
        pairs = B * N * N
        row = {"B": B, "N": N, "pairs": pairs,
               "sor_ms": t_sor, "sor_pairs_per_s": pairs / (t_sor * 1e-3),
               "defense_forward_ms": t_fwd, "fixed_size_entry_ms": t_old, "unsplit_ms": t_unsplit,
               "col_split": (pcd._lib.load().pcd_sor_workspace_bytes(B, N, K, 0) // (B * (K + 1) * N * 8)) or 1,
               "torch_f64_statistic_ms": t_ref, "torch_f64_pairs_per_s": pairs / (t_ref * 1e-3),
               "speedup_vs_torch_f64": t_ref / t_sor,
               "mask_points": B * N, "mask_differ": int(differ.sum()), "mask_differ_outside_band": int((differ & ~band).sum()),
               "points_inside_band": int(band.sum()), "removed_fraction": float(1 - r.keep.float().mean()),
               "max_value_rel_diff_vs_torch_f64": float(((r.value - value).abs() / value.abs().clamp_min(1e-300)).max())}
        print(json.dumps(row))
        res["workloads"].append(row)
        del mask, value, thr, r
        torch.cuda.empty_cache()
    res["ragged"] = ragged(args)
    print(json.dumps(res["ragged"]))
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "sor_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("card", res["card"], "->", path)


def ragged(args):
    B, N = RAGGED
    pc = synth.face_clouds(B, N, seed=13)
    pc = (pc + 0.01 * torch.randn(pc.shape, generator=torch.Generator().manual_seed(14))).cuda()
    lengths = torch.randint(N // 2, N + 1, (B,), generator=torch.Generator().manual_seed(15))
    lens_host = lengths.tolist()
    lengths = lengths.cuda()
    t_sor = event_median(lambda: F.sor(pc, K, ALPHA, lengths=lengths), args.reps, args.warmup)
    t_loop = event_median(lambda: [F.sor(pc[b:b + 1, :n], K, ALPHA) for b, n in enumerate(lens_host)], args.reps,
                          args.warmup)
    t_ref = event_median(lambda: [R.sor_statistic(pc[b:b + 1, :n], K, ALPHA) for b, n in enumerate(lens_host)],
                         args.reps, args.warmup)
    r = F.sor(pc, K, ALPHA, lengths=lengths)
    differ = outside_band_differ = 0
    for b, n in enumerate(lens_host):
        mask, value, thr = R.sor_statistic(pc[b:b + 1, :n], K, ALPHA)
        d = r.keep[b, :n] != mask[0]
        differ += int(d.sum())
        outside_band_differ += int((d & ((value[0] - thr[0]).abs() > 1e-9 * thr[0].abs())).sum())
    pairs = sum(n * n for n in lens_host)
    return {"B": B, "N": N, "lengths_min": min(lens_host), "lengths_max": max(lens_host), "pairs": pairs,
            "sor_ms": t_sor, "sor_pairs_per_s": pairs / (t_sor * 1e-3),
            "per_sample_loop_of_sor_ms": t_loop,
            "torch_f64_statistic_loop_ms": t_ref, "speedup_vs_torch_f64_loop": t_ref / t_sor,
            "mask_points": sum(lens_host), "mask_differ": differ, "mask_differ_outside_band": outside_band_differ}


if __name__ == "__main__":
    main()
