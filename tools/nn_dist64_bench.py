"""Float64 nearest-neighbour distance timing: functional.nn_dist64 against torch.cdist in float64 (the exact
'donot_use_mm_for_euclid_dist' mode) + min / argmin on the same GPU, and scipy's cdist per sample on the host cores.
Every arm's per-point minima are compared with the numpy brute force of the contract in the same run; the card name
and its power limit are read in the same run.  One JSON file is written.

    python tools/nn_dist64_bench.py --out DIR [--reps 20] [--warmup 3]

Workloads: B = 1, N = M = 4096 (the kernel splits the columns over CTAs); B = 32, N = M = 4096 (no split); 4000 vs
5000 points (the sizes of the reference's saved adversarial clouds); SOR-kept clouds, B = 32, N = 4096, against their
originals with per-sample lengths.  The inputs are a few MB and stay in the 126 MB L2; the sweep is bound by the FP64
pipe, not by memory, so the L2 is not flushed.  torch's CUDA kernel may contract into FMA, so its differences from the
brute force are reported, not failed; the kernel's are failed.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch
from scipy.spatial import distance

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
from oracle import nn_dist64_oracle as O  # noqa: E402

F = pcd.functional
CORES = len(os.sched_getaffinity(0))


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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q}


def workload(name, seed):
    g = torch.Generator().manual_seed(seed)
    if name == "sor_kept_B32_N4096":
        ori = synth.face_clouds(32, 4096, seed=seed)
        x = ori + 0.01 * torch.randn(ori.shape, generator=g)
        x[:, :80] = (torch.rand((32, 80, 3), generator=g) * 2 - 1) * 3
        s = F.sor(x.cuda(), 2, 1.1)
        kept = torch.gather(x.cuda(), 1, s.kept_idx.clamp_min(0)[..., None].expand(-1, -1, 3))
        return kept, ori.cuda(), s.lengths.to(torch.int32), None
    B, N, M = {"B1_4096x4096": (1, 4096, 4096), "B32_4096x4096": (32, 4096, 4096), "B8_4000x5000": (8, 4000, 5000)}[name]
    a = synth.face_clouds(B, N, seed=seed)
    b = synth.face_clouds(B, M, seed=seed) + 0.01 * torch.randn((B, M, 3), generator=g)
    return a.cuda(), b.cuda(), None, None


def samples(a, b, la, lb):
    B, N, M = a.shape[0], a.shape[1], b.shape[1]
    la = [N] * B if la is None else la.tolist()
    lb = [M] * B if lb is None else lb.tolist()
    return [(a[i, :la[i]], b[i, :lb[i]]) for i in range(B)]


def torch_arm(pairs):
    """float64 cdist without the matmul expansion, then min / argmin both ways: one batched call for equal sizes, else a
    loop over samples.  -> list of (a_min, a_arg, b_min, b_arg) tensors per sample (Euclidean minima)."""
    if all(p.shape == pairs[0][0].shape and q.shape == pairs[0][1].shape for p, q in pairs):
        a = torch.stack([p for p, _ in pairs]).double()
        b = torch.stack([q for _, q in pairs]).double()
        d = torch.cdist(a, b, compute_mode="donot_use_mm_for_euclid_dist")
        (am, aa), (bm, ba) = d.min(2), d.min(1)
        return [(am[i], aa[i], bm[i], ba[i]) for i in range(len(pairs))]
    out = []
    for p, q in pairs:
        d = torch.cdist(p.double()[None], q.double()[None], compute_mode="donot_use_mm_for_euclid_dist")[0]
        (am, aa), (bm, ba) = d.min(1), d.min(0)
        out.append((am, aa, bm, ba))
    return out


def scipy_one(pq):
    d = distance.cdist(pq[0], pq[1], "euclidean")
    return d.min(1), d.argmin(1), d.min(0), d.argmin(0)


def oracle_one(pq):
    am, aa = O.nearest64(pq[0], pq[1])
    bm, ba = O.nearest64(pq[1], pq[0])
    return am, aa, bm, ba


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for nn_dist64_bench.json")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("nn_dist64_bench needs a CUDA device")
    res = {"card": card(), "host_cores": CORES, "reps": args.reps, "statistic": "median", "workloads": []}
    print("card", res["card"], "host cores", CORES)
    failed = False
    pool = ThreadPoolExecutor(CORES)
    for wi, name in enumerate(["B1_4096x4096", "B32_4096x4096", "B8_4000x5000", "sor_kept_B32_N4096"]):
        a, b, la, lb = workload(name, seed=100 + wi)
        B, N, M = a.shape[0], a.shape[1], b.shape[1]
        t_kernel = event_median(lambda: F.nn_dist64(a, b, la, lb), args.reps, args.warmup)
        r = F.nn_dist64(a, b, la, lb)
        pairs = samples(a, b, la, lb)
        t_torch = event_median(lambda: torch_arm(pairs), max(3, args.reps // 4), 1)
        tp = [[t.cpu().numpy() for t in one] for one in torch_arm(pairs)]
        host = [(p.cpu().numpy().astype(np.float64), q.cpu().numpy().astype(np.float64)) for p, q in pairs]
        t0 = time.perf_counter()
        sp = list(pool.map(scipy_one, host))
        t_scipy = (time.perf_counter() - t0) * 1e3
        orc = list(pool.map(oracle_one, [(p.cpu().numpy(), q.cpu().numpy()) for p, q in pairs]))
        kernel_mismatch, torch_arg, scipy_arg = 0, 0, 0
        torch_diff, scipy_diff, pts = 0.0, 0.0, 0
        for i, (om, oa, obm, oba) in enumerate(orc):
            n, m = len(om), len(obm)
            km, ka = r.a_min[i, :n].cpu().numpy(), r.a_arg[i, :n].cpu().numpy()
            kbm, kba = r.b_min[i, :m].cpu().numpy(), r.b_arg[i, :m].cpu().numpy()
            kernel_mismatch += int((km != om).sum() + (ka != oa).sum() + (kbm != obm).sum() + (kba != oba).sum())
            for got, want in ((tp[i][0], om), (tp[i][2], obm)):
                torch_diff = max(torch_diff, float(np.abs(got - np.sqrt(want)).max()))
            torch_arg += int((tp[i][1] != oa).sum() + (tp[i][3] != oba).sum())
            for got, want in ((sp[i][0], om), (sp[i][2], obm)):
                scipy_diff = max(scipy_diff, float(np.abs(got - np.sqrt(want)).max()))
            scipy_arg += int((sp[i][1] != oa).sum() + (sp[i][3] != oba).sum())
            pts += n + m
        pairs_total = sum(2 * len(p) * len(q) for p, q in pairs)       # both directions are swept
        row = {"workload": name, "B": B, "N": N, "M": M, "pairs_swept": pairs_total, "points": pts,
               "kernel_ms": t_kernel, "kernel_pairs_per_s": pairs_total / (t_kernel * 1e-3),
               "torch_cdist_f64_ms": t_torch, "speedup_vs_torch": t_torch / t_kernel,
               "scipy_host_ms": t_scipy, "scipy_threads": CORES,
               "kernel_per_point_mismatches": kernel_mismatch,
               "torch_max_abs_diff_euclid": torch_diff, "torch_arg_mismatches": torch_arg,
               "scipy_max_abs_diff_euclid": scipy_diff, "scipy_arg_mismatches": scipy_arg}
        print(json.dumps(row), flush=True)
        res["workloads"].append(row)
        failed |= kernel_mismatch != 0
        del r, tp
        torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "nn_dist64_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("->", path)
    if failed:
        raise SystemExit("the kernel's per-point minima differ from the brute force")


if __name__ == "__main__":
    main()
