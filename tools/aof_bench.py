"""AOF timing: one AOFAttack iteration against the PointNet-shaped victim, eager and as a CUDA graph; the low-frequency
projection (functional.low_pass) forward + backward against the torch bmm chain, and its forward launch alone with the
bytes it must read and write; the basis (Laplacian + float64 eigh) against float32 eigh; the reference-shaped host loop
at B = 1.  N = 1024, low_pass = 100, B in {1, 32}.  The card name and power limit are read in the same run; one JSON file.

    python tools/aof_bench.py --out DIR [--reps 50] [--warmup 10] [--steps 20]

Kernel times are medians of CUDA-event windows around the replay of a CUDA graph of 20 calls, divided by 20 (one eager
call at these sizes measures the host's enqueue); the eager-call figures are single calls between events.  The working
sets (at most 13 MB of basis) stay in the 126 MB L2, which is not flushed, so the bandwidth share is against HBM's
7.7 TB/s but the bytes come from L2.  Iteration
times are the attack's own event-timed loop over --steps iterations, median of three runs after one warm-up run; the host
loop is timed by the host clock around --steps iterations ending in a device synchronise.  Basis times are medians of
three runs after one warm-up.
"""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
from oracle import aof_oracle  # noqa: E402
from sor_bench import card, event_median  # noqa: E402
from victims import PointNetVictim  # noqa: E402

F, CL = pcd.functional, pcd.cw_loop
N, KL = 1024, 100
HBM_BYTES_PER_S = 7.7e12


def torch_low(x, V):
    """V^T (V x) as the two bmm's of a torch formulation"""
    return torch.bmm(V.transpose(1, 2), torch.bmm(V, x))


def graph_ms(fn, reps, warmup, calls=20):
    """device time of one fn() call: `calls` calls captured into one CUDA graph, its replay timed by events (a single
    eager call at these sizes is bound by the host's enqueue, not the device)"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(calls):
            fn()
    return event_median(g.replay, reps, warmup) / calls


def kernel_rows(args):
    rows = []
    for B in (1, 32):
        ori = synth.face_clouds(B, N, seed=3).cuda()
        V = pcd.taof.low_frequency_basis(ori.transpose(1, 2), KL)
        x = ori.clone().requires_grad_(True)
        g = torch.randn_like(ori)

        def ours():
            torch.autograd.grad(F.low_pass(x, V), x, g)

        def theirs():
            torch.autograd.grad(torch_low(x, V), x, g)

        fwd_ms = graph_ms(lambda: F.low_pass(ori, V), args.reps, args.warmup)
        nbytes = 2 * V.numel() * 4 + 2 * ori.numel() * 4        # V read in both phases, x read, y written
        row = {"B": B, "N": N, "low_pass": KL,
               "fwd_bwd_kernel_ms": graph_ms(ours, args.reps, args.warmup),
               "fwd_bwd_torch_bmm_ms": graph_ms(theirs, args.reps, args.warmup),
               "fwd_bwd_kernel_eager_call_ms": event_median(ours, args.reps, args.warmup),
               "fwd_bwd_torch_bmm_eager_call_ms": event_median(theirs, args.reps, args.warmup),
               "fwd_kernel_ms": fwd_ms, "fwd_torch_bmm_ms": graph_ms(lambda: torch_low(ori, V), args.reps, args.warmup),
               "fwd_bytes": nbytes,
               "fwd_share_of_hbm_bandwidth": nbytes / (fwd_ms * 1e-3) / HBM_BYTES_PER_S,
               "fwd_max_abs_diff_vs_torch": float((F.low_pass(ori, V) - torch_low(ori, V)).abs().max())}
        print(json.dumps(row))
        rows.append(row)
    return rows


def timed(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t))


def basis_rows():
    rows = []
    for B in (1, 32):
        pc = synth.face_clouds(B, N, seed=5).cuda().transpose(1, 2)
        row = {"B": B, "N": N, "low_pass": KL,
               "laplacian_ms": timed(lambda: pcd.taof.laplacian_from_pc(pc, 30)),
               "basis_float64_eigh_ms": timed(lambda: pcd.taof.low_frequency_basis(pc, KL)),
               "basis_float32_eigh_ms": timed(lambda: torch.linalg.eigh(pcd.taof.laplacian_from_pc(pc, 30)))}
        V64 = pcd.taof.low_frequency_basis(pc, KL).double()
        V32 = torch.linalg.eigh(pcd.taof.laplacian_from_pc(pc, 30))[1][..., :KL].transpose(1, 2).double()
        eye = torch.eye(KL, dtype=torch.float64, device="cuda")
        row["orthonormality_err_float64_eigh"] = float((V64 @ V64.transpose(1, 2) - eye).abs().max())
        row["orthonormality_err_float32_eigh"] = float((V32 @ V32.transpose(1, 2) - eye).abs().max())
        print(json.dumps(row))
        rows.append(row)
    return rows


def attack_rows(args):
    torch.manual_seed(0)
    victim = PointNetVictim(num_classes=40).cuda().eval()
    rows = []
    for B in (1, 32):
        data = synth.face_clouds(B, N, seed=17).cuda()
        target = torch.arange(B, device="cuda") % 40
        basis = pcd.taof.low_frequency_basis(data.transpose(1, 2), KL)
        row = {"B": B, "N": N, "low_pass": KL, "victim": "PointNetVictim(40)", "iterations": args.steps}
        for use_graph in (False, True):
            atk = pcd.taof.AOFAttack(victim, CL.UntargetedLogitsAdvLoss(kappa=0.), pcd.dist_utils.L2Dist(), low_pass=KL,
                                     binary_step=1, num_iter=args.steps, clip_func=CL.ClipPointsLinf(0.18),
                                     use_graph=use_graph)
            atk.attack(data, target, basis=basis)          # warm-up: module loads, algorithm choices, the graph's pool
            t = []
            for _ in range(3):
                atk.attack(data, target, basis=basis)
                t.append(atk.loop_ms / args.steps)
            row["graph_iteration_ms" if use_graph else "eager_iteration_ms"] = float(np.median(t))
        if B == 1:
            noise = torch.randn((1, 1, 3, N))
            host = timed(lambda: aof_oracle.host_loop(victim, F.low_pass, data, target, basis,
                                                      CL.UntargetedLogitsAdvLoss(kappa=0.), pcd.dist_utils.L2Dist(), 0.25,
                                                      noise, binary_step=1, num_iter=args.steps,
                                                      clip_func=CL.ClipPointsLinf(0.18)))
            row["host_loop_iteration_ms"] = host / args.steps
        print(json.dumps(row))
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for aof_bench.json")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("aof_bench needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"card": card(), "reps": args.reps, "statistic": "median", "kernels": kernel_rows(args), "basis": basis_rows(),
           "iteration": attack_rows(args)}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "aof_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("card", res["card"], "->", path)


if __name__ == "__main__":
    main()
