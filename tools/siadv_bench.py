"""SI-Adv timing: one SIAdvAttack iteration (victim forward + backward, the step kernel, estimate_normals) against the
PointNet-shaped victim, eager and as a CUDA graph; the step kernel alone against a torch formulation of the reference's
step; estimate_normals against a torch formulation (topk + batched torch.linalg.eigh).  The card name and power limit
are read in the same run; one JSON file.

    python tools/siadv_bench.py --out DIR [--reps 50] [--warmup 10] [--steps 20]

Kernel and normal times are medians of CUDA-event windows after warm-up; iteration times are the attack's own
event-timed loop over --steps iterations, median of three runs after one warm-up run.  The working sets stay in the
126 MB L2; it is not flushed.  The reference's own loop (open3d normals on the host, B = 1) is not timed: open3d is not
installed where this runs.
"""
import argparse
import importlib
import json
import math
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
from sor_bench import card, event_median  # noqa: E402
from victims import PointNetVictim  # noqa: E402

F = pcd.functional
N, STEP, EPS, K = 1024, 0.007, 0.16, 20
SCALE = math.sqrt(3 * 1024)


def torch_step(pc, ori, normal, grad):
    """the reference's step as torch ops: get_spin_axis_matrix, the transform (a batched matmul), the tangent gradient
    (a second one), the per-sample normalised step, the inverse transform and ClipPointsLinf on [B,N,3]"""
    x, y, z = normal.unbind(-1)
    zero = torch.zeros_like(z)
    den = torch.sqrt(1 - z * z)
    u = torch.stack([torch.stack([y / den, -x / den, zero], -1), torch.stack([x * z / den, y * z / den, -den], -1),
                     normal], -2)
    r = 1 / math.sqrt(2)
    ub = torch.stack([torch.stack([zero + r, zero - r, zero], -1), torch.stack([z / math.sqrt(2), z / math.sqrt(2), zero], -1),
                      torch.stack([zero, zero, z], -1)], -2)
    u = torch.where(((z * z - 1).abs() < 1e-4)[..., None, None], ub, u)
    t = (pc * normal).sum(-1, keepdim=True) * normal
    pp = (u @ (pc + t)[..., None])[..., 0]
    g = (u @ grad[..., None])[..., 0] * torch.tensor([1., 1., 0.], device=pc.device)
    norm = g.pow(2).sum((1, 2), keepdim=True).sqrt()
    pp = pp - STEP * SCALE * g / (norm + 1e-9)
    d = (u.transpose(-1, -2) @ pp[..., None])[..., 0] - t - ori
    s = torch.clamp(EPS / (d.pow(2).sum(1, keepdim=True).sqrt() + 1e-9), max=1)
    return ori + d * s


def torch_normals(pc):
    """k-NN by topk on the full distance matrix, the neighbourhood covariance, batched torch.linalg.eigh (one call per
    cloud: cuSOLVER's batched eigensolver rejects 32 x 1024 3 x 3 matrices in one call, CUSOLVER_STATUS_INVALID_VALUE)"""
    d = (pc * pc).sum(-1)[:, :, None] - 2 * pc @ pc.transpose(1, 2) + (pc * pc).sum(-1)[:, None, :]
    idx = d.topk(K, dim=-1, largest=False)[1]
    nb = torch.gather(pc[:, None].expand(-1, pc.shape[1], -1, -1), 2, idx[..., None].expand(-1, -1, -1, 3))
    cen = nb - nb.mean(2, keepdim=True)
    cov = cen.transpose(-1, -2) @ cen
    return torch.cat([torch.linalg.eigh(c)[1][..., 0] for c in cov.split(1)])


def inputs(B, seed):
    ori = synth.face_clouds(B, N, seed=seed).cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    pc = ori + 0.01 * torch.randn(ori.shape, generator=g, device="cuda")
    grad = torch.randn(ori.shape, generator=g, device="cuda")
    return pc, ori, F.estimate_normals(ori, K), grad


def kernel_rows(args):
    rows = []
    for B in (1, 32):
        pc, ori, normal, grad = inputs(B, 3)
        work = pc.clone()
        row = {"B": B, "N": N,
               "step_kernel_ms": event_median(lambda: F.shape_invariant_step_(work, ori, normal, grad, STEP, EPS), args.reps,
                                              args.warmup),
               "step_torch_ms": event_median(lambda: torch_step(pc, ori, normal, grad), args.reps, args.warmup),
               "normals_ms": event_median(lambda: F.estimate_normals(pc, K), args.reps, args.warmup),
               "normals_torch_ms": event_median(lambda: torch_normals(pc), args.reps, args.warmup)}
        ref = torch_step(pc, ori, normal, grad)
        work.copy_(pc)
        F.shape_invariant_step_(work, ori, normal, grad, STEP, EPS)
        row["step_max_abs_diff_vs_torch"] = float((work - ref).abs().max())
        cos = (F.estimate_normals(pc, K) * torch_normals(pc)).sum(-1).abs()
        row["normals_median_abs_cos_vs_torch"] = float(cos.median())
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
        row = {"B": B, "N": N, "victim": "PointNetVictim(40)", "iterations": args.steps}
        for use_graph in (False, True):
            atk = pcd.siadv.SIAdvAttack(victim, max_steps=args.steps, use_graph=use_graph)
            atk.attack(data, target)                 # warm-up: module loads, algorithm choices, the graph's pool
            t = []
            for _ in range(3):
                atk.attack(data, target)
                t.append(atk.loop_ms / args.steps)
            row["graph_iteration_ms" if use_graph else "eager_iteration_ms"] = float(np.median(t))
        print(json.dumps(row))
        rows.append(row)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for siadv_bench.json")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("siadv_bench needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"card": card(), "reps": args.reps, "statistic": "median", "kernels": kernel_rows(args),
           "iteration": attack_rows(args)}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "siadv_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("card", res["card"], "->", path)


if __name__ == "__main__":
    main()
