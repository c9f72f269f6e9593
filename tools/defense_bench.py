"""Drop-points defence timing: SORDefense.forward with numpy draws against device draws (functional.PointSampler),
functional.sor alone and the sampler kernel alone; SRS in both modes; and one CWAttack iteration through a defended
PointNet-shaped victim, eager and captured.  The card name and power limit are read in the same run; one JSON file.

    python tools/defense_bench.py --out DIR [--reps 30] [--warmup 5]

Times are medians after warm-up.  Calls that synchronise with the host (the numpy forwards) are timed with a host clock
around the call and a device synchronise; the device-only paths with CUDA events, and also with the host clock, so the
two modes compare on the same footing.  The working sets stay in the 126 MB L2; it is not flushed.
"""
import argparse
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
from sor_bench import card, event_median, host_median  # noqa: E402
from victims import PointNetVictim  # noqa: E402

F, D, CL = pcd.functional, pcd.defense, pcd.cw_loop
K, ALPHA, NPOINT = 2, 1.1, 1024
SOR_WORKLOADS = [(64, 1024), (32, 4096), (1, 4096), (1, 10000)]


def cloud(B, N, seed):
    pc = synth.face_clouds(B, N, seed=seed)
    return (pc + 0.01 * torch.randn(pc.shape, generator=torch.Generator().manual_seed(seed + 1))).cuda()


def sor_rows(args):
    rows = []
    for B, N in SOR_WORKLOADS:
        x = cloud(B, N, 11)
        numpy_def = D.SORDefense(K, ALPHA, NPOINT)
        sampler = F.PointSampler(0)
        device_def = D.SORDefense(K, ALPHA, NPOINT, sampler=sampler)
        np.random.seed(0)
        r = F.sor(x, K, ALPHA)
        kept32 = r.kept_idx.int()
        kept_n = r.lengths.int()
        row = {"B": B, "N": N, "npoint": NPOINT, "kept_min": int(r.lengths.min()), "kept_max": int(r.lengths.max()),
               "numpy_forward_ms": host_median(lambda: numpy_def(x), args.reps, args.warmup),
               "device_forward_ms": host_median(lambda: device_def(x), args.reps, args.warmup),
               "device_forward_event_ms": event_median(lambda: device_def(x), args.reps, args.warmup),
               "sor_ms": event_median(lambda: F.sor(x, K, ALPHA), args.reps, args.warmup),
               "sampler_ms": event_median(lambda: F.sample_points(kept_n, N, NPOINT, sampler, table=kept32), args.reps,
                                          args.warmup)}
        row["device_speedup_vs_numpy"] = row["numpy_forward_ms"] / row["device_forward_ms"]
        print(json.dumps(row))
        rows.append(row)
    return rows


def srs_row(args):
    B, N, drop = 64, 1024, 500
    x = cloud(B, N, 13)
    numpy_def, device_def = D.SRSDefense(drop), D.SRSDefense(drop, sampler=F.PointSampler(1))
    np.random.seed(0)
    row = {"B": B, "N": N, "drop_num": drop,
           "numpy_forward_ms": host_median(lambda: numpy_def(x), args.reps, args.warmup),
           "device_forward_ms": host_median(lambda: device_def(x), args.reps, args.warmup),
           "device_forward_event_ms": event_median(lambda: device_def(x), args.reps, args.warmup)}
    print(json.dumps(row))
    return row


def attack_row(args):
    """one defended CWAttack iteration: B = 32, N = 4096 clouds, SOR to 1024 points, the PointNet-shaped victim"""
    B, N = 32, 4096
    torch.manual_seed(0)
    victim = PointNetVictim(num_classes=40).cuda().eval()
    data = cloud(B, N, 17)
    target = torch.arange(B, device="cuda") % 40
    iters = max(args.reps, 10)
    row = {"B": B, "N": N, "npoint": NPOINT, "victim": "PointNetVictim(40)", "iterations": iters}
    for use_graph in (False, True):
        model = D.DefendedVictim(victim, D.SORDefense(K, ALPHA, NPOINT, sampler=F.PointSampler(2)))
        atk = CL.CWAttack(model, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.ChamferDist(method="adv2ori"),
                          attack_lr=1e-2, binary_step=1, num_iter=iters, clip_func=CL.ClipPointsLinf(0.1),
                          use_graph=use_graph)
        atk.attack(data, target)                     # warm-up: module loads, algorithm choices, the graph's pool
        t = []
        for _ in range(3):
            atk.attack(data, target)
            t.append(atk.loop_ms / iters)
        row["graph_iteration_ms" if use_graph else "eager_iteration_ms"] = float(np.median(t))
    print(json.dumps(row))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for defense_bench.json")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("defense_bench needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"card": card(), "k": K, "alpha": ALPHA, "reps": args.reps, "statistic": "median"}
    res["sor"] = sor_rows(args)
    res["srs"] = srs_row(args)
    res["defended_cw_iteration"] = attack_row(args)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "defense_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("card", res["card"], "->", path)


if __name__ == "__main__":
    main()
