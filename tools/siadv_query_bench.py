"""SI-Adv query-based attack timing: SIAdvQueryAttack against the PointNet-shaped victim at N = 1024, B = 1 and 32, eager
and as a CUDA graph; the round kernel alone; the reference's shape (oracle/siadv_query_oracle.host_loop: B = 1, the
logits copied to the host and one Python decision per query) on the same GPU as the comparison arm, and whether its
outputs are the device loop's bits at B = 1.  The card name and power limit are read in the same run; one JSON file.

    python tools/siadv_query_bench.py --out DIR [--rounds 200] [--reps 50] [--warmup 10]

The attack runs --rounds query rounds with no early stop (check_every = rounds; the attack is untargeted against the
victim's own label, and a sample that succeeds early stays frozen while the others go on).  Loop times are the attack's
own CUDA-event window over those rounds, median of three runs after one warm-up run; the round kernel's time is the
median of CUDA-event windows after warm-up.  The working sets stay in the 126 MB L2; it is not flushed.
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
from oracle import siadv_query_oracle as Q  # noqa: E402
from sor_bench import card, event_median  # noqa: E402
from victims import PointNetVictim  # noqa: E402

F = pcd.functional
N, EPS, STEP = 1024, 0.16, 0.05


def data_for(victim, B):
    x = synth.face_clouds(B, N, seed=17).cuda()
    with torch.no_grad():
        label = victim(x.transpose(1, 2))[0].argmax(1)
    return x, label


def loop_row(victim, B, args):
    x, label = data_for(victim, B)
    row = {"B": B, "N": N, "victim": "PointNetVictim(40)", "rounds": args.rounds}
    for use_graph in (False, True):
        atk = pcd.siadv.SIAdvQueryAttack(victim, eps=EPS, step_size=STEP, max_query=args.rounds,
                                         check_every=args.rounds, use_graph=use_graph)
        atk.attack(x, label)                     # warm-up: module loads, algorithm choices, the graph's pool
        t, q = [], []
        for _ in range(3):
            _, _, success, queries = atk.attack(x, label)
            t.append(atk.loop_ms)
            q.append(int(queries.sum()))
        ms = float(np.median(t))
        key = "graph" if use_graph else "eager"
        row[key + "_round_ms"] = ms / atk.rounds
        row[key + "_rounds_per_s"] = atk.rounds / (ms * 1e-3)
        row[key + "_sample_queries_per_s"] = float(np.median(q)) / (ms * 1e-3)
        row["successes"] = int(success.sum())
    # the round kernel alone, on a state that stays active
    normal = F.estimate_normals(x, 20)
    order, dir = F.si_sensitivity(torch.randn_like(x), normal)
    with torch.no_grad():
        logits = victim(x.transpose(1, 2))[0]
    cloud, trial = x.clone(), x.clone()
    state = torch.tensor([[-1, 0, 0, 0]], dtype=torch.int32, device="cuda").repeat(B, 1)
    best = torch.zeros(B, device="cuda")
    row["round_kernel_ms"] = event_median(
        lambda: F.si_query_round_(logits, label, x, normal, order, dir, cloud, trial, state, best, STEP, EPS, 2 ** 30),
        args.reps, args.warmup)
    print(json.dumps(row))
    return row


def host_row(victim, args):
    """the reference's shape at B = 1, and the device loop on the same sample"""
    x, label = data_for(victim, 1)
    points = torch.cat([x, F.estimate_normals(x, 20)], -1)
    normal = pcd.siadv._unit_normals(points, 20)                               # the attack's normals of these points
    Q.host_loop(victim, x[0], normal[0], int(label[0]), EPS, STEP, 5)           # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h_adv, h_pred, h_success, h_queries = Q.host_loop(victim, x[0], normal[0], int(label[0]), EPS, STEP, args.rounds)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    atk = pcd.siadv.SIAdvQueryAttack(victim, eps=EPS, step_size=STEP, max_query=args.rounds, check_every=args.rounds)
    adv, pred, success, queries = atk.attack(points, label)
    row = {"B": 1, "N": N, "queries": h_queries, "host_loop_ms": ms, "host_loop_query_ms": ms / h_queries,
           "host_loop_queries_per_s": h_queries / (ms * 1e-3),
           "same_bits_as_device_loop": bool(torch.equal(adv[0], h_adv) and int(queries[0]) == h_queries
                                             and bool(success[0]) == h_success and int(pred[0]) == h_pred)}
    print(json.dumps(row))
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for siadv_query_bench.json")
    ap.add_argument("--rounds", type=int, default=200)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("siadv_query_bench needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(0)
    victim = PointNetVictim(num_classes=40).cuda().eval()
    res = {"card": card(), "statistic": "median", "loop": [loop_row(victim, B, args) for B in (1, 32)],
           "host_loop": host_row(victim, args)}
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "siadv_query_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("card", res["card"], "->", path)


if __name__ == "__main__":
    main()
