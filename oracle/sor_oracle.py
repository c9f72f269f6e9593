"""References for the SOR defence -- TEST / BENCH INFRASTRUCTURE ONLY (tests/, __graft_entry__.smoke(),
tools/sor_bench.py; the product never imports it).

* sor64 / sor64_threshold: numpy float64 brute force of the pcd_sor_forward contract (include/pcdist.h).
* sor_statistic / sor_outlier_removal: the reference's torch formulation of
  attack/SIadv/baselines/defense/drop_points/SOR.py:24-54 (outlier_removal) as SURVEY §8 a5 records it -- the
  KNNDist statistic in float64, used as a keep-mask; runs on the CPU or the GPU.
* sor_process_data: SORDefense.process_data of IF-Defense's SOR.py (SIadv's baselines/ tree), its per-sample
  resampling loop literally, on numpy arrays.
"""
from collections import namedtuple

import numpy as np
import torch

SOR64 = namedtuple("SOR64", "value threshold keep")


def sor64(pc, k=2, alpha=1.1, row_block=512):
    """pc [B,N,3] float32 -> (value [B,N], threshold [B], keep [B,N] bool).  Same per-pair operation order as the
    contract, so `value` is bit-exact; mean / std use numpy's summation order (the kernel's differs in the last bits)."""
    pc = np.asarray(pc, np.float32).astype(np.float64)
    B, N, _ = pc.shape
    value = np.empty((B, N), np.float64)
    for b in range(B):
        x, y, z = pc[b, :, 0], pc[b, :, 1], pc[b, :, 2]
        xx = (x * x + y * y) + z * z
        for r0 in range(0, N, row_block):
            r = slice(r0, min(r0 + row_block, N))
            dot = (x[r, None] * x[None, :] + y[r, None] * y[None, :]) + z[r, None] * z[None, :]
            with np.errstate(invalid="ignore", over="ignore"):
                d = (xx[None, :] + (-2.0 * dot)) + xx[r, None]
            s = np.sort(np.partition(d, k, axis=1)[:, :k + 1], axis=1)
            acc = s[:, 1].copy()
            for m in range(2, k + 1):
                acc = acc + s[:, m]
            value[b, r] = acc / k
    return SOR64(value, *sor64_threshold(value, alpha))


def sor64_threshold(value, alpha):
    """value [B,N] -> (threshold = mean + alpha * unbiased std [B], keep = value <= threshold [B,N])."""
    threshold = value.mean(1) + alpha * value.std(1, ddof=1)
    return threshold, value <= threshold[:, None]


def sor_statistic(x, k=2, alpha=1.1):
    """SOR.py's outlier_removal up to its keep-mask.  x [B,K,3] on any device -> (bool_mask [B,K],
    value [B,K] float64, threshold [B] float64)."""
    pc = x.clone().detach().double()
    pc = pc.transpose(2, 1)  # [B, 3, K]
    inner = -2. * torch.matmul(pc.transpose(2, 1), pc)  # [B, K, K]
    xx = torch.sum(pc ** 2, dim=1, keepdim=True)  # [B, 1, K]
    dist = xx + inner + xx.transpose(2, 1)  # [B, K, K]
    # the min is self so we take top (k + 1)
    neg_value, _ = (-dist).topk(k=k + 1, dim=-1)
    value = -(neg_value[..., 1:])  # [B, K, k]
    value = torch.mean(value, dim=-1)  # [B, K]
    mean = torch.mean(value, dim=-1)  # [B]
    std = torch.std(value, dim=-1)  # [B]
    threshold = mean + alpha * std  # [B]
    bool_mask = (value <= threshold[:, None])  # [B, K]
    return bool_mask, value, threshold


def sor_outlier_removal(x, k=2, alpha=1.1):
    """SOR.py's outlier_removal: sor_statistic, then the list of kept clouds -> (sel_pc list of [K_i,3], bool_mask,
    value, threshold)."""
    bool_mask, value, threshold = sor_statistic(x, k, alpha)
    sel_pc = [x[i][bool_mask[i]] for i in range(x.shape[0])]
    return sel_pc, bool_mask, value, threshold


def sor_process_data(pcs, npoint):
    """pcs: list of [N_i,3] arrays -> [B,npoint,3]: sample npoint of N_i > npoint points, or repeat the cloud and
    sample the remainder, drawing from numpy's global generator in the reference's order."""
    out = []
    for one_pc in pcs:
        N = len(one_pc)
        if N > npoint:
            idx = np.random.choice(N, npoint, replace=False)
            one_pc = one_pc[idx]
        elif N < npoint:
            duplicated_pc = one_pc
            num = npoint // N - 1
            for _ in range(num):
                duplicated_pc = np.concatenate([duplicated_pc, one_pc], axis=0)
            num = npoint - len(duplicated_pc)
            idx = np.random.choice(N, num, replace=False)
            one_pc = np.concatenate([duplicated_pc, one_pc[idx]], axis=0)
        out.append(one_pc)
    return np.stack(out)
