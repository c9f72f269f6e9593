"""Reference for the float64 nearest-neighbour distances -- TEST / BENCH INFRASTRUCTURE ONLY (tests/,
__graft_entry__.smoke(), tools/nn_dist64_bench.py; the product never imports it).

nn_dist64: numpy float64 brute force of the pcd_nn_dist64_forward contract (include/pcdist.h), row-blocked, with the
contract's per-pair operation order, so the per-point minima and arg-minima are bit-exact.  Lengths, NaN and the
per-sample reductions follow numpy (np.mean's pairwise summation differs from the kernel's order in the last bits).
"""
from collections import namedtuple

import numpy as np

NNDist64 = namedtuple("NNDist64", "a_min a_arg b_min b_arg a_mean_sq a_mean a_max_sq a_max a_argmax "
                                  "b_mean_sq b_mean b_max_sq b_max b_argmax")


def pair_s64(p, q):
    """s[i,j] = ((dx*dx) + (dy*dy)) + (dz*dz) with dx = q_x[j] - p_x[i], in float64: p [n,3], q [m,3] -> [n,m]."""
    p = np.asarray(p, np.float32).astype(np.float64)
    q = np.asarray(q, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        d = [q[None, :, c] - p[:, None, c] for c in range(3)]
        return (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]


def nearest64(p, q, row_block=1024):
    """min / argmin over the columns of pair_s64(p, q), block by block: ([n] float64, [n] int64).  No column: NaN, -1."""
    n = len(p)
    vmin, varg = np.full(n, np.nan), np.full(n, -1, np.int64)
    if len(q):
        for r0 in range(0, n, row_block):
            s = pair_s64(p[r0:r0 + row_block], q)
            vmin[r0:r0 + row_block] = s.min(1)
            varg[r0:r0 + row_block] = s.argmin(1)
    return vmin, varg


def reduce64(v):
    """numpy's mean of v, mean of sqrt(v), max of v, sqrt of it and argmax of v; an empty v gives NaN and -1."""
    if len(v) == 0:
        return np.nan, np.nan, np.nan, np.nan, -1
    with np.errstate(invalid="ignore"):
        mx = v.max()
        return v.mean(), np.sqrt(v).mean(), mx, np.sqrt(mx), int(v.argmax())


def nn_dist64(a, b, a_lengths=None, b_lengths=None, row_block=1024):
    """a [B,N,3], b [B,M,3] float32; lengths None or [B] integers (clamped to [0, N] / [0, M]) -> NNDist64 of numpy
    arrays: per point [B,N] / [B,M] (NaN / -1 past the length), per sample [B]."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    B, N, _ = a.shape
    M = b.shape[1]
    la = np.full(B, N) if a_lengths is None else np.clip(np.asarray(a_lengths, np.int64), 0, N)
    lb = np.full(B, M) if b_lengths is None else np.clip(np.asarray(b_lengths, np.int64), 0, M)
    a_min, a_arg = np.full((B, N), np.nan), np.full((B, N), -1, np.int64)
    b_min, b_arg = np.full((B, M), np.nan), np.full((B, M), -1, np.int64)
    stats, amax = np.empty((2, B, 4)), np.empty((2, B), np.int64)
    for i in range(B):
        n, m = la[i], lb[i]
        a_min[i, :n], a_arg[i, :n] = nearest64(a[i, :n], b[i, :m], row_block)
        b_min[i, :m], b_arg[i, :m] = nearest64(b[i, :m], a[i, :n], row_block)
        for d, v in enumerate((a_min[i, :n], b_min[i, :m])):
            r = reduce64(v)
            stats[d, i], amax[d, i] = r[:4], r[4]
    return NNDist64(a_min, a_arg, b_min, b_arg, *stats[0].T, amax[0], *stats[1].T, amax[1])
