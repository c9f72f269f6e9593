"""Reference for SOR on ragged batches (functional.sor with lengths, pcd_sor_forward_len in include/pcdist.h): the
float64 brute force oracle.sor_oracle.sor64 on every truncated sample, with the padding the contract fixes."""
import numpy as np

from oracle.sor_oracle import SOR64, sor64


def sor64_ragged(pc, lengths, k=2, alpha=1.1):
    """pc [B,N,3] float32, lengths [B] integers (clamped to [0, N]) -> SOR64(value [B,N], threshold [B], keep [B,N]).
    Sample b is pc[b, :n]: sor64 when n >= k + 1, else no statistic (NaN values and threshold, nothing kept).  Rows
    past n get value NaN and keep False."""
    pc = np.asarray(pc, np.float32)
    B, N, _ = pc.shape
    value = np.full((B, N), np.nan)
    threshold = np.full(B, np.nan)
    keep = np.zeros((B, N), bool)
    for b in range(B):
        n = int(min(max(int(lengths[b]), 0), N))
        if n < k + 1:
            continue
        o = sor64(pc[b:b + 1, :n], k, alpha)
        value[b, :n], threshold[b], keep[b, :n] = o.value[0], o.threshold[0], o.keep[0]
    return SOR64(value, threshold, keep)
