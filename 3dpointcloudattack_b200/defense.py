"""SOR (statistical outlier removal) defence <- attack/SIadv/baselines/defense/drop_points/SOR.py.

SIadv's baselines/ tree comes from IF-Defense; the defaults k = 2, alpha = 1.1, npoint = 1024 are IF-Defense's
published values.  The statistic runs in the float64 kernels behind functional.sor; the resampling to npoint points
keeps the reference's numpy draws, so a seeded np.random gives the same clouds.  There is no install() patch for
this module: the class layout of SOR.py is not recorded here.
"""
import numpy as np
import torch
from torch import nn

from . import functional as F

__all__ = ["SORDefense", "draw_indices"]


def draw_indices(sizes, npoint):
    """The resampling draws of SORDefense.process_data, in the reference's order, from numpy's global generator.
    sizes: number of kept points of each sample -> [B, npoint] int64 indices into each sample's kept points:
      N_i > npoint   np.random.choice(N_i, npoint, replace=False)
      N_i < npoint   the whole cloud npoint // N_i times, then np.random.choice(N_i, npoint % N_i, replace=False)
                     (drawn even when that size is 0: the call still advances the generator)
      N_i == npoint  the cloud as is."""
    out = np.empty((len(sizes), npoint), np.int64)
    for b, n in enumerate(sizes):
        n = int(n)
        if n == 0:
            raise ValueError(f"sample {b} has no point left after outlier removal")
        if n > npoint:
            out[b] = np.random.choice(n, npoint, replace=False)
        elif n < npoint:
            reps = npoint // n
            out[b, :reps * n] = np.tile(np.arange(n), reps)
            out[b, reps * n:] = np.random.choice(n, npoint % n, replace=False)
        else:
            out[b] = np.arange(n)
    return out


class SORDefense(nn.Module):
    """Statistical outlier removal: drop the points whose mean squared distance to their k nearest neighbours exceeds
    mean + alpha * std over the cloud, then resample every cloud to npoint points."""

    def __init__(self, k=2, alpha=1.1, npoint=1024):
        super().__init__()
        self.k = k
        self.alpha = alpha
        self.npoint = npoint

    def outlier_removal(self, x, lengths=None):
        """x [B,N,3] -> [x[b][keep[b]] for b], differentiable with respect to x (the mask is a constant).
        lengths: None or an integer tensor [B]; sample b is then x[b, :lengths[b]] (see functional.sor).
        One device-to-host copy: the kept counts."""
        r = F.sor(x, self.k, self.alpha, lengths)
        lengths = r.lengths.cpu().tolist()
        return [x[b].index_select(0, r.kept_idx[b, :n]) for b, n in enumerate(lengths)]

    def process_data(self, pc, npoint=None):
        """pc: list of [N_i,3] kept clouds -> [B, npoint, 3], resampled by draw_indices and built with one gather."""
        npoint = self.npoint if npoint is None else int(npoint)
        sizes = [int(p.shape[0]) for p in pc]
        idx = draw_indices(sizes, npoint)
        offsets = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
        flat = torch.cat(list(pc), 0)
        return flat[torch.from_numpy(idx + offsets[:, None]).to(flat.device)]

    @torch.no_grad()
    def forward(self, x, lengths=None):
        """process_data(outlier_removal(x, lengths)) without building the list: the draws index the kept-index table,
        and one gather reads the points."""
        r = F.sor(x, self.k, self.alpha, lengths)
        idx = draw_indices(r.lengths.cpu().tolist(), self.npoint)
        pts = torch.gather(r.kept_idx, 1, torch.from_numpy(idx).to(x.device))
        return x[torch.arange(x.shape[0], device=x.device)[:, None], pts]
