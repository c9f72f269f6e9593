"""Drop-points defences: SOR (statistical outlier removal) <- attack/SIadv/baselines/defense/drop_points/SOR.py, and
SRS (simple random sampling), the other drop-points baseline of IF-Defense.

SIadv's baselines/ tree comes from IF-Defense; the defaults k = 2, alpha = 1.1, npoint = 1024 are IF-Defense's
published values.  The statistic runs in the float64 kernels behind functional.sor.  Without a sampler, the
resampling to npoint points keeps the reference's numpy draws, so a seeded np.random gives the same clouds.  With a
functional.PointSampler, the draws run on the device (functional.sample_points): no host synchronisation, graph-
capturable, and differentiable with respect to the kept points.  There is no install() patch for this module: the
class layouts of SOR.py and SRS.py are not recorded here.
"""
import numpy as np
import torch
from torch import nn

from . import functional as F

__all__ = ["SORDefense", "SRSDefense", "DefendedVictim", "draw_indices"]


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


def _gather_points(x, idx):
    """x [B,N,3], idx [B,M] int64 with -1 for "no point" -> [B,M,3]: x[b, idx[b]], NaN where idx is -1.  Differentiable
    with respect to x (the backward of the gather is a scatter-add)."""
    pts = torch.gather(x, 1, idx.clamp_min(0)[..., None].expand(-1, -1, x.shape[2]))
    return pts.masked_fill(idx[..., None] < 0, float("nan"))


class SORDefense(nn.Module):
    """Statistical outlier removal: drop the points whose mean squared distance to their k nearest neighbours exceeds
    mean + alpha * std over the cloud, then resample every cloud to npoint points.
    sampler: None (numpy's global generator, the reference's draws) or a functional.PointSampler (device draws)."""

    def __init__(self, k=2, alpha=1.1, npoint=1024, sampler=None):
        super().__init__()
        self.k = k
        self.alpha = alpha
        self.npoint = npoint
        self.sampler = sampler

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

    def forward(self, x, lengths=None):
        """process_data(outlier_removal(x, lengths)) without building the list: the draws index the kept-index table,
        and one gather reads the points.  x [B,N,3] -> [B, npoint, 3].
        Without a sampler: numpy's draws (one device-to-host copy of the kept counts), no gradient, and a ValueError
        when a sample keeps no point.  With one: functional.sample_points draws through the kept-index table on the
        device, with no host synchronisation (graph-capturable); the result is differentiable with respect to x, the
        keep-mask being a constant, so the gradient reaches exactly the drawn points.  A sample that keeps no point
        comes out as npoint NaN points."""
        if self.sampler is None:
            return self._forward_numpy(x, lengths)
        _, _, _, kept, kept_n = F._sor32(x, self.k, self.alpha, lengths)
        idx = F.sample_points(kept_n, x.shape[1], self.npoint, self.sampler, table=kept)
        return _gather_points(x, idx)

    @torch.no_grad()
    def _forward_numpy(self, x, lengths):
        r = F.sor(x, self.k, self.alpha, lengths)
        idx = draw_indices(r.lengths.cpu().tolist(), self.npoint)
        pts = torch.gather(r.kept_idx, 1, torch.from_numpy(idx).to(x.device))
        return x[torch.arange(x.shape[0], device=x.device)[:, None], pts]


class SRSDefense(nn.Module):
    """Simple random sampling: keep K - drop_num of the K points of every cloud, drawn uniformly without replacement.
    IF-Defense's baselines/defense/drop_points/SRS.py draws np.random.choice(K, K - drop_num, replace=False) per sample
    in batch order and gathers the points; that file is not in this repository, so this restates its published
    behaviour.  sampler: None (those numpy draws) or a functional.PointSampler (device draws, no host synchronisation,
    graph-capturable).  Either way the result is differentiable with respect to the kept points."""

    def __init__(self, drop_num=500, sampler=None):
        super().__init__()
        self.drop_num = drop_num
        self.sampler = sampler

    def forward(self, x):
        """x [B,K,3] -> [B, K - drop_num, 3]"""
        B, K = x.shape[:2]
        if not 0 <= self.drop_num < K:
            raise ValueError(f"drop_num must be in [0, {K}) for clouds of {K} points, got {self.drop_num}")
        keep = K - self.drop_num
        if B == 0:
            return x[:, :keep]
        if self.sampler is None:
            idx = np.stack([np.random.choice(K, keep, replace=False) for _ in range(B)])
            idx = torch.from_numpy(idx.astype(np.int64)).to(x.device)
        else:
            idx = F.sample_points(torch.full((B,), K, dtype=torch.int32, device=x.device), K, keep, self.sampler)
        return torch.gather(x, 1, idx[..., None].expand(-1, -1, x.shape[2]))


class DefendedVictim(nn.Module):
    """A victim behind a point-cloud defence, in the victims' calling convention: forward(x [B,3,K]) runs
    defence(x.transpose(1, 2)) on [B,K,3] clouds, hands the defended [B,3,K'] cloud to the victim and returns the
    victim's output unchanged (a tuple with the logits first).  With a device-sampled defence it can be the model of
    cw_loop.CWAttack / KNNAttack, graph capture included: the attack then runs through the defence."""

    def __init__(self, victim, defence):
        super().__init__()
        self.victim = victim
        self.defence = defence

    def forward(self, x):
        return self.victim(self.defence(x.transpose(1, 2)).transpose(1, 2))
