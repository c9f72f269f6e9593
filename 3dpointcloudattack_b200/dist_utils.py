"""Drop-in for the point-set distance wrappers of attack/CW/CW_utils/dist_utils.py (copies:
attack/Gen3DAdv/utils/dist_utils.py, attack/SIadv/baselines/attack/util/dist_utils.py):
L2Dist, ChamferDist, HausdorffDist, KNNDist, ChamferkNNDist -- same constructor / forward signatures.

Differences that do not change results: `weights` is moved to the input's device instead of
the hard-coded `.cuda()` (dist_utils.py:68,105,156), so one process per GPU works unchanged.
"""
import torch
import torch.nn as nn

from . import functional as F
from .distance import chamfer, hausdorff


def _weights(weights, B, device):
    if weights is None:
        return torch.ones((B,), device=device)
    return torch.as_tensor(weights).float().to(device)


class L2Dist(nn.Module):
    """dist_utils.py:9-35: per sample sqrt(sum((adv - ori)^2)) over the points and channels, times weights; the distance
    AOF runs with.  Either layout ([B, K, 3] or [B, 3, K]) as long as both clouds share it."""

    def forward(self, adv_pc, ori_pc, weights=None, batch_avg=True):
        B = adv_pc.shape[0]
        dist = torch.sqrt(torch.sum((adv_pc - ori_pc) ** 2, dim=[1, 2]))
        dist = dist * _weights(weights, B, adv_pc.device)
        if batch_avg:
            return dist.mean()
        return dist


class _SetDist(nn.Module):
    _fn = None

    def __init__(self, method='adv2ori'):
        super().__init__()
        self.method = method

    def forward(self, adv_pc, ori_pc, weights=None, batch_avg=True):
        """adv_pc, ori_pc: [B, K, 3]; weights: [B] or None (dist_utils.py:49-72 / 86-109)."""
        B = adv_pc.shape[0]
        loss1, loss2 = type(self)._fn(adv_pc, ori_pc)          # [B], adv2ori, ori2adv
        if self.method == 'adv2ori':
            loss = loss1
        elif self.method == 'ori2adv':
            loss = loss2
        else:
            loss = (loss1 + loss2) / 2.
        loss = loss * _weights(weights, B, adv_pc.device)
        if batch_avg:
            return loss.mean()
        return loss


class ChamferDist(_SetDist):
    """dist_utils.py:38-72."""
    _fn = staticmethod(lambda a, o: chamfer(a, o))


class HausdorffDist(_SetDist):
    """dist_utils.py:75-109."""
    _fn = staticmethod(lambda a, o: hausdorff(a, o))


class KNNDist(nn.Module):
    """kNN outlier loss of the AAAI'20 kNN attack (dist_utils.py:112-160).

    dist[i,j] = (|p_j|^2 - 2 p_i.p_j) + |p_i|^2 ; top-(k+1) smallest per row, first column
    dropped (assumed self) ; value = mean of the k ; threshold = mean + alpha*std (unbiased,
    no grad) ; loss = mean(value * (value > threshold)).
    """

    def __init__(self, k=5, alpha=1.05):
        super().__init__()
        self.k = k
        self.alpha = alpha

    def forward(self, pc, weights=None, batch_avg=True):
        B, K = pc.shape[:2]
        # k-NN select + ONE fused epilogue kernel (value, unbiased std, threshold, mask, masked mean) and ONE backward
        # kernel through the indices, instead of nine torch launches and their autograd nodes (dist_utils.py:143-153)
        loss, _, _, _ = F.knn_outlier_loss(pc, self.k, self.alpha, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM)   # [B]
        loss = loss * _weights(weights, B, pc.device)
        if batch_avg:
            return loss.mean()
        return loss


class ChamferkNNDist(nn.Module):
    """dist_utils.py:189-223: chamfer_weight * ChamferDist + knn_weight * KNNDist."""

    def __init__(self, chamfer_method='adv2ori', knn_k=5, knn_alpha=1.05, chamfer_weight=5., knn_weight=3.):
        super().__init__()
        self.chamfer_dist = ChamferDist(method=chamfer_method)
        self.knn_dist = KNNDist(k=knn_k, alpha=knn_alpha)
        self.w1 = chamfer_weight
        self.w2 = knn_weight

    def forward(self, adv_pc, ori_pc, weights=None, batch_avg=True):
        chamfer_loss = self.chamfer_dist(adv_pc, ori_pc, weights=weights, batch_avg=batch_avg)
        knn_loss = self.knn_dist(adv_pc, weights=weights, batch_avg=batch_avg)
        return chamfer_loss * self.w1 + knn_loss * self.w2
