"""Drop-in for the knn_points consumers of attack/GeoA3/loss_utils.py (clouds are [b,3,n]).

Every loss below asks knn_points for the adv->ori nearest neighbours; the reference
recomputes that same K=1 query 4-6 times per iteration (GeoA3_attack.py:134-166) -- here the
repeats hit the one-entry NN-1 cache in functional.nn1, so one sweep serves them all.
"""
import torch

from . import functional as F
from .knn_utils import knn_gather, knn_points


def _normalize(input, p=2, dim=1, eps=1e-12):
    """attack/GeoA3/utility.py:_normalize."""
    return input / input.norm(p, dim).clamp(min=eps).unsqueeze(dim).expand_as(input)


def norm_l2_loss(adv_pc, ori_pc):
    """loss_utils.py:33-34."""
    return ((adv_pc - ori_pc) ** 2).sum(1).sum(1)


def _self_knn(pc, K):
    """Self k-NN of a [b,3,n] cloud in knn_points arithmetic: (point-major view, idx int32 [b,n,K])."""
    pts = pc.permute(0, 2, 1)
    det = pts.detach()
    _, idx = F.knn(det, det, K, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM, swap_norms=True)
    return pts, idx


def chamfer_loss(adv_pc, ori_pc):
    """loss_utils.py:36-43."""
    adv_KNN = knn_points(adv_pc.permute(0, 2, 1), ori_pc.permute(0, 2, 1), K=1)
    ori_KNN = knn_points(ori_pc.permute(0, 2, 1), adv_pc.permute(0, 2, 1), K=1)
    return adv_KNN.dists.contiguous().squeeze(-1).mean(-1) + ori_KNN.dists.contiguous().squeeze(-1).mean(-1)


def pseudo_chamfer_loss(adv_pc, ori_pc):
    """loss_utils.py:45-51."""
    adv_KNN = knn_points(adv_pc.permute(0, 2, 1), ori_pc.permute(0, 2, 1), K=1)
    return adv_KNN.dists.contiguous().squeeze(-1).mean(-1)


def hausdorff_loss(adv_pc, ori_pc):
    """loss_utils.py:53-58."""
    adv_KNN = knn_points(adv_pc.permute(0, 2, 1), ori_pc.permute(0, 2, 1), K=1)
    return adv_KNN.dists.contiguous().squeeze(-1).max(-1)[0]


def _get_kappa_ori(pc, normal, k=2):
    """loss_utils.py:60-70: mean_j |<unit(q_j - p), n_p>| over the k nearest neighbours (self excluded) -> [b,n].
    One k-NN select plus one fused kernel; the [b,3,n,k] neighbour gather is never materialised."""
    pts, idx = _self_knn(pc, k + 1)
    return F.kappa(pts, normal.permute(0, 2, 1), idx, nidx=None, skip_first=True)


def _get_kappa_adv(adv_pc, ori_pc, ori_normal, k=2):
    """loss_utils.py:72-90 -> (kappa [b,n], normal of the nearest original point [b,3,n])."""
    intra_KNN = knn_points(adv_pc.permute(0, 2, 1), ori_pc.permute(0, 2, 1), K=1)
    nidx = intra_KNN.idx.squeeze(-1)
    normal = knn_gather(ori_normal.permute(0, 2, 1), intra_KNN.idx).permute(0, 3, 1, 2).squeeze(3).contiguous()
    pts, idx = _self_knn(adv_pc, k + 1)
    return F.kappa(pts, ori_normal.permute(0, 2, 1), idx, nidx=nidx, skip_first=True), normal


def curvature_loss(adv_pc, ori_pc, adv_kappa, ori_kappa, k=2):
    """loss_utils.py:92-105."""
    intra_KNN = knn_points(adv_pc.permute(0, 2, 1), ori_pc.permute(0, 2, 1), K=1)
    onenn_ori_kappa = torch.gather(ori_kappa, 1, intra_KNN.idx.squeeze(-1)).contiguous()
    return ((adv_kappa - onenn_ori_kappa) ** 2).mean(-1)


# The four losses below are brute force in the reference -- [b,n,n] matrices of DIRECT differences
# ((p_i - p_j)^2 summed) and a topk.  Here the neighbours come from the k-NN select (expansion form, the arithmetic of
# every other k-NN in the reference); the two forms order candidates identically except where two distances agree to
# fp32 rounding.  Whatever a loss reads off the neighbours (their squared distances included) is recomputed from the
# gathered points in the reference's direct form, so values carry no expansion-form cancellation error.
def _neighbours(pc, k):
    """[b,3,n] -> (idx [b,n,k] int64 of the k nearest other points, nn_pts [b,3,n,k] gathered, differentiable).
    In the reference's direct form d(i,i) = 0 exactly, so self is always dropped.  In the expansion form a twin less than
    ~3e-4 away (unit scale) can rank before self, so the entry equal to the point's own index is dropped wherever it is
    (the last one when self is not among the k + 1)."""
    b, _, n = pc.size()
    pts, idx = _self_knn(pc, k + 1)
    idx = idx.long()
    is_self = idx == torch.arange(n, device=idx.device).view(1, n, 1)
    drop = torch.where(is_self.any(2), is_self.int().argmax(2), torch.full_like(idx[:, :, 0], k))
    idx = idx[torch.arange(k + 1, device=idx.device) != drop.unsqueeze(2)].view(b, n, k)
    nn_pts = knn_gather(pts, idx).permute(0, 3, 1, 2)
    return idx, nn_pts


def displacement_loss(adv_pc, ori_pc, k=16):
    """loss_utils.py:107-115."""
    b, _, n = adv_pc.size()
    with torch.no_grad():
        inter_idx, _ = _neighbours(ori_pc, k)
    theta_distance = ((adv_pc - ori_pc) ** 2).sum(1)
    nn_theta_distances = torch.gather(theta_distance, 1, inter_idx.reshape(b, n * k)).view(b, n, k)
    return ((nn_theta_distances - theta_distance.unsqueeze(2)) ** 2).mean(2)


def corresponding_normal_loss(adv_pc, normal, k=2):
    """loss_utils.py:116-125 (the kappa of _get_kappa_ori with a given normal field)."""
    pts, idx = _self_knn(adv_pc, k + 1)
    return F.kappa(pts, normal.permute(0, 2, 1), idx, nidx=None, skip_first=True)


def repulsion_loss(pc, k=4, h=0.03):
    """loss_utils.py:127-131."""
    _, nn_pts = _neighbours(pc, k)
    dis = ((nn_pts - pc.unsqueeze(3)) ** 2).sum(1)                     # [b,n,k] direct form, as the reference's matrix entries
    return -(dis * torch.exp(-(dis ** 2) / (h ** 2))).mean(2)


def distance_kmean_loss(pc, k):
    """loss_utils.py:133-141."""
    b, _, n = pc.size()
    idx, nn_pts = _neighbours(pc, k)
    dis = ((pc.unsqueeze(3) - nn_pts + 1e-12) ** 2).sum(1).sqrt()      # [b,n,k]
    dis_mean = dis.mean(-1)
    dis_mean_k = torch.gather(dis_mean, 1, idx.reshape(b, n * k)).view(b, n, k)
    return torch.abs(dis_mean.unsqueeze(2) - dis_mean_k).mean(-1)


def kNN_smoothing_loss(adv_pc, k, threshold_coef=1.05):
    """loss_utils.py:143-157.  The reference computes the threshold inside the autograd graph, but the comparison that
    consumes it is a .float() of a boolean, so no gradient flows through it: same fused epilogue as KNNDist."""
    loss, _, _, _ = F.knn_outlier_loss(adv_pc.permute(0, 2, 1), k, threshold_coef, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM,
                                       swap_norms=True)
    return loss
