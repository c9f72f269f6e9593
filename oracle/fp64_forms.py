"""float64 closed forms of the differentiable pieces of the path -- TEST INFRASTRUCTURE ONLY.

The reference differentiates in fp32 (torch autograd over its matmul / topk / gather chains); where that gradient is a
cancellation (1/(d + 1e-8) weights, unit vectors of 1e-2-long offsets) its own rounding noise exceeds the 1e-5 bar.  The tests
therefore pin the kernels' gradients against these float64 evaluations of the SAME formulas on the SAME neighbour indices
(torch.float64 on CPU; the indices are the kernels' / the oracle's bit-exact ones), and report the reference's fp32 error
against the same float64 values next to it.  Each function cites the reference lines whose formula it evaluates.
"""
import numpy as np
import torch


def _t(a, grad=False):
    return torch.from_numpy(np.ascontiguousarray(np.asarray(a, np.float64))).requires_grad_(grad)


def _gather_pm(x_pm, idx):                      # x [B,M,U], idx [B,L,K] -> [B,L,K,U]
    B, M, U = x_pm.shape
    _, L, K = idx.shape
    return x_pm[:, :, None].expand(B, M, K, U).gather(1, idx[:, :, :, None].expand(B, L, K, U))


VALUE_SQUARED, VALUE_SQRT_CLAMP = 0, 1          # include/pcdist.h pcd_value_transform


def _i64(a):
    return a.long() if torch.is_tensor(a) else torch.from_numpy(np.asarray(a, np.int64))


def _gather_pts(x, idx, taps=None):
    """x [B,M,3] float64, idx [B,L] -> x[b, idx[b,l]] [B,L,3].  With `taps` (a list) the gathered copy keeps its gradient --
    the per-pair contributions before autograd scatters them onto x -- and (x, idx, copy) is appended to it."""
    g = torch.gather(x, 1, idx[:, :, None].expand(-1, -1, x.shape[2]))
    if taps is not None:
        g.retain_grad()
        taps.append((x, idx, g))
    return g


def _pair_d2(rows, cols, i, j, swap, taps):
    """d2 of the pairs (i[b,l], j[b,l]): sum((r_i - c_j)^2), or with swapped norms |c_i|^2 - 2 r_i.c_j + |r_j|^2
    (attack/GeoA3/knn_utils.py:13-15, N == M)."""
    r_i, c_j = _gather_pts(rows, i, taps), _gather_pts(cols, j, taps)
    if not swap:
        return ((r_i - c_j) ** 2).sum(-1)
    c_i, r_j = _gather_pts(cols, i, taps), _gather_pts(rows, j, taps)
    return (c_i * c_i).sum(-1) - 2.0 * (r_i * c_j).sum(-1) + (r_j * r_j).sum(-1)


def _transform64(d2, v32, transform):
    if transform == VALUE_SQUARED:
        return d2
    v = torch.from_numpy(np.asarray(v32, np.float64))
    pos = v > 0
    return torch.where(pos, d2 / torch.where(pos, 2.0 * v, torch.ones_like(v)), d2 * 0.0)


def nn1_surrogates64(rows, cols, row_arg, col_arg, row_min32, col_min32, swap, transform, taps=None):
    """Differentiable per-point values (v_row [B,N], v_col [B,M]) of the NN-1 minima at the given arg-mins.
    rows [B,N,3], cols [B,M,3]: float64 torch tensors (the caller's leaves).  VALUE_SQUARED: v = d2.  VALUE_SQRT_CLAMP:
    v = d2 / (2 v32), v32 the stored fp32 minimum (0 where v32 == 0) -- linear in d2, with the gradient of sqrt(d2) taken at
    the value torch's cdist backward divides by; its value is not the minimum.  Every loss over the minima (sums, maxima
    at a given arg-max, per-point weights) is then a torch expression of these, differentiated by autograd."""
    B, N, _ = rows.shape
    M = cols.shape[1]
    own_r = torch.arange(N).expand(B, N)
    own_c = torch.arange(M).expand(B, M)
    v_row = _transform64(_pair_d2(rows, cols, own_r, _i64(row_arg), swap, taps), row_min32, transform)
    v_col = _transform64(_pair_d2(rows, cols, _i64(col_arg), own_c, swap, taps), col_min32, transform)
    return v_row, v_col


def knn_pairs64(rows, cols, idx, swap, taps=None):
    """d2 [B,N,K] of the pairs (i, idx[b,i,k]) in float64 (forms as nn1_surrogates64); rows, cols float64 torch tensors
    (may be the same tensor)."""
    B, N, K = idx.shape
    i = torch.arange(N).repeat_interleave(K).expand(B, N * K)
    return _pair_d2(rows, cols, i, _i64(idx).reshape(B, N * K), swap, taps).reshape(B, N, K)


def kappa64(adv_pm, normal_pm, idx_self, nidx=None):
    """attack/GeoA3/loss_utils.py:60-90 in float64 (differentiable torch expression)."""
    idx = torch.from_numpy(np.asarray(idx_self[:, :, 1:], np.int64))
    q = _gather_pm(adv_pm, idx)
    d = q - adv_pm[:, :, None, :]
    u = d / d.norm(dim=-1, keepdim=True).clamp(min=1e-12)
    n = normal_pm if nidx is None else torch.gather(normal_pm, 1, torch.from_numpy(np.asarray(nidx, np.int64))[:, :, None].expand(-1, -1, 3))
    return (u * n[:, :, None, :]).sum(-1).abs().mean(-1)


def curvature_loss_grad64(adv_cf, normal_cf, ori_kappa, idx_self, nidx, gB):
    """loss_utils.py:72-105: value [b] and gradient w.r.t. adv [b,3,n] of sum_b gB[b] * mean_i (kappa_adv - ori_kappa[nidx])^2."""
    a = _t(np.asarray(adv_cf).transpose(0, 2, 1), True)
    kap = kappa64(a, _t(np.asarray(normal_cf).transpose(0, 2, 1)), idx_self, nidx)
    ok = torch.gather(_t(ori_kappa), 1, torch.from_numpy(np.asarray(nidx, np.int64)))
    v = ((kap - ok) ** 2).mean(-1)
    (v * _t(gB)).sum().backward()
    return v.detach().numpy(), kap.detach().numpy(), a.grad.numpy().transpose(0, 2, 1)


def knn_outlier_loss_grad64(pc_pm, dists, idx_self, alpha, gB):
    """attack/CW/CW_utils/dist_utils.py:143-153 / attack/GeoA3/loss_utils.py:148-157: value, mask and gradient w.r.t. the cloud.
    `dists` [B,N,K1] are the fp32 k-NN distances (the values the fp32 losses threshold); the gradient is evaluated in float64
    through d_ij = |p_i - p_j|^2 on the given indices."""
    p = _t(pc_pm, True)
    idx = torch.from_numpy(np.asarray(idx_self[:, :, 1:], np.int64))
    q = _gather_pm(p, idx)
    d = ((q - p[:, :, None, :]) ** 2).sum(-1)
    value = d.mean(-1)
    v32 = torch.from_numpy(np.asarray(dists, np.float64)[:, :, 1:]).mean(-1)
    thr = v32.mean(-1) + alpha * v32.std(-1)
    mask = (v32 > thr[:, None]).double()
    loss = (value * mask).mean(1)
    (loss * _t(gB)).sum().backward()
    return loss.detach().numpy(), mask.numpy(), p.grad.numpy()


def three_nn_interpolate_grad64(xyz1, xyz2, feat2, idx, gw, d32):
    """model/pointnet2_utils.py:289-300: out [B,N,D] and gradients w.r.t. xyz1, xyz2, feat2 of sum(out * gw).
    The weights 1/(d + 1e-8) amplify the fp32 cancellation error of the expansion-form distances (1e-3 relative on d ~ 1e-4), so
    the forward is evaluated on the SAME fp32 distances d32 [B,N,3] the reference and the kernels produce (bit-identical); what
    float64 pins is everything after them: the weights, the interpolation and the chain rule d(d_ij) = 2 (x1_i - x2_j)."""
    f2 = _t(feat2, True)
    d = _t(d32, True)
    ii = torch.from_numpy(np.asarray(idx, np.int64))
    r = 1.0 / (d + 1e-8)
    w = r / r.sum(-1, keepdim=True)
    out = (_gather_pm(f2, ii) * w[..., None]).sum(2)
    (out * _t(gw)).sum().backward()
    x1, x2 = _t(xyz1), _t(xyz2)
    diff = x1[:, :, None, :] - _gather_pm(x2, ii)                       # [B,N,3,3]
    t = 2.0 * d.grad[..., None] * diff
    g1 = t.sum(2)
    g2 = torch.zeros_like(x2)
    g2.scatter_add_(1, ii.reshape(ii.shape[0], -1, 1).expand(-1, -1, 3), (-t).reshape(t.shape[0], -1, 3))
    return out.detach().numpy(), g1.numpy(), g2.numpy(), f2.grad.numpy()
