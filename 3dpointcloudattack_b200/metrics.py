"""Exact float64 Chamfer and Hausdorff metrics for reporting how far a cloud moved, for batches of clouds of unequal
valid sizes (functional.nn_dist64, pcd_nn_dist64_forward in include/pcdist.h).

The reference reports these distances from utils/dis_utils_numpy.py:13-38 (scipy distance_matrix in float64, one cloud
at a time on the host).  The bodies of its functions are not recorded in this repository, so nothing here claims to be
a drop-in copy of them and there is no install() patch.  Both conventions in use are given, without choosing between
them:
    squared=True   mean / max of the squared nearest-neighbour distances (the CW ChamferDistance convention)
    squared=False  mean / max of the Euclidean nearest-neighbour distances (scipy cdist / distance_matrix)
Each function returns the two directional values (a_to_b [B], b_to_a [B]) in float64; sum or average them as the
report needs.  a [B,N,3] and b [B,M,3] are float32 CUDA tensors with any strides; a_lengths / b_lengths are None or
integer tensors [B] (sample i uses a[i, :a_lengths[i]] and b[i, :b_lengths[i]]), so SOR-kept clouds
(functional.sor's kept_idx / lengths) are scored without a loop over samples.  No autograd.
"""
from . import functional as F

__all__ = ["chamfer64", "hausdorff64"]


def chamfer64(a, b, a_lengths=None, b_lengths=None, squared=False):
    """Directional means of the nearest-neighbour distances: (a_to_b [B], b_to_a [B]) float64.  a_to_b averages, over
    the valid points of a, the distance to the nearest valid point of b."""
    r = F.nn_dist64(a, b, a_lengths, b_lengths)
    return (r.a_mean_sq, r.b_mean_sq) if squared else (r.a_mean, r.b_mean)


def hausdorff64(a, b, a_lengths=None, b_lengths=None, squared=False):
    """Directional maxima of the nearest-neighbour distances: (a_to_b [B], b_to_a [B]) float64.  The symmetric
    Hausdorff distance is their elementwise maximum."""
    r = F.nn_dist64(a, b, a_lengths, b_lengths)
    return (r.a_max_sq, r.b_max_sq) if squared else (r.a_max, r.b_max)
