"""The point stage of the pruned NN-1 sweep's filter (DESIGN.md section 4.0): its lower bound on the distance from a point
to a chunk, evaluated with the kernel's fp32 roundings, checked in float64 on the CPU against exact distances."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from test_nn1_prune_margin_cpu import clouds  # noqa: E402


LB_SCALE = np.float32(1.0 - 2.0 ** -20)


@pytest.mark.parametrize("kind", ["uniform", "near_copies_far_from_origin", "mixed_scales", "subnormal", "ulp_neighbours"])
def test_point_to_box_bound_below_exact_distance(kind):
    """The point stage of the filter skips chunk C for a lane only when fl(LB - E) exceeds the lane's minimum, with LB the
    fp32 squared gap between the lane's point and C's box, times (1 - 2^-20).  That is exact only if LB, with every
    rounding of the kernel (gap, squares, two sums, scale), never exceeds the exact squared distance from the point to a
    point of C, except by the absolute error of rounding into the subnormal range (at most 2^-150 for each of the five
    roundings), which the 2^-100 term of E absorbs many times over."""
    rs = np.random.RandomState(sum(map(ord, kind)) + 3)
    a, b = (np.asarray(x, np.float32) for x in clouds(kind, rs))
    checked = 0
    for pts, other in ((a, b), (b, a)):
        for s in range(pts.shape[0]):
            perm = rs.permutation(other.shape[1])
            for k in range(0, other.shape[1], 32):
                chunk = other[s, perm[k:k + 32]]
                lo, hi = chunk.min(0), chunk.max(0)                     # fp32 box, as nn1_bucket writes it
                p = pts[s]
                with np.errstate(over="ignore", under="ignore"):
                    g = np.maximum(np.maximum(lo[None] - p, p - hi[None]), np.float32(0))
                    g2 = g * g
                    lb = ((g2[:, 0] + g2[:, 1]) + g2[:, 2]) * LB_SCALE
                assert lb.dtype == np.float32
                exact = ((p.astype(np.float64)[:, None, :] - chunk.astype(np.float64)[None]) ** 2).sum(-1).min(1)
                assert (lb.astype(np.float64) <= exact + 5 * 2.0 ** -150).all(), float((lb - exact).max())
                checked += int((lb > 0).sum())
    assert checked > 0
