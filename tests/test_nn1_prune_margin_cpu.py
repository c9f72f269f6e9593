"""The rounding margin of the pruned NN-1 sweep (DESIGN.md section 4.1), checked in float64 on the CPU.

The pruned sweep skips a chunk pair only when LB - E > U, which is safe only if every computed fp32 pair value lies within
E = 40 * 2^-24 * (|p|^2 + |q|^2) + 2^-100 (computed norms) of the exact squared distance of its two fp32 points.  The oracle
evaluates the pair values with the kernels' rounding sequence for every form and norm kind."""
import numpy as np
import pytest

from oracle import pcd_oracle as O

MARGIN_REL = 40.0 * 2.0 ** -24
MARGIN_ABS = 2.0 ** -100
FORMS = [(O.FORM_ROW_COL, O.NORM_MULSUM), (O.FORM_COL_ROW, O.NORM_MULSUM), (O.FORM_SUM_FIRST, O.NORM_FMA),
         (O.FORM_ROW_COL, O.NORM_FMA), (O.FORM_COL_ROW, O.NORM_FMA), (O.FORM_SUM_FIRST, O.NORM_MULSUM)]


def clouds(kind, rs):
    if kind == "uniform":
        c = rs.uniform(-1, 1, (2, 96, 3))
        return c, rs.uniform(-1, 1, (2, 80, 3))
    if kind == "near_copies_far_from_origin":      # the cancellation the margin exists for: big norms, tiny distances
        c = rs.uniform(-1, 1, (2, 96, 3)) * 3e3 + 1e4
        return c, c[:, :80] + rs.randn(2, 80, 3) * 1e-3
    if kind == "mixed_scales":
        c = rs.randn(2, 96, 3) * 10.0 ** rs.randint(-6, 7, (2, 96, 1))
        return c, rs.randn(2, 80, 3) * 10.0 ** rs.randint(-6, 7, (2, 80, 1))
    if kind == "subnormal":
        c = rs.randn(2, 96, 3) * 1e-20
        return c, c[:, :80] * (1 + 1e-3 * rs.randn(2, 80, 3))
    # exact copies and single-ulp neighbours
    c = rs.uniform(-2, 2, (2, 96, 3)).astype(np.float32)
    r = c[:, :80].copy()
    r[:, ::2] = np.nextafter(r[:, ::2], np.float32(np.inf))
    return c, r


@pytest.mark.parametrize("kind", ["uniform", "near_copies_far_from_origin", "mixed_scales", "subnormal", "ulp_neighbours"])
@pytest.mark.parametrize("form,norm", FORMS)
def test_pair_value_error_within_prune_margin(kind, form, norm):
    rs = np.random.RandomState(sum(map(ord, kind)) + 7 * form + norm)
    cols, rows = (np.asarray(a, np.float32) for a in clouds(kind, rs))
    nr, nc = O.norms(norm, rows), O.norms(norm, cols)
    d = O.pairwise(form, rows, cols, nr, nc).astype(np.float64)
    r64, c64 = rows.astype(np.float64), cols.astype(np.float64)
    exact = ((r64[:, :, None, :] - c64[:, None, :, :]) ** 2).sum(-1)
    e = MARGIN_REL * (nr.astype(np.float64)[:, :, None] + nc.astype(np.float64)[:, None, :]) + MARGIN_ABS
    assert np.isfinite(d).all()
    err = np.abs(d - exact)
    assert (err <= e).all(), float((err / e).max())
    # the constant keeps a factor of four over the bound derived in DESIGN.md (10 units of 2^-24)
    assert (err <= e / 4).all(), float((err / e).max())
