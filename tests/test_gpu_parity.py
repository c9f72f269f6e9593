"""GPU parity: the sm_100a kernels (through the ctypes C ABI and the drop-in Python surface)
against the CPU oracle and against the golden vectors produced by the unmodified reference.

Bar (BASELINE.json north_star): argmin / kNN indices bit-exact under the lowest-index tie-break,
distances and gradients within 1e-5 relative (fp32).  Where the arithmetic is op-order
faithful we assert the stronger property: bit-identical fp32 values.
"""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from conftest import load_golden, rel_inf
from knn_proof import assert_knn_near_tie_proof
from oracle import fp64_forms as F64
from oracle import pcd_oracle as O

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
F = pcd.functional

RTOL = 1e-5


def cu(a, grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return t.requires_grad_(grad)


def npy(t):
    return t.detach().cpu().numpy()


FORMS = {
    "row_col_mulsum": (F.FORM_ROW_COL, F.NORM_MULSUM, O.FORM_ROW_COL, O.NORM_MULSUM),
    "col_row_mulsum": (F.FORM_COL_ROW, F.NORM_MULSUM, O.FORM_COL_ROW, O.NORM_MULSUM),
    "sum_first_fma": (F.FORM_SUM_FIRST, F.NORM_FMA, O.FORM_SUM_FIRST, O.NORM_FMA),
}


def oracle_nn1(rows, cols, oform, onorm, swap=False):
    nr, nc = O.norms(onorm, rows), O.norms(onorm, cols)
    if swap:
        nr, nc = O.norms(onorm, cols), O.norms(onorm, rows)
    return O.nn1(oform, rows, cols, nr, nc)


def check_nn1(rows, cols, form_key, swap=False):
    form, norm, oform, onorm = FORMS[form_key]
    r = F.nn1(cu(rows), cu(cols), form, norm, swap_norms=swap, cache=False)
    o = oracle_nn1(rows, cols, oform, onorm, swap)
    assert np.array_equal(npy(r.row_min), o.row_min)
    assert np.array_equal(npy(r.col_min), o.col_min)
    assert np.array_equal(npy(r.row_arg), o.row_arg)
    assert np.array_equal(npy(r.col_arg), o.col_arg)
    np.testing.assert_allclose(npy(r.row_sum), o.row_min.sum(1, dtype=np.float64), rtol=2e-6)
    np.testing.assert_allclose(npy(r.col_sum), o.col_min.sum(1, dtype=np.float64), rtol=2e-6)
    assert np.array_equal(npy(r.row_max), o.row_min.max(1)) and np.array_equal(npy(r.col_max), o.col_min.max(1))
    assert np.array_equal(npy(r.row_argmax), o.row_min.argmax(1))
    assert np.array_equal(npy(r.col_argmax), o.col_min.argmax(1))


# ------------------------------------------------------------------ NN-1 sweep vs the oracle
@pytest.mark.parametrize("form_key", list(FORMS))
@pytest.mark.parametrize("shape", [(1, 1, 1), (2, 33, 257), (3, 700, 1000), (1, 1025, 31), (2, 1024, 1024),
                                   (5, 300, 300), (1, 4096, 4096), (4, 2048, 513)])
def test_nn1_bit_exact_random(form_key, shape):
    B, N, M = shape
    rs = np.random.RandomState(B * 7919 + N * 31 + M)
    cols = (rs.rand(B, M, 3) - 0.5).astype(np.float32)
    rows = (rs.rand(B, N, 3) - 0.5).astype(np.float32)
    k = min(N, M)
    rows[:, :k] = cols[:, :k] + 0.01 * rs.randn(B, k, 3).astype(np.float32)
    check_nn1(rows, cols, form_key)


@pytest.mark.parametrize("form_key", list(FORMS))
def test_nn1_swapped_norms(form_key):
    g = load_golden("a3_knn_utils")
    check_nn1(g["adv"], g["ori"], form_key, swap=True)


@pytest.mark.parametrize("form_key", list(FORMS))
def test_nn1_ties_and_duplicates(form_key):
    g = load_golden("a2_distance_ties")
    check_nn1(g["gts"], g["preds"], form_key)
    # all points identical: every distance equal -> every argmin must be index 0
    same = np.full((2, 300, 3), 0.25, np.float32)
    form, norm, _, _ = FORMS[form_key]
    r = F.nn1(cu(same), cu(same[:, :77]), form, norm, cache=False)
    assert int(r.row_arg.abs().max()) == 0 and int(r.col_arg.abs().max()) == 0
    # integer grid: exact ties everywhere
    gx = np.stack(np.meshgrid(np.arange(8), np.arange(8), np.arange(8), indexing="ij"), -1).reshape(1, -1, 3)
    check_nn1(gx.astype(np.float32), (gx[:, ::3] + 0.5).astype(np.float32), form_key)


@pytest.mark.parametrize("layout", ["channel_first", "strided"])
def test_nn1_layouts(layout):
    rs = np.random.RandomState(5)
    rows = rs.randn(2, 500, 3).astype(np.float32); cols = rs.randn(2, 400, 3).astype(np.float32)
    if layout == "channel_first":
        tr = cu(np.ascontiguousarray(rows.transpose(0, 2, 1))).transpose(1, 2)
        tc = cu(np.ascontiguousarray(cols.transpose(0, 2, 1))).transpose(1, 2)
    else:
        big_r = torch.zeros(2, 500, 7, device="cuda"); big_r[:, :, 2:5] = cu(rows); tr = big_r[:, :, 2:5]
        big_c = torch.zeros(3, 400, 3, device="cuda"); big_c[1:] = cu(cols); tc = big_c[1:]
    r = F.nn1(tr, tc, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    o = oracle_nn1(rows, cols, O.FORM_SUM_FIRST, O.NORM_FMA)
    assert np.array_equal(npy(r.row_min), o.row_min) and np.array_equal(npy(r.col_arg), o.col_arg)


@pytest.mark.parametrize("tiling", [(2, 32), (4, 64), (8, 256), (8, 128), (16, 256), (16, 64)])
def test_nn1_every_tiling(tiling):
    F.force_tiling(*tiling)
    try:
        g = load_golden("a2_distance_ragged")
        check_nn1(g["gts"], g["preds"], "sum_first_fma")
        rs = np.random.RandomState(1)
        # 1500 x 2100: dense, streamed raw; 1501 x 2102: not a multiple of 4 -> packed through the workspace
        check_nn1(rs.randn(3, 1500, 3).astype(np.float32), rs.randn(3, 2100, 3).astype(np.float32), "row_col_mulsum")
        check_nn1(rs.randn(2, 1501, 3).astype(np.float32), rs.randn(2, 2102, 3).astype(np.float32), "col_row_mulsum")
    finally:
        F.force_tiling(0, 0)


def test_nn1_clouds_too_large_for_shared_memory_staging():
    """> 17 K points per cloud: the fix-up re-scans from global memory instead of a staged copy (same results)."""
    rs = np.random.RandomState(77)
    cols = (rs.rand(1, 17408, 3) - 0.5).astype(np.float32)
    rows = (cols[:, :17200] + 0.002 * rs.randn(1, 17200, 3)).astype(np.float32)
    check_nn1(rows, cols, "sum_first_fma")
    check_nn1(np.ascontiguousarray(cols[:, :17100]), rows, "row_col_mulsum")


def test_nn1_full_size_c2_against_oracle():
    """BASELINE config 2 (B=32, N=M=4096, sigma=0.01): every index and value against the C oracle."""
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    ori = synth.face_clouds(32, 4096, seed=1234)
    adv = synth.perturb(ori, 0.01, seed=99)
    check_nn1(ori.numpy(), adv.numpy(), "sum_first_fma")


def test_nn1_large_properties():
    """Size-independent properties at a size the oracle is not asked to do: role swap symmetry
    (rows<->cols gives transposed answers bit-for-bit for the symmetric form) and idempotence."""
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    ori = synth.face_clouds(8, 16384, seed=7).cuda(); adv = synth.perturb(ori.cpu(), 0.01, seed=8).cuda()
    a = F.nn1(ori, adv, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    b = F.nn1(adv, ori, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    assert torch.equal(a.row_min, b.col_min) and torch.equal(a.col_min, b.row_min)
    assert torch.equal(a.row_arg, b.col_arg) and torch.equal(a.col_arg, b.row_arg)
    c = F.nn1(ori, adv, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    assert torch.equal(a.row_min, c.row_min) and torch.equal(a.col_arg, c.col_arg)
    # a cloud against itself: every point's nearest neighbour is itself at (rounded) zero
    s = F.nn1(ori, ori, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    ar = torch.arange(16384, device="cuda", dtype=torch.int32).expand(8, -1)
    assert torch.equal(s.row_arg, ar) and torch.equal(s.col_arg, ar)


# ------------------------------------------------- a2: distance.py against the reference
@pytest.mark.parametrize("tag", ["face", "iter0", "ragged"])
def test_a2_distance_vs_reference(tag):
    g = load_golden("a2_distance_" + tag)
    for name, mod in (("chamfer", pcd.distance.chamfer), ("hausdorff", pcd.distance.hausdorff)):
        p, t = cu(g["preds"], True), cu(g["gts"], True)
        l1, l2 = mod(p, t)
        ((l1 * cu(g["g1"])).sum() + (l2 * cu(g["g2"])).sum()).backward()
        np.testing.assert_allclose(npy(l1), g[name + "_l1"], rtol=RTOL, atol=1e-12)
        np.testing.assert_allclose(npy(l2), g[name + "_l2"], rtol=RTOL, atol=1e-12)
        if tag != "iter0":      # |adv-ori| ~ 1e-7: the reference's own fp32 gradient is rounding noise
            assert rel_inf(npy(p.grad), g[name + "_gp"]) < RTOL
            assert rel_inf(npy(t.grad), g[name + "_gg"]) < RTOL
        gp, gg = (O.chamfer_distance_grads if name == "chamfer" else O.hausdorff_distance_grads)(
            g["preds"], g["gts"], g["g1"], g["g2"])
        assert rel_inf(npy(p.grad), gp) < RTOL and rel_inf(npy(t.grad), gg) < RTOL
    r = F.nn1(cu(g["gts"]), cu(g["preds"]), F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    assert np.array_equal(npy(r.row_min), g["row_min"]) and np.array_equal(npy(r.col_min), g["col_min"])
    assert np.array_equal(npy(r.row_arg), g["row_arg"]) and np.array_equal(npy(r.col_arg), g["col_arg"])


def test_a2_set_distance_variant():
    g = load_golden("a2_set_distance")
    np.testing.assert_allclose(npy(pcd.set_distance.chamfer(cu(g["preds"]), cu(g["gts"]))), g["chamfer"], rtol=RTOL)
    np.testing.assert_allclose(npy(pcd.set_distance.hausdorff(cu(g["preds"]), cu(g["gts"]))), g["hausdorff"], rtol=RTOL)


def test_fused_chamfer_hausdorff_shares_one_sweep():
    g = load_golden("a2_distance_face")
    p, t = cu(g["preds"], True), cu(g["gts"])
    n0 = F.launches()
    c1, c2 = pcd.distance.chamfer(p, t)
    h1, h2 = pcd.distance.hausdorff(p, t)
    assert F.launches() - n0 == 3          # arm + sweep + fix-up; the second call is served by the one-entry cache
    (c1.sum() + c2.sum() + h1.sum() + h2.sum()).backward()
    with torch.no_grad():
        p.add_(0.001)                        # in-place update bumps the version -> no stale hit
    c1b, _ = pcd.distance.chamfer(p, t)
    assert F.launches() - n0 == 3 + 1 + 3
    assert not torch.equal(c1, c1b)


# ------------------------------------------------- a1: dis_utils_torch.py against the reference
def test_a1_dis_utils_torch_vs_reference():
    g = load_golden("a1_dis_utils_torch")
    D = pcd.dis_utils_torch
    for fn in ("chamfer", "sgd_hausdorff_dis", "bid_hausdorff_dis"):
        a, b = cu(g["a"], True), cu(g["b"], True)
        v = getattr(D, fn)(a, b)
        assert v.dim() == 0
        v.backward()
        np.testing.assert_allclose(npy(v), g[fn], rtol=RTOL)
        # closed-form float64 gradient: 1e-5.  The reference's own fp32 cdist backward
        # (x*sum(ratio) - ratio@y, a cancellation) carries ~1e-5 of rounding noise itself: 5e-5.
        wa = {"chamfer": dict(w_col_sum=1 / 3, w_row_sum=1 / 3), "sgd_hausdorff_dis": dict(w_row_max=1.0)}.get(fn)
        if wa is None:
            row_wins = O.dis_sgd_hausdorff(g["a"], g["b"]) >= O.dis_sgd_hausdorff(g["b"], g["a"])
            wa = dict(w_row_max=1.0) if row_wins else dict(w_col_max=1.0)
        oga, ogb = O.dis_grads(g["a"], g["b"], **wa)
        assert rel_inf(npy(a.grad), oga) < RTOL and rel_inf(npy(b.grad), ogb) < RTOL, fn
        # against the reference's fp32 autograd: 1e-5 plus the reference's OWN distance from the float64 closed form (measured
        # here, printed): its cdist backward x*sum(ratio) - ratio@y is a cancellation
        ref_a, ref_b = rel_inf(g[fn + "_ga"], oga), rel_inf(g[fn + "_gb"], ogb)
        print(f"a1 {fn}: reference fp32 autograd vs float64 closed form {ref_a:.1e} / {ref_b:.1e}; ours {rel_inf(npy(a.grad), oga):.1e} / {rel_inf(npy(b.grad), ogb):.1e}")
        assert rel_inf(npy(a.grad), g[fn + "_ga"]) < RTOL + ref_a, fn
        assert rel_inf(npy(b.grad), g[fn + "_gb"]) < RTOL + ref_b, fn
    np.testing.assert_allclose(npy(D.chamfer(cu(g["ka"]), cu(g["kb"]))), g["k_chamfer"], rtol=RTOL)
    np.testing.assert_allclose(npy(D.sgd_hausdorff_dis(cu(g["ka"]), cu(g["kb"]))), g["k_sgd"], rtol=RTOL)
    np.testing.assert_allclose(npy(D.bid_hausdorff_dis(cu(g["ka"]), cu(g["kb"]))), g["k_bid"], rtol=RTOL)
    # oracle (correctly rounded sqrt) agrees bit for bit on the reductions that do not sum
    assert npy(D.sgd_hausdorff_dis(cu(g["a"]), cu(g["b"]))) == O.dis_sgd_hausdorff(g["a"], g["b"])
    assert npy(D.bid_hausdorff_dis(cu(g["a"]), cu(g["b"]))) == O.dis_bid_hausdorff(g["a"], g["b"])


def test_a1_hausdorff_exact_ties_are_pinned():
    """Exact ties of the OUTER max (utils/dis_utils_torch.py:19-28).  `torch.max(v)` (full reduce) hands every tied maximum an
    equal share of the gradient; the kernels route it to the FIRST maximum (lowest index), the rule of torch.max(dim) that the
    rest of the path follows.  Pinned here: values identical; the gradient mass is the same, it lands on the first of the
    tied points instead of being split; `bid_hausdorff_dis`'s 0.5 / 0.5 split between the two DIRECTIONS is reproduced
    (it is torch's own elementwise max in the shim).  Listed in INTEGRATION.md."""
    D = pcd.dis_utils_torch
    rs = np.random.RandomState(3)
    b_ = (rs.rand(1, 3, 40).astype(np.float32) - 0.5) * 0.2
    a_ = b_.copy() + 0.001
    a_[0, :, 7] = [2.0, 0.5, -0.25]
    a_[0, :, 23] = a_[0, :, 7]                       # two identical farthest points: exact tie of max_i min_j
    ar, br = torch.from_numpy(a_).requires_grad_(True), torch.from_numpy(b_).requires_grad_(True)
    M = torch.cdist(ar.permute(0, 2, 1), br.permute(0, 2, 1), p=2)      # the reference formulation, on CPU
    ref = torch.max(torch.min(M[0], dim=1)[0]); ref.backward()
    a, b = cu(a_, True), cu(b_, True)
    v = D.sgd_hausdorff_dis(a, b); v.backward()
    np.testing.assert_allclose(npy(v), ref.item(), rtol=RTOL)
    ga, gr = npy(a.grad)[0], ar.grad.numpy()[0]
    assert np.abs(gr[:, 7] - gr[:, 23]).max() == 0 and np.abs(gr[:, 7]).max() > 0          # reference: even split
    assert np.abs(ga[:, 23]).max() == 0                                                      # ours: all on the first maximum
    np.testing.assert_allclose(ga[:, 7], gr[:, 7] + gr[:, 23], rtol=1e-5)                     # same gradient mass
    np.testing.assert_allclose(npy(b.grad)[0], br.grad.numpy()[0], rtol=1e-5, atol=1e-7)      # the shared partner sees the same total
    # direction tie of bid_hausdorff_dis: one pair, d_ab == d_ba exactly -> torch.max(a, b) gives each direction 0.5
    a1 = np.array([[[0.0], [0.0], [0.0]]], np.float32); b1 = np.array([[[0.3], [0.4], [0.0]]], np.float32)
    a, b = cu(np.repeat(a1, 4, 2) , True), cu(np.repeat(b1, 4, 2), True)
    ar, br = torch.from_numpy(np.repeat(a1, 4, 2)).requires_grad_(True), torch.from_numpy(np.repeat(b1, 4, 2)).requires_grad_(True)
    Mr = torch.cdist(ar.permute(0, 2, 1), br.permute(0, 2, 1), p=2)
    refb = torch.max(torch.max(torch.min(Mr[0], dim=1)[0]), torch.max(torch.min(Mr[0], dim=0)[0])); refb.backward()
    vb = D.bid_hausdorff_dis(a, b); vb.backward()
    np.testing.assert_allclose(npy(vb), refb.item(), rtol=RTOL)
    np.testing.assert_allclose(npy(a.grad).sum(2), ar.grad.numpy().sum(2), rtol=1e-5)        # total per cloud identical; within the
    np.testing.assert_allclose(npy(b.grad).sum(2), br.grad.numpy().sum(2), rtol=1e-5)        # cloud it sits on the first tied point


# ------------------------------------------------- L3 wrappers against the reference
def test_l3_dist_utils_vs_reference():
    g = load_golden("l3_dist_utils")
    DU = pcd.dist_utils
    w = torch.from_numpy(g["weights"])          # CPU weights, like the reference's callers pass
    for method in ("adv2ori", "ori2adv", "avg"):
        for cls in ("ChamferDist", "HausdorffDist"):
            a = cu(g["adv"], True)
            v = getattr(DU, cls)(method=method)(a, cu(g["ori"]), weights=w, batch_avg=False)
            (v * cu(g["gB"])).sum().backward()
            np.testing.assert_allclose(npy(v), g[f"{cls}_{method}"], rtol=RTOL)
            assert rel_inf(npy(a.grad), g[f"{cls}_{method}_g"]) < RTOL
    a = cu(g["adv"], True)
    v = DU.ChamferDist()(a, cu(g["ori"])); v.backward()
    np.testing.assert_allclose(npy(v), g["ChamferDist_default_mean"], rtol=RTOL)
    assert rel_inf(npy(a.grad), g["ChamferDist_default_mean_g"]) < RTOL
    for k in (5, 16):
        a = cu(g["adv"], True)
        v = DU.KNNDist(k=k, alpha=1.05)(a, weights=w, batch_avg=False)
        (v * cu(g["gB"])).sum().backward()
        np.testing.assert_allclose(npy(v), g[f"KNNDist_k{k}"], rtol=RTOL)
        assert rel_inf(npy(a.grad), g[f"KNNDist_k{k}_g"]) < RTOL
    a = cu(g["adv"], True)
    v = DU.ChamferkNNDist(knn_k=16)(a, cu(g["ori"]), weights=w, batch_avg=True); v.backward()
    np.testing.assert_allclose(npy(v), g["ChamferkNNDist_k16"], rtol=RTOL)
    assert rel_inf(npy(a.grad), g["ChamferkNNDist_k16_g"]) < RTOL


# ------------------------------------------------- a3: knn_utils.py against the reference
def assert_knn_idx(idx, ref_idx, dists, matrix):
    """Same contract as tests/test_oracle_golden.py: bit-identical distances at every rank;
    where indices differ it is an exact tie and ours are the lowest tied indices."""
    ref_d = np.take_along_axis(matrix, ref_idx.astype(np.int64), axis=2)
    assert np.array_equal(ref_d, dists)
    diff = idx != ref_idx
    assert diff.mean() < 0.01
    for b, r, c in np.argwhere(diff):
        tied = dists[b, r] == dists[b, r, c]
        lo = np.flatnonzero(matrix[b, r] == dists[b, r, c])
        assert sorted(idx[b, r][tied]) == sorted(lo[:tied.sum()])


def test_a3_knn_points_vs_reference():
    g = load_golden("a3_knn_utils")
    KU = pcd.knn_utils
    for tag, p1, p2, K in (("cross1", g["adv"], g["ori"], 1), ("self17", g["adv"], g["adv"], 17),
                           ("cross4", g["ori"], g["adv"], 4)):
        same = p1 is p2
        a = cu(p1, True); b = a if same else cu(p2, True)
        r = KU.knn_points(a, b, K=K, return_nn=True)
        assert r.idx.dtype == torch.int64 and tuple(r.dists.shape) == g[tag + "_dists"].shape
        (r.dists * cu(g[tag + "_gw"])).sum().backward()
        assert np.array_equal(npy(r.dists), g[tag + "_dists"]), tag
        od, oi = O.knn_points(p1, p2, K)
        assert np.array_equal(npy(r.idx), oi), tag                      # lowest-index contract
        assert_knn_idx(npy(r.idx), g[tag + "_idx"], npy(r.dists), O.knn_points_matrix(p1, p2))
        assert np.array_equal(npy(r.knn), O.knn_gather(p2, oi))
        # gradients: closed form (float64) through OUR indices everywhere ...
        og1, og2 = O.knn_points_grads(p1, p2, oi, g[tag + "_gw"])
        ours1 = npy(a.grad); ref1 = g[tag + "_g1"]
        assert rel_inf(ours1, og1 + og2 if same else og1) < RTOL, tag
        # ... and the reference's autograd wherever its (arbitrary) tie choice did not differ
        touched = np.zeros(p1.shape[:2], bool)
        for bb, rr, cc in np.argwhere(npy(r.idx) != g[tag + "_idx"]):
            touched[bb, [rr, oi[bb, rr, cc], g[tag + "_idx"][bb, rr, cc]]] = True
        assert touched.mean() < 0.01
        assert rel_inf(ours1[~touched], ref1[~touched]) < RTOL, tag
        if not same:
            assert rel_inf(npy(b.grad), og2) < RTOL, tag
            assert rel_inf(npy(b.grad)[~touched], g[tag + "_g2"][~touched]) < RTOL, tag
    out = KU.knn_gather(cu(g["gather_x"]), torch.from_numpy(g["self17_idx"]).cuda())
    assert np.array_equal(npy(out), g["gather_out"])
    with pytest.raises(RuntimeError):
        KU.knn_points(cu(g["adv"][:, :100]), cu(g["ori"][:, :90]), K=1)
    with pytest.raises(ValueError):
        KU.knn_points(cu(g["adv"][:1]), cu(g["ori"]), K=1)


@pytest.mark.parametrize("K", [1, 2, 5, 17, 21, 32, 33, 64])
@pytest.mark.parametrize("form_key", ["col_row_mulsum", "row_col_mulsum"])
def test_knn_bit_exact_random(K, form_key):
    form, norm, oform, onorm = FORMS[form_key]
    rs = np.random.RandomState(K)
    rows = rs.randn(2, 333, 3).astype(np.float32); cols = rs.randn(2, 1100, 3).astype(np.float32)
    cols[:, 500:600] = cols[:, :100]            # duplicated candidates: exact ties
    d, i = F.knn(cu(rows), cu(cols), K, form=form, norm=norm)
    od, oi = O.knn(oform, rows, cols, O.norms(onorm, rows), O.norms(onorm, cols), K)
    assert np.array_equal(npy(d), od) and np.array_equal(npy(i), oi)


@pytest.mark.parametrize("case", ["random4096", "sorted_overflow", "duplicates", "ragged", "k64", "sum_first", "swap"])
def test_knn_collect_pipeline(case):
    """xyz k-NN through pre-pass + collect + final select (and its overflow hand-over to the
    warp-per-row kernel), bit-exact against the oracle."""
    rs = np.random.RandomState(len(case))
    form, norm, oform, onorm = FORMS["col_row_mulsum"]
    K, swap = 17, False
    rows = rs.rand(2, 2048, 3).astype(np.float32); cols = rows
    if case == "random4096":
        rows = cols = rs.randn(1, 4096, 3).astype(np.float32)
    elif case == "sorted_overflow":
        # points sorted along x: a row's neighbours share one or two chunks, the chunk-minima bound is loose
        # and the candidate lists overflow -> exercised fallback
        rows = cols = np.sort(rs.rand(2, 2048, 3).astype(np.float32), axis=1)
        rows = cols = np.ascontiguousarray(rows[:, np.argsort(rows[0, :, 0])])
    elif case == "duplicates":
        cols = rows.copy(); cols[:, 1024:] = cols[:, :1024]; cols[:, 100:140] = cols[:, 7:8]
    elif case == "ragged":
        rows = rs.rand(3, 700, 3).astype(np.float32); cols = rs.rand(3, 1500, 3).astype(np.float32)
    elif case == "k64":
        K = 64
    elif case == "sum_first":
        form, norm, oform, onorm = FORMS["sum_first_fma"]
    elif case == "swap":
        cols = (rows + 0.01 * rs.randn(*rows.shape)).astype(np.float32); swap = True
    d, i = F.knn(cu(rows), cu(cols), K, form=form, norm=norm, swap_norms=swap)
    nr, nc = O.norms(onorm, rows), O.norms(onorm, cols)
    if swap:
        nr, nc = nc, nr
    od, oi = O.knn(oform, rows, cols, nr, nc, K)
    assert np.array_equal(npy(i), oi) and np.array_equal(npy(d), od)


def test_knn_collect_matches_select_only():
    rs = np.random.RandomState(5)
    x = cu(rs.rand(4, 3000, 3).astype(np.float32))
    d1, i1 = F.knn(x, x, 20)
    try:
        F.force_knn_strategy(F.KNN_BOUND_SELECT)
        d2, i2 = F.knn(x, x, 20)
        F.force_knn_strategy(F.KNN_SELECT_ONLY)
        d3, i3 = F.knn(x, x, 20)
    finally:
        F.force_knn_strategy(F.KNN_AUTO)
    assert torch.equal(i1, i2) and torch.equal(d1, d2) and torch.equal(i1, i3) and torch.equal(d1, d3)


@pytest.mark.parametrize("C", [1, 2, 5, 64, 128])
def test_knn_feature_channels(C):
    rs = np.random.RandomState(C)
    x = rs.randn(2, 300, C).astype(np.float32)
    d, i = F.knn(cu(x), cu(x), 20)
    nrm = O.norms(O.NORM_MULSUM, x)
    od, oi = O.knn(O.FORM_COL_ROW, x, x, nrm, nrm, 20)
    assert np.array_equal(npy(d), od) and np.array_equal(npy(i), oi)


# ------------------------------------------------- a4: GeoA3 losses against the reference
def test_a4_geoa3_losses_vs_reference():
    g = load_golden("a4_geoa3_losses")
    LU = pcd.loss_utils
    for fn in ("chamfer_loss", "pseudo_chamfer_loss", "hausdorff_loss"):
        a = cu(g["adv"], True)
        v = getattr(LU, fn)(a, cu(g["ori"])); (v * cu(g["gB"])).sum().backward()
        np.testing.assert_allclose(npy(v), g[fn], rtol=RTOL)
        assert rel_inf(npy(a.grad), g[fn + "_g"]) < RTOL, fn
    # float64 closed forms on the oracle's bit-exact neighbour indices pin the 1e-5 bar; the reference's own fp32 distance
    # from them is measured and printed beside ours
    pm = O._cf_to_pm(g["adv"])
    idx17 = O.self_knn_idx(g["adv"], 17)
    d17, _ = O.knn_points(pm, pm, 17)
    nidx = O.knn_points(pm, O._cf_to_pm(g["ori"]), 1)[1][:, :, 0]
    a = cu(g["adv"], True)
    v = LU.kNN_smoothing_loss(a, 16); (v * cu(g["gB"])).sum().backward()
    np.testing.assert_allclose(npy(v), g["kNN_smoothing_loss"], rtol=RTOL)
    l64, mask64, g64 = F64.knn_outlier_loss_grad64(pm, d17, idx17, 1.05, g["gB"])
    np.testing.assert_allclose(npy(v), l64, rtol=RTOL)
    assert rel_inf(npy(a.grad).transpose(0, 2, 1), g64) < RTOL
    assert rel_inf(npy(a.grad), g["kNN_smoothing_loss_g"]) < RTOL + rel_inf(g["kNN_smoothing_loss_g"].transpose(0, 2, 1), g64)
    ori_kappa = LU._get_kappa_ori(cu(g["ori"]), cu(g["normal"]), 16)
    np.testing.assert_allclose(npy(ori_kappa), g["ori_kappa"], rtol=RTOL, atol=3e-7)
    a = cu(g["adv"], True)
    adv_kappa, normal_curr = LU._get_kappa_adv(a, cu(g["ori"]), cu(g["normal"]), 16)
    assert np.array_equal(npy(normal_curr), g["normal_curr"])
    np.testing.assert_allclose(npy(adv_kappa), g["adv_kappa"], rtol=RTOL, atol=3e-7)
    v = LU.curvature_loss(a, cu(g["ori"]), adv_kappa, ori_kappa); (v * cu(g["gB"])).sum().backward()
    v64, kap64, gc64 = F64.curvature_loss_grad64(g["adv"], g["normal"], g["ori_kappa"], idx17, nidx, g["gB"])
    np.testing.assert_allclose(npy(adv_kappa), kap64, rtol=RTOL, atol=3e-7)
    np.testing.assert_allclose(npy(v), v64, rtol=RTOL)
    np.testing.assert_allclose(npy(v), g["curvature_loss"], rtol=RTOL)
    ref_err = rel_inf(g["curvature_loss_g"], gc64)
    print(f"a4 curvature gradient: reference fp32 autograd vs float64 {ref_err:.1e}; ours {rel_inf(npy(a.grad), gc64):.1e}")
    assert rel_inf(npy(a.grad), gc64) < RTOL
    assert rel_inf(npy(a.grad), g["curvature_loss_g"]) < RTOL + ref_err


# ------------------------------------------------- a6 / a7 against the reference
def test_a6_knn_graph_vs_reference():
    g = load_golden("a6_knn_graph")
    x3 = cu(g["x3"])
    pm = O._cf_to_pm(g["x3"]); nrm = O.norms(O.NORM_MULSUM, pm)
    mat = -O.dgcnn_neg_matrix(g["x3"])
    d20, i20 = O.knn(O.FORM_COL_ROW, pm, pm, nrm, nrm, 20)
    d21, i21 = O.knn(O.FORM_COL_ROW, pm, pm, nrm, nrm, 21)
    ours = pcd.dgcnn.knn(x3, 20)
    assert ours.dtype == torch.int64 and np.array_equal(npy(ours), i20)
    assert_knn_idx(npy(ours), g["dgcnn_k20"], d20, mat)
    assert np.array_equal(npy(pcd.curvenet_util.knn(x3, 20)), i21)
    assert_knn_idx(npy(pcd.curvenet_util.knn(x3, 20)), g["curvenet_k20"], d21, mat)
    assert np.array_equal(npy(pcd.curvenet_util.normal_knn(x3, 20)), i20)
    f64 = cu(g["f64"])
    assert np.array_equal(npy(pcd.dgcnn.knn(f64, 20)), O.dgcnn_knn(g["f64"], 20))
    assert_knn_near_tie_proof(npy(pcd.dgcnn.knn(f64, 20)), g["dgcnn_f64_k20"], g["f64"], "gaussian C=64")
    # get_graph_feature: gather + concat, compared with a direct numpy restatement
    feat = npy(pcd.dgcnn.get_graph_feature(x3, k=20))
    xt = g["x3"].transpose(0, 2, 1)
    nb = xt[np.arange(2)[:, None, None], i20]
    ref = np.concatenate([nb - xt[:, :, None, :], np.broadcast_to(xt[:, :, None, :], nb.shape)], -1).transpose(0, 3, 1, 2)
    assert np.array_equal(feat, ref)


def test_a6_knn_graph_feature_layers_vs_reference():
    """The four knn() calls of the reference DGCNN forward (C = 3, 64, 64, 128): the kernel is bit-identical to the
    oracle's sequential chain; against the reference's own indices (CPU BLAS order, committed golden) and against
    the reference formulation run HERE on the GPU (cuBLAS order -- what a user of the reference actually gets)
    every difference is a provable near tie (tests/knn_proof.py), no agreement fraction is assumed."""
    g = load_golden("a6_knn_graph_features")
    torch.backends.cuda.matmul.allow_tf32 = False
    for li, C in enumerate((3, 64, 64, 128)):
        x = g[f"x{li}"]
        ours = npy(pcd.dgcnn.knn(cu(x), 20))
        assert np.array_equal(ours, O.dgcnn_knn(x, 20)), f"layer {li}"
        st_cpu = assert_knn_near_tie_proof(ours, g[f"idx{li}"].astype(np.int64), x, f"layer {li} vs reference CPU")
        xt = cu(x)                                            # model/dgcnn.py:194-200 verbatim arithmetic, on the GPU
        inner = -2 * torch.matmul(xt.transpose(2, 1), xt)
        xx = torch.sum(xt ** 2, dim=1, keepdim=True)
        ref_gpu = npy((-xx - inner - xx.transpose(2, 1)).topk(k=20, dim=-1)[1])
        st_gpu = assert_knn_near_tie_proof(ours, ref_gpu, x, f"layer {li} vs reference formulation on GPU")
        print(f"a6 layer {li} C={C}: vs reference CPU {st_cpu}; vs reference-on-GPU {st_gpu}")


def test_a7_pointnet2_utils_vs_reference():
    g = load_golden("a7_pointnet2_utils")
    P2 = pcd.pointnet2_utils
    xyz, new_xyz = cu(g["xyz"]), cu(g["new_xyz"])
    q = P2.query_ball_point(0.2, 32, xyz, new_xyz)
    assert q.dtype == torch.int64 and np.array_equal(npy(q), g["ball_r02_n32"])
    assert np.array_equal(npy(P2.query_ball_point(0.4, 64, xyz[:, :512], new_xyz[:, :128])), g["ball_r04_n64"])
    assert np.array_equal(npy(P2.query_ball_point(0.02, 8, xyz, new_xyz[:, :64])), g["ball_r002_n8"])
    # radius so small that rows without any hit exist -> filled with N
    far = new_xyz[:, :16] + 10.0
    assert np.array_equal(npy(P2.query_ball_point(0.01, 4, xyz, far)), O.query_ball_point(0.01, 4, g["xyz"], npy(far)))
    np.testing.assert_allclose(npy(P2.square_distance(new_xyz[:, :64], xyz[:, :96])), g["sqdist_block"], atol=1e-6)


# ------------------------------------------------- f-4: local geometry on the k-NN graph (round 2)
def test_f4_estimate_normal_and_frames():
    g = load_golden("f4_local_geometry")
    adv = g["adv"]; pm = O._cf_to_pm(adv)
    U = pcd.utility
    for k in (3, 8, 16):
        idx = O.self_knn_idx(adv, k + 1)
        w, v, nsum = O.local_frames(pm, idx)
        ours = npy(U.estimate_normal(cu(adv), k)).transpose(0, 2, 1)                      # [b,n,3]
        nrm, evecs, evals = F.local_frames(cu(pm), cu(idx.astype(np.int32)), frames=True)
        assert np.array_equal(npy(nrm), ours)
        gap = (w[..., 1] - w[..., 0]) / np.maximum(w[..., 2], 1e-30)
        well = gap > 1e-3
        unit = np.linalg.norm(ours, axis=-1) > 0.5
        assert unit.mean() > 0.95 and np.abs(np.linalg.norm(ours[unit], axis=-1) - 1).max() < 1e-6
        # fp64 Jacobi on the fp32 covariance vs numpy's fp64 eigh of the same matrix: the frames agree to fp32 output rounding
        cos = np.abs((npy(evecs)[:, :, 0, :] * v[:, :, 0, :]).sum(-1))
        assert cos[well].min() > 1 - 1e-6
        np.testing.assert_allclose(npy(evals), w, rtol=1e-4, atol=1e-9 * float(w.max()) + 1e-12)
        # sign rule: -sign(<n, sum of centred neighbours>) with the fp32 neighbour sum
        d = (npy(evecs)[:, :, 0, :].astype(np.float64) * nsum).sum(-1)
        sure = unit & (np.abs(d) > 1e-9)
        assert (np.sign((ours[sure] * npy(evecs)[:, :, 0, :][sure]).sum(-1)) == -np.sign(d[sure])).all()
        # against the reference itself (sign-free: the reference's sign is rounding noise, utility.py:67-69)
        nref = g[f"normal_k{k}"].transpose(0, 2, 1)
        both = unit & (np.linalg.norm(nref, axis=-1) > 0.5)
        assert np.abs((ours * nref).sum(-1))[both].min() > 1 - 1e-5
    # the tangent-plane jitter uses the two other eigenvectors: orthogonal to the normal, bounded by the clip
    torch.manual_seed(0)
    jit = npy(U.estimate_perpendicular(cu(adv), 8, sigma=0.01, clip=0.05)).transpose(0, 2, 1)
    n8 = npy(U.estimate_normal(cu(adv), 8)).transpose(0, 2, 1)
    assert np.abs(jit).max() <= 0.1 + 1e-6
    small = np.abs(jit).max(-1) < 0.04                                             # unclipped draws stay in the tangent plane
    assert np.abs((jit * n8).sum(-1))[small & (np.linalg.norm(n8, axis=-1) > 0.5)].max() < 1e-5


def test_f4_kappa_and_knn_losses_vs_reference():
    g = load_golden("f4_local_geometry")
    LU = pcd.loss_utils
    adv, ori, gN = g["adv"], g["ori"], g["gN"]
    pm = O._cf_to_pm(adv)
    nrm = g["normal_k8"]
    # kappa: fp32 op-order oracle bit for bit, reference value to rounding, gradient against the fp64 closed form
    a = cu(adv, True)
    kap, normal = LU._get_kappa_adv(a, cu(ori), cu(nrm), 16)
    (kap * cu(gN)).sum().backward()
    nidx = O.knn_points(pm, O._cf_to_pm(ori), 1)[1][:, :, 0]
    idx = O.self_knn_idx(adv, 17)
    ok = O.kappa(pm, nrm.transpose(0, 2, 1), idx, nidx=nidx)
    assert np.abs(npy(kap) - ok).max() <= 6e-8 and (npy(kap) == ok).mean() > 0.9       # division / sqrt are correctly rounded on both sides
    np.testing.assert_allclose(npy(kap), g["kappa_adv_k16"], rtol=0, atol=3e-7)
    g64 = O.kappa_grad64(pm, nrm.transpose(0, 2, 1), idx, gN, nidx=nidx)
    assert rel_inf(npy(a.grad).transpose(0, 2, 1), g64) < RTOL
    assert rel_inf(npy(a.grad), g["kappa_adv_k16_g"]) < RTOL
    assert np.array_equal(npy(normal), np.take_along_axis(nrm, nidx[:, None, :].repeat(3, 1), 2))
    for name, fn in (("displacement_loss", lambda x: LU.displacement_loss(x, cu(ori), k=16)),
                     ("corresponding_normal_loss", lambda x: LU.corresponding_normal_loss(x, cu(nrm), k=2)),
                     ("repulsion_loss", lambda x: LU.repulsion_loss(x, k=4, h=0.03)),
                     ("distance_kmean_loss", lambda x: LU.distance_kmean_loss(x, 8))):
        a = cu(adv, True)
        v = fn(a)
        (v * cu(gN)).sum().backward()
        # every neighbour set matches the brute-force topk on this fixture (self is dropped by index, not by rank)
        rel = np.abs(npy(v) - g[name]) / (np.abs(g[name]).max() + 1e-30)
        assert (rel < RTOL).all(), (name, float((rel < RTOL).mean()))
        assert rel_inf(npy(a.grad), g[name + "_g"]) < RTOL, name


def test_f4_graph_laplacian_vs_reference():
    g = load_golden("f4_local_geometry")
    small = g["lap_pc"]
    L = npy(pcd.taof.laplacian_from_pc(cu(small), 30))
    Lo = O.graph_laplacian(O._cf_to_pm(small), O.dgcnn_knn(small, 30))
    assert ((L != 0) == (Lo != 0)).all() and ((L != 0) == (g["lap_L"] != 0)).all()
    np.testing.assert_allclose(L, Lo, rtol=3e-7, atol=2e-6)                  # expf vs numpy exp: ulps; diagonal = a sum of ~30 terms
    np.testing.assert_allclose(L, g["lap_L"], rtol=1e-6, atol=1e-5)
    assert np.abs(L.sum(2)).max() < 1e-4                                     # rows of a Laplacian sum to zero
    e, v = pcd.taof.get_Laplace_from_pc(cu(small))
    # the dense eigensolver is torch's (cuSOLVER here, LAPACK in the golden run; not part of the path): fp32 eigh agrees to ~1e-4
    np.testing.assert_allclose(npy(e), g["lap_e"], rtol=3e-4, atol=1e-4)


def test_launch_counts_of_the_fused_chains():
    """Device-side launch counts (torch profiler, kernels + memsets issued by this library): the Chamfer+Hausdorff forward is
    three kernels and its backward one; KNNDist forward + backward is at most eight (k-NN select pipeline, ONE epilogue, ONE backward)."""
    from torch.profiler import ProfilerActivity, profile
    g = load_golden("a2_distance_face")
    p, t = cu(g["preds"], True), cu(g["gts"])

    def count(fn):
        fn(); torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn(); torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        ours = [n for n in names if "pcd::" in n]
        return ours, [n for n in names if "Memset" in n or "memset" in n]

    def cd_hd():
        p.grad = None
        c1, c2 = pcd.distance.chamfer(p, t); h1, h2 = pcd.distance.hausdorff(p, t)
        (c1.sum() + c2.sum() + h1.sum() + h2.sum()).backward()
    ours, memsets = count(cd_hd)
    assert len(ours) == 4 and not memsets, (ours, memsets)           # arm, sweep, fix-up | backward
    pc = cu(g["preds"], True)

    def knn_loss():
        pc.grad = None
        pcd.dist_utils.KNNDist(k=16, alpha=1.05)(pc, batch_avg=False).sum().backward()
    ours, memsets = count(knn_loss)
    assert len(ours) + len(memsets) <= 8, (ours, memsets)


# ------------------------------------------------- robustness of the NN-1 chain (ADVICE r1)
@pytest.mark.parametrize("n", [1024, 1022])          # 1024: streamed raw, 1022: packed through the workspace
def test_nn1_nan_and_inf_points_do_not_fault(n):
    """A NaN / inf coordinate (a diverged adversarial cloud) must not fault: the untouched column key
    used to decode to a negative row index (pcd_nn1.cu fix-up).  Finite points keep exact results."""
    rs = np.random.RandomState(11)
    rows = rs.randn(3, n, 3).astype(np.float32); cols = rs.randn(3, n, 3).astype(np.float32)
    rows[0, 5] = np.nan; cols[0, 7, 1] = np.inf; cols[1, :, :] = np.nan; rows[2, :, 0] = np.inf
    for form_key in FORMS:
        form, norm, oform, onorm = FORMS[form_key]
        r = F.nn1(cu(rows), cu(cols), form, norm, cache=False)
        torch.cuda.synchronize()
        ra, ca = npy(r.row_arg), npy(r.col_arg)
        assert ra.min() >= 0 and ra.max() < n and ca.min() >= 0 and ca.max() < n
        # sample 0: rows other than the NaN one against the finite columns are exact
        ok_r = np.ones(n, bool); ok_r[5] = False
        ok_c = np.ones(n, bool); ok_c[7] = False
        o = oracle_nn1(rows[:1, ok_r], cols[:1, ok_c], oform, onorm)
        assert np.array_equal(npy(r.row_min)[0, ok_r], o.row_min[0])
        assert np.array_equal(npy(r.col_min)[0, ok_c], o.col_min[0])
        # sample 1: every distance NaN -> no finite minimum anywhere: arg 0, value NaN or +inf
        assert not np.isfinite(npy(r.row_min)[1]).any() and not np.isfinite(npy(r.col_min)[1]).any()
        assert (ra[1] == 0).all() and (ca[1] == 0).all()


@pytest.mark.parametrize("B,N,M,kind", [(3, 1024, 1024, "perturbed"), (2, 4096, 2048, "random"), (2, 512, 1500 // 4 * 4, "duplicates"),
                                         (1, 2048, 2048, "identical"), (4, 260, 36, "tiny"), (2, 216, 512, "lattice")])
def test_nn1_near_ties_and_duplicates_against_oracle(B, N, M, kind):
    """Minima and lowest-index arg-mins bit-equal to the oracle for every form on the hardest near-tie inputs: perturbed
    clouds (many close second-best candidates), unrelated clouds, clouds full of exact duplicates (every point has a tie),
    all-identical clouds, tiny clouds, and a shuffled lattice whose distances are exact ties (every point has several
    equidistant nearest neighbours, so only the lowest-index rule decides)."""
    rs = np.random.RandomState(B * N + M)
    cols = rs.randn(B, M, 3).astype(np.float32)
    if kind == "perturbed":
        rows = (cols[:, :N] + 0.01 * rs.randn(B, N, 3)).astype(np.float32)
    elif kind == "duplicates":
        rows = cols[:, rs.randint(0, M, size=N)].copy()
        cols[:, M // 2:] = cols[:, :M - M // 2]                      # every column exists twice
    elif kind == "identical":
        rows = np.tile(cols[:, :1], (1, N, 1)); cols = np.tile(cols[:, :1], (1, M, 1))
    elif kind == "lattice":
        # columns on an 8^3 grid of step 1/4, rows at the centres of 6^3 of its cells: every coordinate, norm and distance is
        # exact in fp32, so each row has 8 equidistant nearest columns and each inner column 8 equidistant nearest rows
        g = lambda idx: np.stack(np.meshgrid(idx, idx, idx, indexing="ij"), -1).reshape(-1, 3).astype(np.float32) * 0.25
        grid_c, grid_r = g(np.arange(8) - 3.5), g(np.arange(1, 7) - 3.0)
        assert grid_c.shape[0] == M and grid_r.shape[0] == N
        cols = np.stack([grid_c[rs.permutation(M)] for _ in range(B)])
        rows = np.stack([grid_r[rs.permutation(N)] for _ in range(B)])
    else:
        rows = rs.randn(B, N, 3).astype(np.float32)
    for form_key in FORMS:
        form, norm, oform, onorm = FORMS[form_key]
        r = F.nn1(cu(rows), cu(cols), form, norm, cache=False)
        o = oracle_nn1(rows, cols, oform, onorm)
        assert np.array_equal(npy(r.row_min), o.row_min) and np.array_equal(npy(r.row_arg), o.row_arg)
        assert np.array_equal(npy(r.col_min), o.col_min) and np.array_equal(npy(r.col_arg), o.col_arg)


def test_nn1_raw_and_packed_paths_agree():
    """The same clouds through the dense (streamed) and the strided (packed) path: identical outputs and gradients."""
    rs = np.random.RandomState(12)
    rows = rs.randn(4, 1200, 3).astype(np.float32); cols = (rows[:, :1000] + 0.02 * rs.randn(4, 1000, 3)).astype(np.float32)
    wide_r = torch.zeros(4, 1200, 5, device="cuda"); wide_r[:, :, 1:4] = cu(rows)
    wide_c = torch.zeros(4, 1000, 4, device="cuda"); wide_c[:, :, :3] = cu(cols)
    outs = []
    for tr, tc in ((cu(rows), cu(cols)), (wide_r[:, :, 1:4], wide_c[:, :, :3]),
                   (cu(rows.transpose(0, 2, 1)).transpose(1, 2), cu(cols.transpose(0, 2, 1)).transpose(1, 2))):
        tr = tr.detach().requires_grad_(True); tc = tc.detach().requires_grad_(True)
        r = F.nn1(tr, tc, F.FORM_ROW_COL, F.NORM_MULSUM, transform=F.VALUE_SQRT_CLAMP, cache=False)
        (r.row_sum.sum() + 2 * r.col_max.sum() + (r.col_min * r.col_min).sum()).backward()
        outs.append([npy(x) for x in (r.row_min, r.row_arg, r.col_min, r.col_arg, r.row_sum, r.col_max, r.col_argmax, tr.grad, tc.grad)])
    for other in outs[1:]:
        for k, (a, b) in enumerate(zip(outs[0][:7], other[:7])):
            if k == 4:
                np.testing.assert_allclose(a, b, rtol=2e-6)      # per-sample sums: the paths fold in different (fixed) orders
            else:
                assert np.array_equal(a, b)
        for a, b in zip(outs[0][7:], other[7:]):
            assert rel_inf(a, b) < 2e-6          # atomics: summation order only


def test_nn1_prezeroed_backward_and_retain_graph():
    """The forward clears the gradient buffers of the first backward; a second backward through a
    retained graph must allocate afresh and give the same gradient (not an accumulated one)."""
    g = load_golden("a2_distance_ragged")
    a = cu(g["preds"], grad=True); o = cu(g["gts"])
    c1, c2 = pcd.distance.chamfer(a, o)
    loss = c1.sum() + c2.sum()
    g1, = torch.autograd.grad(loss, a, retain_graph=True)
    g1 = g1.clone()
    g2, = torch.autograd.grad(loss, a)
    assert rel_inf(npy(g2), npy(g1)) < 2e-6
    w = np.ones(g["preds"].shape[0], np.float32)
    ref, _ = O.chamfer_distance_grads(g["preds"], g["gts"], w, w)
    assert rel_inf(npy(g1), ref) < RTOL


def test_nn1_cache_is_not_served_under_no_grad_after_data_mutation():
    """ADVICE r1: x.data.add_() does not bump x._version; a no_grad result must never come from the cache."""
    g = load_golden("a2_distance_ragged")
    a = cu(g["preds"], grad=True); o = cu(g["gts"])
    with torch.no_grad():
        c_before = npy(pcd.distance.chamfer(a, o)[0]).copy()
        a.data.add_(0.05)
        c_after = npy(pcd.distance.chamfer(a, o)[0])
    assert not np.array_equal(c_before, c_after)
    ref = O.chamfer_distance(g["preds"] + np.float32(0.05), g["gts"])[0]
    np.testing.assert_allclose(c_after, ref, rtol=RTOL)
    # with a graph being recorded the second call of the same forward IS served by the cache (one sweep) ...
    n0 = F.launches()
    pcd.distance.chamfer(a, o); pcd.distance.hausdorff(a, o)
    assert F.launches() - n0 == 3
    # ... and after an in-place clip the documented clear_cache() makes the next call recompute
    a.data.sub_(0.05); F.clear_cache()
    np.testing.assert_allclose(npy(pcd.distance.chamfer(a, o)[0]), O.chamfer_distance(npy(a), g["gts"])[0], rtol=RTOL)


# ------------------------------------------------- error behaviour
def test_errors_are_loud():
    with pytest.raises(RuntimeError):
        F.nn1(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3), F.FORM_SUM_FIRST, F.NORM_FMA)     # CPU tensors
    with pytest.raises(ValueError):
        F.nn1(torch.zeros(1, 4, 3, device="cuda"), torch.zeros(2, 4, 3, device="cuda"), 0, 0)
    with pytest.raises(TypeError):
        F.nn1(torch.zeros(1, 4, 3, device="cuda", dtype=torch.float64), torch.zeros(1, 4, 3, device="cuda"), 0, 0)
    with pytest.raises(ValueError):
        F.knn(torch.zeros(1, 4, 3, device="cuda"), torch.zeros(1, 4, 3, device="cuda"), 5)       # K > M
    lib = pcd._lib.load()
    assert lib.pcd_nn1_forward(None, 0, 0, 0, None, 0, 0, 0, 1, 1, 1, 0, 0, 0, 0, 1.0, 1.0,
                               None, None, None, None, None, None, None, 0, None, 0, None, 0, 0, 0, 0,
                               None, None, None) == 1
    assert b"NULL" in lib.pcd_last_error()


# ------------------------------------------------- section 8f-1: device-resident CW loop
def test_cw_loop_eager_and_graph_agree():
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import victims
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    torch.manual_seed(0)
    model = victims.PointNetVictim(16).cuda().eval()
    data = synth.face_clouds(4, 512, seed=11).cuda()
    target = torch.tensor([0, 1, 2, 3], device="cuda")
    cd = pcd.dist_utils.ChamferDist(method="avg"); hd = pcd.dist_utils.HausdorffDist(method="avg")
    dist = lambda a, o, w, batch_avg=False: cd(a, o, weights=w, batch_avg=batch_avg) + hd(a, o, weights=w, batch_avg=batch_avg)
    res = {}
    for use_graph in (False, True):
        atk = pcd.cw_loop.CWAttack(model, pcd.cw_loop.UntargetedLogitsAdvLoss(kappa=5.), dist, attack_lr=1e-2,
                                   binary_step=2, num_iter=12, clip_func=pcd.cw_loop.ClipPointsLinf(0.18), use_graph=use_graph)
        best, adv, ok = atk.attack(data, target, seed=3)
        assert adv.shape == (4, 512, 3) and best.shape == (4,) and ok.dtype == torch.bool
        assert torch.isfinite(adv).all()
        assert float((adv - data).norm(dim=-1).max()) <= 0.18 + 1e-5          # projection respected
        res[use_graph] = adv
    assert torch.allclose(res[False], res[True], atol=1e-4)                      # atomics reorder sums only


# ------------------------------------------------------------- f-2 / f-3 (SURVEY 8f rows 2-3)
def test_f_get_graph_feature_vs_reference():
    g = load_golden("f_graph_sampling")
    x = cu(g["adv_cf"], True)
    f = pcd.dgcnn.get_graph_feature(x, k=20)
    assert f.shape == g["ggf3"].shape and np.array_equal(npy(f), g["ggf3"])       # bit-exact incl. the kNN
    (f * cu(g["ggf3_gw"])).sum().backward()
    assert rel_inf(g["ggf3_gx"], npy(x.grad)) < RTOL
    x = cu(g["f16"], True)
    f = pcd.dgcnn.get_graph_feature(x, k=10, idx=cu(g["ggf16_idx"]))
    assert np.array_equal(npy(f), g["ggf16"])
    (f * cu(g["ggf16_gw"])).sum().backward()
    assert rel_inf(g["ggf16_gx"], npy(x.grad)) < RTOL
    # odd k: scalar (non-float4) path
    f = pcd.dgcnn.get_graph_feature(cu(g["f16"]), k=7, idx=cu(g["idx7"]))
    assert np.array_equal(npy(f), g["ggf16_idx7"])
    with pytest.raises(RuntimeError):
        pcd.dgcnn.get_graph_feature(cu(g["f16"]), k=5, idx=cu(g["idx7"]))


def test_f_lpfa_group_feature_vs_reference():
    g = load_golden("f_graph_sampling")
    xyz = cu(g["adv_cf"], True)
    idx = pcd.curvenet_util.knn(xyz, 20)[:, :, :20]
    assert np.array_equal(npy(idx), g["lpfa9_idx"])
    pf = pcd.curvenet_util.lpfa_point_feature(xyz, idx)
    assert np.array_equal(npy(pf), g["lpfa9"])
    (pf * cu(g["lpfa9_gw"])).sum().backward()
    assert rel_inf(g["lpfa9_gx"], npy(xyz.grad)) < RTOL


@pytest.mark.parametrize("gather", [True, False])
@pytest.mark.parametrize("B,C,N,k,ops", [(3, 64, 500, 20, (2, 0)), (2, 5, 1000, 9, (0, 1, 2)), (1, 128, 2048, 20, (2,)),
                                         (2, 3, 4096, 32, (1, 2, 0, 2)), (2, 1, 33, 4, (2, 0)), (2, 4, 777, 12, (1,)),
                                         (1, 2, 4100, 8, (2, 0)), (2, 3, 300, 5, (2, 0)), (1, 2, 64, 128, (0, 2, 1))])
def test_f_edge_feature_random(B, C, N, k, ops, gather):
    """Forward bit-exact, backward to RTOL against the oracle, through both backward forms (gather over the inverted
    graph / shared-memory atomics); shapes cover ragged last chunks, N > 4096 and 4 !| N*k (atomics only), 1..4 blocks."""
    rs = np.random.RandomState(B * 1000 + C)
    x = rs.randn(B, C, N).astype(np.float32)
    idx = rs.randint(0, N, size=(B, N, k))
    xt = cu(x, True)
    prev = F.deterministic_edge_backward(gather)
    try:
        out = F.edge_feature(xt, cu(idx), ops)
        assert np.array_equal(npy(out), O.edge_feature(x, idx, ops))
        gw = rs.randn(*out.shape).astype(np.float32)
        (out * cu(gw)).sum().backward()
    finally:
        F.deterministic_edge_backward(prev)
    assert rel_inf(O.edge_feature_grad(gw, idx, ops, C), npy(xt.grad)) < RTOL


def test_f_edge_feature_backward_gather_is_reproducible_and_handles_hubs():
    """The gather backward has a fixed summation order: two runs are bit-identical (the atomics form is not), also on a
    graph where every point names the same few neighbours (in-degree N: the per-target lists are as long as a chunk)
    and with out-of-range indices (clamped, as in the forward)."""
    rs = np.random.RandomState(5)
    B, C, N, k = 2, 6, 1500, 20
    lib = importlib.import_module("3dpointcloudattack_b200._lib").load()
    assert lib.pcd_edge_feature_backward_workspace(B, N, k, 2) > 0
    assert lib.pcd_edge_feature_backward_workspace(B, 5000, k, 2) == 0          # N > 4096: atomics form only
    assert lib.pcd_edge_feature_backward_workspace(B, 33, 5, 2) == 0            # 4 does not divide N*k
    x = rs.randn(B, C, N).astype(np.float32)
    hub = np.tile(np.arange(k)[None, None, :], (B, N, 1))                       # every row -> points 0..k-1
    hub[1, :, 0] = 7                                                            # one column of sample 1 -> a single point
    wild = rs.randint(-50, N + 50, size=(B, N, k))
    prev = F.deterministic_edge_backward(True)
    try:
        for idx in (rs.randint(0, N, size=(B, N, k)), hub, wild):
            grads = []
            for _ in range(2):
                xt = cu(x, True)
                out = F.edge_feature(xt, cu(idx), (2, 0))
                gw = np.random.RandomState(9).randn(*out.shape).astype(np.float32)
                (out * cu(gw)).sum().backward()
                grads.append(npy(xt.grad))
            assert np.array_equal(grads[0], grads[1])
            assert rel_inf(O.edge_feature_grad(gw, np.clip(idx, 0, N - 1), (2, 0), C), grads[0]) < RTOL
    finally:
        F.deterministic_edge_backward(prev)


# ------------------------------------------------------------- f-1: fused clip / projection epilogues
def _torch_clip_chains(adv, ori, normal, budget, cc):
    """the reference's op chains (clip_utils.py:22-29, :50-56, :78-109; GeoA3_attack.py:92-101) on whatever device the
    tensors are on, with dim=1 spelled out for torch.cross"""
    d = adv - ori
    linf = ori + d * torch.clamp(budget / (torch.sum(d ** 2, dim=1) ** 0.5 + 1e-9), max=1.)[:, None, :]
    l2 = ori + d * torch.clamp(budget / (torch.sum(d ** 2, dim=[1, 2]) ** 0.5 + 1e-9), max=1.)[:, None, None]
    inner = torch.sum(d * normal, dim=1) < 0.
    vng = torch.cross(normal, d, dim=1)
    vref = torch.cross(vng, normal, dim=1)
    proj = d * vref / (torch.sum(vref ** 2, dim=1) ** 0.5 + 1e-9)[:, None, :]
    proj = torch.where((inner & (torch.sum(vng ** 2, dim=1) ** 0.5 < 1e-6))[:, None, :], torch.zeros_like(proj), proj)
    p1 = ori + torch.where(inner[:, None, :], proj, d)
    d1 = p1 - ori
    project_linf = ori + d1 * torch.clamp(budget / (torch.sum(d1 ** 2, dim=1) ** 0.5 + 1e-9), max=1.)[:, None, :]
    ln = (d ** 2).sum(1, keepdim=True).sqrt()
    lp = torch.where(ln < cc, d, torch.where(ln > 1e-6, d / ln.expand_as(d) * cc, torch.zeros_like(d)))
    return linf, l2, project_linf, lp


def test_f1_clip_epilogues_vs_oracle_torch_and_reference():
    """One-launch clip / projection epilogues: bit-identical to the oracle (which is pinned on the reference's CPU outputs
    in tests/test_oracle_golden.py); against the reference's golden to 2 ulp of the largest coordinate; against the same
    torch chain run on THIS GPU bit-identical for the per-point clips (ClipPointsLinf, lp_clip, find_offset)."""
    g = load_golden("f1_clips")
    ori, adv, normal = g["ori"], g["adv"], g["normal"]
    off = adv - ori
    eps2 = 2 * np.finfo(np.float32).eps

    def close(ours, ref):
        return np.abs(ours - ref).max() <= eps2 * np.abs(ref).max()

    ours = {
        "linf": npy(F.clip_points_(cu(adv), cu(ori), 0.03, F.CLIP_LINF)),
        "l2": npy(F.clip_points_(cu(adv), cu(ori), 0.5, F.CLIP_L2)),
        "project_linf": npy(F.clip_points_(cu(adv), cu(ori), 0.03, F.CLIP_PROJECT_LINF, normal=cu(normal))),
        "lp_clip": npy(pcd.geoa3_loop.lp_clip(cu(off), 0.02)),
        "offset_proj": npy(pcd.geoa3_loop.offset_proj(cu(off), cu(ori), cu(normal))),
        "find_offset": npy(pcd.geoa3_loop.find_offset(cu(ori), cu(adv))),
    }
    assert np.array_equal(ours["linf"], O.clip_points_linf(adv, ori, 0.03))
    assert np.array_equal(ours["project_linf"], O.project_inner_clip_linf(adv, ori, normal, 0.03))
    assert close(ours["l2"], O.clip_points_l2(adv, ori, 0.5))                  # the 3K-term sum: order differs
    assert np.array_equal(ours["lp_clip"], O.lp_clip(off, 0.02))
    assert np.array_equal(ours["offset_proj"], O.offset_proj(off, ori, normal))
    assert np.array_equal(ours["find_offset"], O.find_offset(ori, adv))
    for k, v in ours.items():
        assert close(v, g[k]), k
    t_linf, t_l2, t_proj, t_lp = (npy(x) for x in _torch_clip_chains(cu(adv), cu(ori), cu(normal), 0.03, 0.02))
    assert np.array_equal(ours["linf"], t_linf) and np.array_equal(ours["lp_clip"], t_lp)
    assert close(ours["project_linf"], t_proj)                                  # torch.cross contracts its products into FMAs
    assert close(npy(F.clip_points_(cu(adv), cu(ori), 0.03, F.CLIP_L2)), npy(_torch_clip_chains(cu(adv), cu(ori), cu(normal), 0.03, 0.02)[1]))
    # the module-level wrappers the loops call are the same kernels, in place
    a = cu(adv)
    assert pcd.cw_loop.ClipPointsLinf(0.03)(a, cu(ori)) is a and np.array_equal(npy(a), ours["linf"])
    a = cu(adv)
    pcd.cw_loop.ProjectInnerClipLinf(0.03)(a, cu(ori), cu(normal))
    assert np.array_equal(npy(a), ours["project_linf"])
    a = cu(adv)
    pcd.cw_loop.ProjectInnerClipLinf(0.03)(a, cu(ori))                          # no normals: the clip alone
    assert np.array_equal(npy(a), ours["linf"])


@pytest.mark.parametrize("B,K", [(1, 1), (3, 257), (32, 1024), (2, 5000)])
def test_f1_clip_epilogues_random_and_degenerate(B, K):
    """Random clouds with NaN / inf / zero offsets planted: kernel == oracle bit for bit (NaN positions included)."""
    rs = np.random.RandomState(B * 7 + K)
    ori = rs.randn(B, 3, K).astype(np.float32)
    adv = (ori + 0.05 * rs.randn(B, 3, K)).astype(np.float32)
    normal = rs.randn(B, 3, K).astype(np.float32)
    if K > 8:
        adv[0, :, 1] = ori[0, :, 1]
        adv[0, 0, 2] = np.nan
        adv[0, 1, 3] = np.inf
        normal[0, :, 4] = 0.0
        adv[0, :, 5] = ori[0, :, 5] - 0.01 * normal[0, :, 5]
    off = adv - ori
    with np.errstate(all="ignore"):
        assert np.array_equal(npy(F.clip_points_(cu(adv), cu(ori), 0.04)), O.clip_points_linf(adv, ori, 0.04), equal_nan=True)
        assert np.array_equal(npy(F.clip_points_(cu(adv), cu(ori), 0.04, F.CLIP_PROJECT_LINF, normal=cu(normal))),
                              O.project_inner_clip_linf(adv, ori, normal, 0.04), equal_nan=True)
        assert np.array_equal(npy(F.lp_clip(cu(off), 0.03)), O.lp_clip(off, 0.03), equal_nan=True)
        idx = rs.randint(0, K, size=(B, K))
        assert np.array_equal(npy(F.offset_proj(cu(off), cu(normal), cu(idx))), O.offset_proj(off, ori, normal, idx), equal_nan=True)
        assert np.array_equal(npy(F.find_offset(cu(adv), cu(ori), cu(idx))), O.find_offset(ori, adv, idx), equal_nan=True)
        fin = np.isfinite(adv).all((1, 2))
        l2 = npy(F.clip_points_(cu(adv), cu(ori), 0.5, F.CLIP_L2))
        ref = O.clip_points_l2(adv, ori, 0.5)
        assert np.abs(l2[fin] - ref[fin]).max() <= 4 * np.finfo(np.float32).eps * np.abs(ref[fin]).max() if fin.any() else True


def test_smem_opt_in_is_per_kernel_instantiation():
    """Kernels that are instantiations of one template share their pointer TYPE; the >48 KB shared-memory opt-in has
    to be remembered per kernel ADDRESS.  Order that used to fail: the 128 KB instantiation first, then a 64 KB one."""
    rs = np.random.RandomState(3)
    big = rs.rand(1, 8000, 3).astype(np.float32)
    mid = rs.rand(1, 4000, 3).astype(np.float32)
    for xyz in (big, mid):
        start = np.zeros(1, np.int64)
        fps = F.farthest_point_sample(cu(xyz), 8, start=cu(start))
        assert np.array_equal(npy(fps), O.farthest_point_sample(xyz, 8, start))
    x = rs.randn(1, 2, 20000).astype(np.float32)                   # 80 KB of staged rows per channel
    for k in (4, 3):                                               # vectorised instantiation first, scalar one second
        idx = rs.randint(0, 20000, size=(1, 20000, k))
        assert np.array_equal(npy(F.edge_feature(cu(x), cu(idx), (2, 0))), O.edge_feature(x, idx, (2, 0)))


def test_f_farthest_point_sample_vs_reference():
    g = load_golden("f_graph_sampling")
    adv = cu(g["adv"])
    assert np.array_equal(npy(F.farthest_point_sample(adv, 512, cu(g["fps_start"]))), g["fps_512"])
    torch.manual_seed(7)                      # the seed make_golden.py drew the start indices under
    assert np.array_equal(npy(pcd.pointnet2_utils.farthest_point_sample(adv, 512)), g["fps_512"])
    assert np.array_equal(npy(pcd.curvenet_util.farthest_point_sample(adv, 128)), g["fps0_128"])
    assert np.array_equal(npy(pcd.curvenet_util.farthest_point_sample(adv[:, :300], 300)), g["fps0_all"])
    fidx = cu(g["fps_512"])
    assert np.array_equal(npy(pcd.pointnet2_utils.index_points(adv, fidx)), g["index_points_2d"])
    bq = pcd.pointnet2_utils.query_ball_point(0.2, 32, adv, pcd.pointnet2_utils.index_points(adv, fidx))
    assert np.array_equal(npy(bq), g["ball_idx"])
    assert np.array_equal(npy(pcd.pointnet2_utils.index_points(adv, bq[:, :64])), g["index_points_3d"])


def test_f_three_nn_interpolation_vs_reference():
    g = load_golden("f_graph_sampling")
    x1, x2, f2 = cu(g["fp_xyz1"], True), cu(g["fp_xyz2"], True), cu(g["fp_feat"], True)
    out = pcd.pointnet2_utils.three_nn_interpolate(x1.permute(0, 2, 1), x2.permute(0, 2, 1), f2.permute(0, 2, 1)).permute(0, 2, 1)
    np.testing.assert_allclose(npy(out), g["fp_out"], rtol=1e-5, atol=1e-6)
    (out * cu(g["fp_gw"])).sum().backward()
    assert rel_inf(g["fp_gf"], npy(f2.grad)) < RTOL
    # float64 evaluation of everything behind the (bit-identical) fp32 distances: weights, interpolation, chain rule
    p1, p2, pf = g["fp_xyz1"].transpose(0, 2, 1), g["fp_xyz2"].transpose(0, 2, 1), g["fp_feat"].transpose(0, 2, 1)
    _, d32, i3 = O.three_nn_interpolate(p1, p2, pf)
    o64, g1, g2, gf = F64.three_nn_interpolate_grad64(p1, p2, pf, i3, g["fp_gw"].transpose(0, 2, 1), d32)
    e1, e2 = rel_inf(npy(x1.grad).transpose(0, 2, 1), g1), rel_inf(npy(x2.grad).transpose(0, 2, 1), g2)
    r1, r2 = rel_inf(g["fp_g1"].transpose(0, 2, 1), g1), rel_inf(g["fp_g2"].transpose(0, 2, 1), g2)
    print(f"3-NN interpolation gradients vs float64: ours {e1:.1e} / {e2:.1e}; reference fp32 autograd {r1:.1e} / {r2:.1e}")
    assert e1 < RTOL and e2 < RTOL and rel_inf(npy(f2.grad).transpose(0, 2, 1), gf) < RTOL
    assert rel_inf(g["fp_g1"], npy(x1.grad)) < RTOL + r1 and rel_inf(g["fp_g2"], npy(x2.grad)) < RTOL + r2


@pytest.mark.parametrize("N,npoint", [(100, 100), (257, 64), (513, 128), (1500, 512), (3000, 256), (4096, 1024),
                                      (6000, 128), (10000, 64)])
def test_f_farthest_point_sample_every_variant(N, npoint):
    rs = np.random.RandomState(N)
    xyz = rs.rand(3, N, 3).astype(np.float32)
    xyz[1, N // 2:] = xyz[1, :N - N // 2]                        # duplicated points: first-index ties
    start = rs.randint(0, N, size=3)
    got = F.farthest_point_sample(cu(xyz), npoint, cu(start))
    assert np.array_equal(npy(got), O.farthest_point_sample(xyz, npoint, start))
    cf = cu(np.ascontiguousarray(xyz.transpose(0, 2, 1)))         # channel-first storage through strides
    assert np.array_equal(npy(F.farthest_point_sample(cf.transpose(1, 2), npoint, cu(start))), npy(got))


# ------------------------------------------- L4: attack loops against the reference's own loops
# Loop-level parity is only as well conditioned as the loss: Adam turns a gradient into a step of
# ~lr * g/|g|, so wherever the loss is discontinuous (Hausdorff's single arg-max pair, the kNN loss's
# outlier mask, ProjectInnerPoints' sign test) two correct implementations differ by O(lr) on the few
# points that sit on the discontinuity.  Chamfer (smooth) is compared tightly, the others by the
# fraction of coordinates that agree.
def _loop_fixture():
    import tiny_victim
    g = load_golden("l4_attack_loops")
    return g, tiny_victim.from_npz(g).cuda()


def _agree(a, b, tol=1e-4):
    return float((np.abs(a - b) < tol).mean())


@pytest.mark.parametrize("use_graph", [False, True])
def test_l4_cw_loop_chamfer_vs_reference(use_graph):
    """attack/CW/CW_attack.py:57-260 run unmodified on CPU (B=1, 3 binary steps x 12 iterations, its own
    torch.randn draws replayed) vs. the device-resident loop: same best distance and adversarial cloud."""
    g, victim = _loop_fixture()
    CL = pcd.cw_loop
    atk = CL.CWAttack(victim, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.ChamferDist(method="adv2ori"),
                      attack_lr=1e-2, init_weight=10., max_weight=80., binary_step=3, num_iter=12,
                      clip_func=CL.ClipPointsLinf(0.18), use_graph=use_graph)
    bestdist, bestattack, ok = atk.attack(cu(g["data"]), cu(g["label"]), init_noise=torch.from_numpy(g["cw_chamfer_noise"]))
    assert bool(ok.all())
    np.testing.assert_allclose(npy(bestdist), g["cw_chamfer_bestdist"], rtol=2e-4)
    d = np.abs(npy(bestattack) - g["cw_chamfer_bestattack"])
    assert d.max() < 2e-4 and np.quantile(d, 0.99) < 5e-6          # measured: max 5.9e-5, p99 5e-7 (lr = 1e-2)


def test_l4_cw_loop_hausdorff_vs_reference():
    g, victim = _loop_fixture()
    CL = pcd.cw_loop
    atk = CL.CWAttack(victim, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.HausdorffDist(method="ori2adv"),
                      attack_lr=1e-2, init_weight=10., max_weight=80., binary_step=3, num_iter=12,
                      clip_func=CL.ClipPointsLinf(0.18))
    bestdist, bestattack, ok = atk.attack(cu(g["data"]), cu(g["label"]), init_noise=torch.from_numpy(g["cw_hausdorff_noise"]))
    assert bool(ok.all())
    np.testing.assert_allclose(npy(bestdist), g["cw_hausdorff_bestdist"], rtol=3e-2)
    assert _agree(npy(bestattack), g["cw_hausdorff_bestattack"]) > 0.98          # measured 0.996


def test_l4_knn_attack_loop_vs_reference():
    """attack/KNN/KNN_attack.py:56-246 (ChamferkNNDist k=5, ProjectInnerClipLinf, 20 iterations) on CPU vs.
    the device-resident loop."""
    g, victim = _loop_fixture()
    CL = pcd.cw_loop
    dist = pcd.dist_utils.ChamferkNNDist(chamfer_method="adv2ori", knn_k=5, knn_alpha=1.05, chamfer_weight=5., knn_weight=3.)
    for use_graph in (False, True):
        atk = CL.KNNAttack(victim, CL.UntargetedLogitsAdvLoss(kappa=15.), dist, CL.ProjectInnerClipLinf(0.1),
                           attack_lr=1e-3, num_iter=20, use_graph=use_graph)
        adv, _ = atk.attack(cu(g["data"]), cu(g["label"]), init_noise=torch.from_numpy(g["knn_noise"][0]))
        d = np.abs(npy(adv) - g["knn_adv"])
        assert np.median(d) < 1e-6 and _agree(npy(adv), g["knn_adv"]) > 0.93     # measured: median 7e-9, 0.956
        assert np.abs(npy(adv) - g["data"]).max() > 1e-2                         # the cloud did move


def _geoa3(g, tag, use_graph=False, reps=1, **kw):
    import tiny_victim
    victim = tiny_victim.from_npz(g).cuda()
    G = pcd.geoa3_loop
    atk = G.GeoA3Attack(victim, classes=7, initial_const=10., lr=0.01, binary_max_steps=3, iter_max_steps=15,
                        hd_loss_weight=0.1, curv_loss_weight=1.0, curv_loss_knn=16, use_graph=use_graph, **kw)
    data = cu(np.repeat(g["data"], reps, 0)); label = cu(np.repeat(g["label"], reps, 0))
    off = torch.from_numpy(np.repeat(g[tag + "_offsets"], reps, 1))
    best, ok, best_loss, best_step = atk.attack(data, label, init_offset=off)
    return atk, npy(best), npy(ok), npy(best_loss), npy(best_step)


@pytest.mark.parametrize("tag,kw", [("plain", {}), ("proj_clip", dict(is_pro_grad=True, cc_linf=0.02, is_use_lr_scheduler=True))])
def test_l4_geoa3_loop_vs_reference(tag, kw):
    """The reference's own geoA3_attack (GeoA3_attack.py:185-473), run unmodified on CPU at B = 1 by
    oracle/make_golden.py --geoa3 from recorded offset draws, against the device-resident GeoA3Attack: same success
    flag and best step, best adversarial cloud to 1e-4 of the cloud's extent (3 x 15 Adam steps through
    Hausdorff arg-max / nearest-neighbour switches)."""
    g = load_golden("l4_geoa3_loop")
    atk, best, ok, best_loss, best_step = _geoa3(g, tag, **kw)
    assert ok.tolist() == g[tag + "_success"].tolist()
    if tag == "plain":
        assert best_step.tolist() == g[tag + "_best_step"].tolist()
    d = np.abs(best - g[tag + "_best_attack"])
    # Adam turns a rounding-level gradient difference at a discontinuity (Hausdorff arg-max, a nearest-neighbour switch)
    # into a +-lr step of that one point, on any two correct implementations: median to 2e-6, >= 99 % of the coordinates
    # to 1e-5, the handful of switched points by at most a few lr
    frac = float((d < 1e-5).mean())
    print(f"geoa3 {tag}: median {np.median(d):.2e}  max {d.max():.2e}  within 1e-5: {frac:.4f}")
    # measured: plain 1.0000 within 1e-5 (max 2.8e-6).  With is_pro_grad the reference projects each offset onto the normal
    # of the original point nearest to the OFFSET VECTOR (GeoA3_attack.py:68), a query among near-origin points that flips
    # on rounding and then moves the point by up to cc_linf: 0.86 of the coordinates agree, the rest differ by <= cc_linf
    need = 0.99 if tag == "plain" else 0.80
    assert np.median(d) < 2e-6 and frac > need and d.max() < 5e-2, (float(d.max()), float(np.median(d)), frac)
    if "cc_linf" in kw:
        ori = g["data"].transpose(0, 2, 1)
        assert np.sqrt(((best - ori) ** 2).sum(1)).max() <= kw["cc_linf"] * (1 + 1e-5)


def test_l4_geoa3_loop_batch_safe_and_graph():
    """Three copies of the fixture in one batch give the B = 1 result three times (the reference's loop reads
    .item() and one shared output_label, i.e. is B = 1 only); the CUDA-graph loop reproduces the eager one."""
    g = load_golden("l4_geoa3_loop")
    _, b1, ok1, l1, s1 = _geoa3(g, "plain")
    # global_batch=1: the reference's loss is a batch MEAN, so B = 3 scales every gradient by 1/3 and Adam's eps = 1e-8 then
    # perturbs the steps; with the B = 1 normalisation the three copies must reproduce the single run
    _, b3, ok3, l3, s3 = _geoa3(g, "plain", reps=3, global_batch=1)
    for k in range(3):
        assert (np.abs(b3[k] - b1[0]) < 1e-5).mean() > 0.99 and ok3[k] == ok1[0] and s3[k] == s1[0]
    _, bg, okg, lg, sg = _geoa3(g, "plain", use_graph=True)
    # capturable Adam evaluates its bias corrections with fp32 tensor ops (eager: Python doubles): updates differ by 1e-7
    # relative per step, 45 steps
    dg = np.abs(bg - b1)
    assert (dg < 1e-4).mean() > 0.99 and np.median(dg) < 1e-5 and okg.tolist() == ok1.tolist(), (float(dg.max()), float(np.median(dg)))


def test_l4_loops_are_batch_safe():
    """B > 1 (which the reference loops cannot do: .item() on batch tensors): every sample evolves as it
    does alone."""
    g, victim = _loop_fixture()
    CL = pcd.cw_loop
    data = torch.cat([cu(g["data"]), cu(g["data"])[:, torch.randperm(256, generator=torch.Generator().manual_seed(1))] * 0.9], 0)
    with torch.no_grad():
        label = victim(data.transpose(1, 2))[0].argmax(1)
    noise = torch.randn(3, 2, 3, 256, generator=torch.Generator().manual_seed(2)) * 1e4
    mk = lambda: CL.CWAttack(victim, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.ChamferDist(method="adv2ori"),
                             attack_lr=1e-2, binary_step=3, num_iter=12, clip_func=CL.ClipPointsLinf(0.18), global_batch=1)
    d2, a2, _ = mk().attack(data, label, init_noise=noise)
    for b in range(2):
        d1, a1, _ = mk().attack(data[b:b + 1], label[b:b + 1], init_noise=noise[:, b:b + 1])
        np.testing.assert_allclose(npy(d2[b:b + 1]), npy(d1), rtol=1e-3)
        assert _agree(npy(a2[b:b + 1]), npy(a1)) > 0.98


# ------------------------------------------------------------- randomized shapes / layouts / edge cases
def _layout(a, kind):
    """the same [B,N,C] cloud as contiguous, channel-first view, or a strided slice of a larger buffer"""
    t = cu(a)
    if kind == 1:
        return cu(np.ascontiguousarray(a.transpose(0, 2, 1))).transpose(1, 2)
    if kind == 2:
        big = torch.zeros(a.shape[0], a.shape[1], a.shape[2] + 2, device="cuda")
        big[:, :, 1:1 + a.shape[2]] = t
        return big[:, :, 1:1 + a.shape[2]]
    return t


@pytest.mark.parametrize("seed", range(24))
def test_random_nn1_shapes(seed):
    rs = np.random.RandomState(1000 + seed)
    B = int(rs.randint(1, 5)); N = int(rs.choice([1, 2, 31, 33, 127, 500, 1025, 2500])); M = int(rs.choice([1, 3, 32, 64, 129, 700, 2049]))
    form_key = ["row_col_mulsum", "col_row_mulsum", "sum_first_fma"][seed % 3]
    form, norm, oform, onorm = FORMS[form_key]
    rows = rs.randn(B, N, 3).astype(np.float32); cols = rs.randn(B, M, 3).astype(np.float32)
    if seed % 4 == 0 and M > 2:
        cols[:, M // 2:] = cols[:, :M - M // 2]                   # duplicates: lowest-index ties
    if seed % 5 == 0:
        rows *= 1e-3; cols *= 1e-3                                 # tiny coordinates (denormal-free, cancellation heavy)
    r = F.nn1(_layout(rows, seed % 3), _layout(cols, (seed // 3) % 3), form, norm, cache=False)
    o = oracle_nn1(rows, cols, oform, onorm)
    assert np.array_equal(npy(r.row_arg), o.row_arg) and np.array_equal(npy(r.col_arg), o.col_arg)
    assert np.array_equal(npy(r.row_min), o.row_min) and np.array_equal(npy(r.col_min), o.col_min)


@pytest.mark.parametrize("seed", range(24))
def test_random_knn_shapes(seed):
    rs = np.random.RandomState(2000 + seed)
    B = int(rs.randint(1, 4)); C = int(rs.choice([1, 2, 3, 3, 3, 5, 16, 64])); N = int(rs.choice([1, 7, 64, 300, 1100]))
    M = int(rs.choice([1, 5, 33, 256, 257, 900, 2100]))
    K = int(min(M, rs.choice([1, 2, 3, 8, 17, 20, 33, 64])))
    form_key = ["col_row_mulsum", "row_col_mulsum"][seed % 2]
    form, norm, oform, onorm = FORMS[form_key]
    rows = rs.randn(B, N, C).astype(np.float32); cols = rs.randn(B, M, C).astype(np.float32)
    if seed % 3 == 0 and M > 4:
        cols[:, M // 2:] = cols[:, :M - M // 2]
    d, i = F.knn(_layout(rows, seed % 3), _layout(cols, (seed // 3) % 3), K, form=form, norm=norm)
    od, oi = O.knn(oform, rows, cols, O.norms(onorm, rows), O.norms(onorm, cols), K)
    assert np.array_equal(npy(i), oi) and np.array_equal(npy(d), od)


@pytest.mark.parametrize("seed", range(8))
def test_random_ball_query_and_fps(seed):
    rs = np.random.RandomState(3000 + seed)
    B = int(rs.randint(1, 4)); N = int(rs.choice([5, 64, 333, 1500])); S = int(rs.choice([1, 17, 128]))
    ns = int(rs.choice([1, 8, 32, 64])); radius = float(rs.choice([0.05, 0.2, 0.6, 3.0]))
    xyz = rs.rand(B, N, 3).astype(np.float32); q = rs.rand(B, S, 3).astype(np.float32)
    got = pcd.pointnet2_utils.query_ball_point(radius, ns, _layout(xyz, seed % 3), _layout(q, (seed + 1) % 3))
    assert np.array_equal(npy(got), O.query_ball_point(radius, ns, xyz, q))
    npoint = int(min(N, rs.choice([1, 4, 60])))
    start = rs.randint(0, N, size=B)
    fps = F.farthest_point_sample(_layout(xyz, (seed + 2) % 3), npoint, cu(start))
    assert np.array_equal(npy(fps), O.farthest_point_sample(xyz, npoint, start))


def test_pipelined_loss_matches_eager():
    """graph.PipelinedLoss (one CUDA graph, per-slice upload -> forward+backward -> download) against the eager
    drop-in surface: per-sample losses bit-identical, gradient to 1e-6 (atomic summation order)."""
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    ori_h = synth.face_clouds(10, 1024, seed=21).pin_memory()
    adv_h = synth.perturb(ori_h, 0.01, seed=22).pin_memory()

    def loss_fn(a, o):
        c1, c2 = pcd.distance.chamfer(a, o)
        h1, h2 = pcd.distance.hausdorff(a, o)
        l = torch.stack([c1, c2, h1, h2])
        return l.sum(), (l,)

    a = adv_h.cuda().requires_grad_(True)
    loss, (l_ref,) = loss_fn(a, ori_h.cuda())
    loss.backward()
    for kw in (dict(chunks=1), dict(slice_sizes=[3, 7], prioritize=False), dict(chunks=3)):
        p = pcd.graph.PipelinedLoss(loss_fn, adv_h, ori_h, **kw)
        for _ in range(2):                                   # replay twice: static buffers, same answer
            aux, grad = p.replay()
            torch.cuda.synchronize()
            assert torch.equal(torch.cat([x[0] for x in aux], 1), l_ref.detach().cpu())
            assert rel_inf(npy(a.grad), grad.numpy()) < 1e-6
    # new inputs are written into the pinned buffers in place
    adv_h.copy_(synth.perturb(ori_h, 0.02, seed=23))
    aux, grad = p.replay()
    torch.cuda.synchronize()
    a2 = adv_h.cuda().requires_grad_(True)
    loss2, (l2,) = loss_fn(a2, ori_h.cuda())
    loss2.backward()
    assert torch.equal(torch.cat([x[0] for x in aux], 1), l2.detach().cpu()) and rel_inf(npy(a2.grad), grad.numpy()) < 1e-6


# ------------------------------------------------------------- model-level: the callers either side of the path
def test_dgcnn_victim_with_kernels_matches_torch_formulation():
    """A DGCNN-shaped victim (tools/victims.py) forward + backward w.r.t. the cloud with this package's
    k-NN + edge-feature kernels vs. the reference's torch formulation (model/dgcnn.py:194-227), same weights."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import victims
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(0)
    ours = victims.DGCNNVictim(lambda x, k: pcd.dgcnn.get_graph_feature(x, k=k), k=8, emb_dims=64, num_classes=5).cuda().eval()
    ref = victims.DGCNNVictim(victims.torch_graph_feature, k=8, emb_dims=64, num_classes=5).cuda().eval()
    ref.load_state_dict(ours.state_dict())
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    x0 = synth.face_clouds(2, 512, seed=9).cuda().transpose(1, 2).contiguous()
    outs, grads = [], []
    for m in (ours, ref):
        x = x0.clone().requires_grad_(True)
        o = m(x)[0]
        o[:, 1].sum().backward()
        outs.append(npy(o)); grads.append(npy(x.grad))
    np.testing.assert_allclose(outs[0], outs[1], rtol=1e-4, atol=1e-5)
    assert rel_inf(grads[1], grads[0]) < 1e-3          # feature-space graphs can differ at near-ties (cuBLAS order)


def test_sample_and_group_matches_reference_formulation_on_cpu():
    """PointNet++ set-abstraction grouping (model/pointnet2_utils.py:107-135): FPS + ball query + gathers on the
    GPU kernels vs. the reference's formulation restated with torch on the CPU (same torch.randint start draw)."""
    rs = np.random.RandomState(4)
    xyz = rs.rand(3, 700, 3).astype(np.float32)
    pts = rs.randn(3, 700, 5).astype(np.float32)
    npoint, radius, nsample = 64, 0.25, 16
    torch.manual_seed(123)
    new_xyz, new_points = pcd.pointnet2_utils.sample_and_group(npoint, radius, nsample, cu(xyz), cu(pts))
    torch.manual_seed(123)
    x, p = torch.from_numpy(xyz), torch.from_numpy(pts)
    B, N, _ = x.shape
    cent = torch.zeros(B, npoint, dtype=torch.long)
    dist = torch.ones(B, N) * 1e10
    far = torch.randint(0, N, (B,), dtype=torch.long)
    bi = torch.arange(B)
    for i in range(npoint):                                        # :59-81
        cent[:, i] = far
        c = x[bi, far, :].view(B, 1, 3)
        d = torch.sum((x - c) ** 2, -1)
        m = d < dist
        dist[m] = d[m]
        far = torch.max(dist, -1)[1]
    nx = x[bi[:, None], cent]
    sq = -2 * torch.matmul(nx, x.permute(0, 2, 1)) + torch.sum(nx ** 2, -1).view(B, npoint, 1) + torch.sum(x ** 2, -1).view(B, 1, N)
    gi = torch.arange(N).view(1, 1, N).repeat(B, npoint, 1)        # :84-104
    gi[sq > radius ** 2] = N
    gi = gi.sort(dim=-1)[0][:, :, :nsample]
    first = gi[:, :, 0].view(B, npoint, 1).repeat(1, 1, nsample)
    gi[gi == N] = first[gi == N]
    gx = x[bi[:, None, None], gi] - nx.view(B, npoint, 1, 3)
    ref_points = torch.cat([gx, p[bi[:, None, None], gi]], dim=-1)
    assert np.array_equal(npy(new_xyz), nx.numpy())
    assert np.array_equal(npy(new_points), ref_points.numpy())
