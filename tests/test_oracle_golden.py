"""CPU: the oracle (oracle/pcd_oracle.{c,py}) against vectors produced by the unmodified
reference (oracle/make_golden.py).  This is what pins the oracle."""
import numpy as np
import pytest

from conftest import load_golden, rel_inf
from oracle import pcd_oracle as O


def test_a1_known_answer_example():
    # utils/dis_utils_torch.py:30-35 (commented example); values recorded in SURVEY.md section 4
    g = load_golden("a1_dis_utils_torch")
    assert np.isclose(g["k_chamfer"], 3.7032, atol=1e-4)
    assert np.isclose(g["k_sgd"], 1.7321, atol=1e-4)
    assert np.isclose(g["k_bid"], 2.4495, atol=1e-4)
    # N, M <= 25 makes torch.cdist take its direct kernel (<= 2.4e-7 from the mm path)
    np.testing.assert_allclose(O.dis_chamfer(g["ka"], g["kb"]), g["k_chamfer"], rtol=1e-6)
    np.testing.assert_allclose(O.dis_sgd_hausdorff(g["ka"], g["kb"]), g["k_sgd"], rtol=1e-6)
    np.testing.assert_allclose(O.dis_bid_hausdorff(g["ka"], g["kb"]), g["k_bid"], rtol=1e-6)


def test_a1_dis_utils_torch():
    g = load_golden("a1_dis_utils_torch")
    a, b = g["a"], g["b"]
    M = O.dis_pairwise_distances(a[:, :, :96], b[:, :, :80])
    # torch's vectorised CPU sqrt is not correctly rounded (99.4 % of lanes): <= 1 ulp
    assert np.abs(M - g["pairwise_distances"]).max() <= 1.2e-7 * np.abs(M).max()
    assert (M == g["pairwise_distances"]).mean() > 0.98
    np.testing.assert_allclose(O.dis_chamfer(a, b), g["chamfer"], rtol=2e-6)
    np.testing.assert_allclose(O.dis_sgd_hausdorff(a, b), g["sgd_hausdorff_dis"], rtol=2e-7)
    np.testing.assert_allclose(O.dis_bid_hausdorff(a, b), g["bid_hausdorff_dis"], rtol=2e-7)


def test_a1_gradients_closed_form_vs_reference_autograd():
    g = load_golden("a1_dis_utils_torch")
    ga, gb = O.dis_grads(g["a"], g["b"], w_col_sum=1 / 3, w_row_sum=1 / 3)
    assert rel_inf(g["chamfer_ga"], ga) < 5e-5 and rel_inf(g["chamfer_gb"], gb) < 5e-5
    ga, gb = O.dis_grads(g["a"], g["b"], w_row_max=1.0)
    assert rel_inf(g["sgd_hausdorff_dis_ga"], ga) < 5e-5 and rel_inf(g["sgd_hausdorff_dis_gb"], gb) < 5e-5


@pytest.mark.parametrize("tag", ["face", "iter0", "ragged", "ties"])
def test_a2_nn1_bit_exact(tag):
    g = load_golden("a2_distance_" + tag)
    r = O._nn1_cw(g["preds"], g["gts"])
    assert np.array_equal(r.row_min, g["row_min"])
    assert np.array_equal(r.col_min, g["col_min"])
    assert np.array_equal(r.row_arg, g["row_arg"])       # lowest-index == torch.min(dim)
    assert np.array_equal(r.col_arg, g["col_arg"])
    if "P_block" in g:
        P = O.batch_pairwise_dist(g["gts"], g["preds"])
        assert np.array_equal(P[:, :64, :48], g["P_block"])


@pytest.mark.parametrize("tag", ["face", "iter0", "ragged"])
def test_a2_losses_and_grads(tag):
    g = load_golden("a2_distance_" + tag)
    l1, l2 = O.chamfer_distance(g["preds"], g["gts"])
    np.testing.assert_allclose(l1, g["chamfer_l1"], rtol=2e-6, atol=1e-12)
    np.testing.assert_allclose(l2, g["chamfer_l2"], rtol=2e-6, atol=1e-12)
    h1, h2 = O.hausdorff_distance(g["preds"], g["gts"])
    assert np.array_equal(h1, g["hausdorff_l1"]) and np.array_equal(h2, g["hausdorff_l2"])
    if tag == "iter0":
        return   # |adv-ori| ~ 1e-7: the reference's own fp32 gradient is rounding noise there
    gp, gg = O.chamfer_distance_grads(g["preds"], g["gts"], g["g1"], g["g2"])
    assert rel_inf(g["chamfer_gp"], gp) < 1e-5 and rel_inf(g["chamfer_gg"], gg) < 1e-5
    gp, gg = O.hausdorff_distance_grads(g["preds"], g["gts"], g["g1"], g["g2"])
    assert rel_inf(g["hausdorff_gp"], gp) < 1e-5 and rel_inf(g["hausdorff_gg"], gg) < 1e-5


def test_a2_set_distance_variant():
    g = load_golden("a2_set_distance")
    l1, l2 = O.chamfer_distance(g["preds"], g["gts"])
    np.testing.assert_allclose((l1 + l2) / 2, g["chamfer"], rtol=2e-6)
    h1, h2 = O.hausdorff_distance(g["preds"], g["gts"])
    np.testing.assert_allclose((h1 + h2) / 2, g["hausdorff"], rtol=1e-7)


def assert_idx_equal_up_to_ties(idx, ref_idx, dists, matrix):
    """torch.topk does not break exact-distance ties by lowest index (the real face scans sit
    on a pixel grid, so exact ties occur); inside a group of equal distances the reference's
    choice is arbitrary.  Contract: the reference's picks have bit-identical distances at every
    rank, and wherever the two differ our pick is the lower index."""
    ref_d = np.take_along_axis(matrix, ref_idx.astype(np.int64), axis=2)
    assert np.array_equal(ref_d, dists)
    diff = idx != ref_idx
    assert diff.mean() < 0.01
    for b, r, c in np.argwhere(diff):
        tied = dists[b, r] == dists[b, r, c]
        lo = np.flatnonzero(matrix[b, r] == dists[b, r, c])
        assert sorted(idx[b, r][tied]) == sorted(lo[:tied.sum()])      # ours = lowest indices


def test_a3_knn_points():
    g = load_golden("a3_knn_utils")
    for tag, p1, p2, K in (("cross1", g["adv"], g["ori"], 1), ("self17", g["adv"], g["adv"], 17),
                           ("cross4", g["ori"], g["adv"], 4)):
        d, i = O.knn_points(p1, p2, K)
        assert np.array_equal(d, g[tag + "_dists"]), tag
        assert_idx_equal_up_to_ties(i, g[tag + "_idx"], d, O.knn_points_matrix(p1, p2))
        assert np.array_equal(O.knn_gather(p2, g[tag + "_idx"]), g[tag + "_nn"])
    assert np.array_equal(O.knn_gather(g["gather_x"], g["self17_idx"]), g["gather_out"])
    with pytest.raises(RuntimeError):
        O.knn_points(g["adv"][:, :100], g["ori"][:, :90], 1)


def test_a5_knn_dist():
    g = load_golden("l3_dist_utils")
    for k in (5, 16):
        loss, _, _ = O.knn_dist_loss(g["adv"], k=k, alpha=1.05)
        np.testing.assert_allclose(loss * g["weights"], g[f"KNNDist_k{k}"], rtol=3e-6)


def test_a6_knn_graph():
    g = load_golden("a6_knn_graph")
    pm = O._cf_to_pm(g["x3"]); nrm = O.norms(O.NORM_MULSUM, pm)
    mat = -O.dgcnn_neg_matrix(g["x3"])
    d20, i20 = O.knn(O.FORM_COL_ROW, pm, pm, nrm, nrm, 20)
    d21, i21 = O.knn(O.FORM_COL_ROW, pm, pm, nrm, nrm, 21)
    assert np.array_equal(i20, O.dgcnn_knn(g["x3"], 20))
    assert_idx_equal_up_to_ties(i20, g["dgcnn_k20"], d20, mat)
    assert_idx_equal_up_to_ties(i21, g["curvenet_k20"], d21, mat)          # CurveNet asks for k+1
    assert_idx_equal_up_to_ties(i20, g["curvenet_normal_k20"], d20, mat)
    # C = 64: the reference's GEMM / sum order is library-blocked (not sequential), so agreement is
    # asserted as a proof (tests/knn_proof.py): differing picks are within the fp32 rounding bound of
    # each other, and wherever the true gaps exceed that bound sets / rows are identical.
    from knn_proof import assert_knn_near_tie_proof
    assert_knn_near_tie_proof(O.dgcnn_knn(g["f64"], 20), g["dgcnn_f64_k20"], g["f64"], "gaussian C=64")


def test_a6_knn_graph_feature_layers():
    """The four knn() calls of the unmodified reference DGCNN forward (C = 3, 64, 64, 128; model/dgcnn.py:299-311),
    recorded by oracle/make_golden.py --features, against the oracle's sequential fp32 chain."""
    from knn_proof import assert_knn_near_tie_proof
    g = load_golden("a6_knn_graph_features")
    for li, C in enumerate((3, 64, 64, 128)):
        x, ref = g[f"x{li}"], g[f"idx{li}"].astype(np.int64)
        assert x.shape[1] == C
        st = assert_knn_near_tie_proof(O.dgcnn_knn(x, 20), ref, x, f"layer {li} C={C}")
        print(f"a6 layer {li} C={C}: oracle vs reference(CPU): {st}")
        if C == 3:
            assert st["differing_entries"] == 0.0       # tie-free fixture, sequential K=3 chain: bit-exact


def test_a7_pointnet2_utils():
    g = load_golden("a7_pointnet2_utils")
    xyz, new_xyz = g["xyz"], g["new_xyz"]
    assert np.array_equal(O.square_distance(new_xyz[:, :64], xyz[:, :96]), g["sqdist_block"])
    assert np.array_equal(O.query_ball_point(0.2, 32, xyz, new_xyz), g["ball_r02_n32"])
    assert np.array_equal(O.query_ball_point(0.4, 64, xyz[:, :512], new_xyz[:, :128]), g["ball_r04_n64"])
    assert np.array_equal(O.query_ball_point(0.02, 8, xyz, new_xyz[:, :64]), g["ball_r002_n8"])


def test_topk_tie_rule_is_lowest_index():
    # torch.topk is not lowest-index on ties (SURVEY.md section 7 hard part 4); the oracle is.
    pc = np.zeros((1, 6, 3), np.float32)
    pc[0, :, 0] = [0, 1, 1, 1, 5, 1]
    d, i = O.knn(O.FORM_COL_ROW, pc, pc, O.norms(0, pc), O.norms(0, pc), 3)
    assert i[0, 0].tolist() == [0, 1, 2]
    assert i[0, 1].tolist() == [1, 2, 3]


def test_ref_torch_port_matches_golden():
    """bench.py's CPU baseline is a torch restatement of the reference path; pin it too."""
    import torch
    from oracle import ref_torch_port as RP
    g = load_golden("a2_distance_face")
    p, t = torch.from_numpy(g["preds"]), torch.from_numpy(g["gts"])
    c1, c2 = RP.chamfer_distance(p, t)
    h1, h2 = RP.hausdorff_distance(p, t)
    np.testing.assert_allclose(c1.numpy(), g["chamfer_l1"], rtol=1e-6)
    np.testing.assert_allclose(c2.numpy(), g["chamfer_l2"], rtol=1e-6)
    assert np.array_equal(h1.numpy(), g["hausdorff_l1"]) and np.array_equal(h2.numpy(), g["hausdorff_l2"])
    assert np.array_equal(RP.batch_pairwise_dist(t, p)[:, :64, :48].numpy(), g["P_block"])


def test_a3_knn_gradients_closed_form_vs_reference_autograd():
    g = load_golden("a3_knn_utils")
    for tag, p1, p2 in (("cross1", g["adv"], g["ori"]), ("cross4", g["ori"], g["adv"]), ("self17", g["adv"], g["adv"])):
        g1, g2 = O.knn_points_grads(p1, p2, g[tag + "_idx"], g[tag + "_gw"])
        if tag == "self17":
            assert rel_inf(g[tag + "_g1"], g1 + g2) < 1e-5
        else:
            assert rel_inf(g[tag + "_g1"], g1) < 1e-5 and rel_inf(g[tag + "_g2"], g2) < 1e-5


# ------------------------------------------------------------- f-2 / f-3 (SURVEY 8f rows 2-3)
def test_f_graph_feature_bit_exact():
    g = load_golden("f_graph_sampling")
    assert np.array_equal(O.dgcnn_knn(g["adv_cf"], 20), g["ggf3_idx"])
    assert np.array_equal(O.get_graph_feature(g["adv_cf"], 20), g["ggf3"])
    assert np.array_equal(O.get_graph_feature(g["f16"], 10, idx=g["ggf16_idx"]), g["ggf16"])
    assert np.array_equal(O.get_graph_feature(g["f16"], 7, idx=g["idx7"]), g["ggf16_idx7"])
    assert np.array_equal(O.lpfa_point_feature(g["adv_cf"], g["lpfa9_idx"]), g["lpfa9"])


def test_f_graph_feature_grads():
    g = load_golden("f_graph_sampling")
    E = (O.EDGE_DIFF, O.EDGE_CENTER)
    assert rel_inf(g["ggf3_gx"], O.edge_feature_grad(g["ggf3_gw"], g["ggf3_idx"], E, 3)) < 1e-5
    assert rel_inf(g["ggf16_gx"], O.edge_feature_grad(g["ggf16_gw"], g["ggf16_idx"], E, 16)) < 1e-5
    L = (O.EDGE_CENTER, O.EDGE_NEIGHBOR, O.EDGE_DIFF)
    assert rel_inf(g["lpfa9_gx"], O.edge_feature_grad(g["lpfa9_gw"], g["lpfa9_idx"], L, 3)) < 1e-5


def test_f_farthest_point_sample_bit_exact():
    g = load_golden("f_graph_sampling")
    assert np.array_equal(O.farthest_point_sample(g["adv"], 512, g["fps_start"]), g["fps_512"])
    assert np.array_equal(O.farthest_point_sample(g["adv"], 128), g["fps0_128"])
    assert np.array_equal(O.farthest_point_sample(g["adv"][:, :300], 300), g["fps0_all"])
    assert np.array_equal(O.index_points(g["adv"], g["fps_512"]), g["index_points_2d"])
    assert np.array_equal(O.index_points(g["adv"], g["ball_idx"][:, :64]), g["index_points_3d"])


def test_f_three_nn_interpolation():
    g = load_golden("f_graph_sampling")
    x1, x2 = g["fp_xyz1"].transpose(0, 2, 1), g["fp_xyz2"].transpose(0, 2, 1)
    out, d, i = O.three_nn_interpolate(x1, x2, g["fp_feat"].transpose(0, 2, 1))
    assert d.min() > 1e-6                                           # well conditioned: no coincident pairs
    np.testing.assert_allclose(out.transpose(0, 2, 1), g["fp_out"], rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------ f-4: local geometry (round 2)
def test_f4_local_geometry_oracle_vs_reference():
    """oracle/make_golden.py --geometry ran the UNMODIFIED estimate_normal / kappa / brute-force losses / AOF
    Laplacian (torch.symeig provided as torch.linalg.eigh, the environment shim its deprecation note prescribes)."""
    g = load_golden("f4_local_geometry")
    adv = g["adv"]; pm = O._cf_to_pm(adv)
    for k in (3, 8, 16):
        idx = O.self_knn_idx(adv, k + 1)
        cov, _ = O.patch_covariance(pm, idx)
        assert rel_inf(cov, g[f"cov_k{k}"]) < 3e-7                         # library bmm / mean order: rounding only
        w, v, _ = O.local_frames(pm, idx)
        nref = g[f"normal_k{k}"].transpose(0, 2, 1)
        unit = np.linalg.norm(nref, axis=-1) > 0.5                          # the reference's sign(0) = 0 zeroes a few normals
        assert unit.mean() > 0.95
        cos = np.abs((v[:, :, 0, :] * nref).sum(-1))
        assert cos[unit].min() > 1 - 1e-5                                   # sign-free comparison (see utility.py:67-69)
    nrm = g["normal_k8"].transpose(0, 2, 1)
    nidx = O.knn_points(pm, O._cf_to_pm(g["ori"]), 1)[1][:, :, 0]
    idx = O.self_knn_idx(adv, 17)
    kap = O.kappa(pm, nrm, idx, nidx=nidx)
    np.testing.assert_allclose(kap, g["kappa_adv_k16"], rtol=0, atol=3e-7)
    g64 = O.kappa_grad64(pm, nrm, idx, g["gN"], nidx=nidx)
    assert rel_inf(g["kappa_adv_k16_g"].transpose(0, 2, 1), g64) < 1e-5      # reference fp32 autograd vs fp64 closed form
    small = g["lap_pc"]
    L = O.graph_laplacian(O._cf_to_pm(small), O.dgcnn_knn(small, 30))
    np.testing.assert_allclose(L, g["lap_L"], rtol=0, atol=1e-5)
    assert ((L != 0) == (g["lap_L"] != 0)).all()                            # identical sparsity: same symmetrised graph


def test_f1_clip_epilogues():
    """oracle restatements of clip_utils.py:5-136 and GeoA3_attack.py:62-101 vs the reference's own CPU outputs
    (oracle/make_golden.py --clips).  The bar is 2 ulp of the largest coordinate, not bit equality, because torch's CPU
    kernels are not a bit-level specification: its vectorised sqrt is not correctly rounded (3 of 512 lengths of the
    fixture are one ulp off the IEEE result numpy and sqrt.rn give), its cross product is compiled with FMA contraction,
    tensor * python-scalar may multiply in double, and ClipPointsL2's 3K-term sum has an order of its own.  The kernels
    are held bit-for-bit to THIS oracle (tests/test_gpu_parity.py) and to torch's own GPU chain where that is exact."""
    g = load_golden("f1_clips")
    ori, adv, normal = g["ori"], g["adv"], g["normal"]
    off = adv - ori

    def close(ours, ref):
        return np.abs(ours - ref).max() <= 2 * np.finfo(np.float32).eps * np.abs(ref).max()

    assert close(O.clip_points_linf(adv, ori, 0.03), g["linf"])
    assert close(O.project_inner_clip_linf(adv, ori, normal, 0.03), g["project_linf"])
    assert close(O.clip_points_l2(adv, ori, 0.5), g["l2"])
    assert close(O.lp_clip(off, 0.02), g["lp_clip"])
    assert close(O.offset_proj(off, ori, normal), g["offset_proj"])
    assert np.array_equal(O.find_offset(ori, adv), g["find_offset"])
    # the fixture exercises every branch
    d = g["linf"] - ori
    assert (np.abs(np.sqrt((d ** 2).sum(1)) - 0.03) < 1e-6).sum() > 100 and (g["linf"] == adv).all(1).sum() > 10
    assert (g["project_linf"][1, :, 5:9] == ori[1, :, 5:9]).all() and (g["lp_clip"] == off).all(1).sum() > 10


@pytest.mark.parametrize("swap", [False, True])
@pytest.mark.parametrize("transform", [0, 1])          # VALUE_SQUARED, VALUE_SQRT_CLAMP
def test_fp64_nn1_and_knn_references_vs_central_differences(swap, transform):
    """The float64 references of the NN-1 / k-NN backward tests (oracle/fp64_forms.py) against central differences of the
    losses they stand for, recomputed from scratch at every step (brute-force minima / k smallest, sqrt where asked) on small
    inputs without ties: the references' gradients are those of the real losses, not of a restated kernel formula."""
    import torch
    from oracle import fp64_forms as F64
    rs = np.random.RandomState(17 + 2 * swap + transform)
    B, N = 2, 7
    M = N if swap else 5
    K = 3
    cols0 = rs.randn(B, M, 3)
    # swapped norms: rows near the columns keep the surrogate's minima positive (the (i, i) entry is |r_i - c_i|^2)
    rows0 = cols0 + 0.2 * rs.randn(B, N, 3) if swap else rs.randn(B, N, 3)
    g_row, g_col, w_max = rs.randn(B, N), rs.randn(B, M), rs.randn(B)
    g_knn = rs.randn(B, N, K)

    def mat(rows, cols):                                   # d[b,i,j] in the form the references evaluate
        if swap:
            return (cols ** 2).sum(-1)[:, :, None] - 2 * rows @ cols.transpose(0, 2, 1) + (rows ** 2).sum(-1)[:, None, :]
        return ((rows[:, :, None] - cols[:, None]) ** 2).sum(-1)

    def val(d):
        return np.sqrt(d) if transform == F64.VALUE_SQRT_CLAMP else d

    def loss(rows, cols):
        d = mat(rows, cols)
        vr, vc = val(d.min(2)), val(d.min(1))
        knn = np.sort(d, 2)[:, :, :K]
        return (g_row * vr).sum() + (g_col * vc).sum() + (w_max * vr.max(1)).sum() + (g_knn * knn).sum()

    d = mat(rows0, cols0)
    srt = np.sort(d, 2)
    assert (np.diff(srt, axis=2)[:, :, :K] > 1e-3).all() and (np.diff(np.sort(d, 1), axis=1)[:, 0] > 1e-3).all()   # no ties
    assert transform == F64.VALUE_SQUARED or min(d.min(2).min(), d.min(1).min()) > 1e-3      # sqrt away from its kink
    row_arg, col_arg = d.argmin(2), d.argmin(1)
    row_min32, col_min32 = val(d.min(2)).astype(np.float32), val(d.min(1)).astype(np.float32)
    r, c = torch.tensor(rows0, requires_grad=True), torch.tensor(cols0, requires_grad=True)
    v_row, v_col = F64.nn1_surrogates64(r, c, row_arg, col_arg, row_min32, col_min32, swap, transform)
    amax = torch.from_numpy(row_min32.argmax(1))
    d2k = F64.knn_pairs64(r, c, np.argsort(d, 2, kind="stable")[:, :, :K], swap)
    L = ((torch.from_numpy(g_row) * v_row).sum() + (torch.from_numpy(g_col) * v_col).sum()
         + (torch.from_numpy(w_max) * v_row.gather(1, amax[:, None])[:, 0]).sum() + (torch.from_numpy(g_knn) * d2k).sum())
    L.backward()
    h = 1e-6
    for leaf, x0 in ((r, rows0), (c, cols0)):
        fd = np.zeros_like(x0)
        for e in np.ndindex(x0.shape):
            xp, xm = x0.copy(), x0.copy()
            xp[e] += h; xm[e] -= h
            args_p = (xp, cols0) if leaf is r else (rows0, xp)
            args_m = (xm, cols0) if leaf is r else (rows0, xm)
            fd[e] = (loss(*args_p) - loss(*args_m)) / (2 * h)
        # fp32 minima under sqrt: the chain factor is taken at v32, 2^-24 relative from the exact root
        assert rel_inf(leaf.grad.numpy(), fd) < (1e-6 if transform == F64.VALUE_SQRT_CLAMP else 1e-8), (swap, transform)
