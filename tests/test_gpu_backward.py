"""GPU: every backward kernel against float64 autograd of the loss it differentiates, at random and edge-case shapes,
layouts and upstream gradients.

The references (oracle/fp64_forms.py) are torch float64 expressions of the loss formulas, evaluated at the kernels' own
indices (pinned bit-for-bit by the forward tests in test_gpu_parity.py) and differentiated by autograd on the CPU; none of
them restates a kernel's closed form.  The bar is rel_inf < 1e-5.  An element that receives more than 64 atomic
contributions may instead stay within the a-priori bound of fp32 summation, n_e 2^-24 sum_k |t_k|, with sum_k |t_k| the
float64 sum of the absolute per-pair contributions.
"""
import ctypes
import importlib
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from conftest import rel_inf
from oracle import fp64_forms as F64

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
F = pcd.functional

RTOL = 1e-5
NAN = float("nan")
FORMS = [(F.FORM_ROW_COL, F.NORM_MULSUM), (F.FORM_COL_ROW, F.NORM_MULSUM), (F.FORM_SUM_FIRST, F.NORM_FMA)]


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def npy(t):
    return t.detach().cpu().numpy()


def t64(a, grad=True):
    return torch.tensor(np.asarray(a, np.float64), requires_grad=grad)


def layout(a, kind, grad=False):
    """the cloud a [B,N,C] as a contiguous tensor (0), a channel-first view (1) or a strided slice of a wider buffer (2)"""
    if kind == 1:
        t = cu(a.transpose(0, 2, 1)).transpose(1, 2)
    elif kind == 2:
        big = torch.zeros(a.shape[0], a.shape[1], a.shape[2] + 2, device="cuda")
        big[:, :, 1:1 + a.shape[2]] = cu(a)
        t = big[:, :, 1:1 + a.shape[2]]
    else:
        t = cu(a)
    return t.detach().requires_grad_(grad)


def fp32(a):
    return np.asarray(a, np.float32)


def bound(leaf, taps):
    """(n_e [B,P], sum_k |t_k| [B,P,C]) of the non-zero per-pair contributions autograd scattered onto `leaf`"""
    B, P, C = leaf.shape
    cnt = torch.zeros(B, P, dtype=torch.float64)
    s = torch.zeros(B, P, C, dtype=torch.float64)
    for x, idx, g in taps:
        if x is leaf and g.grad is not None:
            idx = idx.contiguous()
            cnt.scatter_add_(1, idx, (g.grad != 0).any(-1).double())
            s.scatter_add_(1, idx[:, :, None].expand(-1, -1, C).contiguous(), g.grad.abs())
    return cnt.numpy(), s.numpy()


def assert_grad(ours, ref, bnd=None, what=""):
    ours = np.asarray(ours, np.float64)
    assert ours.shape == ref.shape, what
    err = np.abs(ours - ref)
    den = np.abs(ref).max()
    ok = err <= RTOL * (den if den > 0 else 1.0)
    if bnd is not None:
        cnt, s = bnd
        ok |= (cnt[..., None] > 64) & (err <= cnt[..., None] * 2.0 ** -24 * s)
    assert np.isfinite(ours).all() and ok.all(), (what, rel_inf(ours, ref), int((~ok).sum()))


# ------------------------------------------------------------------------------------------- NN-1
STATS = ("row_sum", "row_max", "col_sum", "col_max")


def upstream_terms(rs, mix, B, N, M):
    """the loss as a list of (NN1Result field, weight): a [B] / per-point float32 array, or 'sum' / 'mean' (autograd hands
    the backward a stride-0 expanded gradient for those)"""
    terms = []
    if mix in ("point", "all"):
        terms += [("row_min", fp32(rs.randn(B, N))), ("col_min", fp32(rs.randn(B, M)))]
    if mix in ("sum", "all"):
        terms += [("row_sum", "sum"), ("col_sum", "mean"), ("row_max", "mean"), ("col_max", "sum")]
    if mix in ("weights", "all"):
        terms += [(s, fp32(rs.randn(B))) for s in STATS]
    return terms


def _reduce(x, w):
    if isinstance(w, str):
        return x.sum() if w == "sum" else x.mean()
    return (x * (cu(w) if x.is_cuda else torch.from_numpy(np.asarray(w, np.float64)))).sum()


def gpu_loss(res, terms):
    return sum(_reduce(getattr(res, name), w) for name, w in terms)


def nn1_ref(rows, cols, res, swap, transform, terms, row_scale=1.0, col_scale=1.0):
    """float64 gradients of the loss `terms` at the kernel's arg-mins / arg-maxes: ((g_rows, bound), (g_cols, bound))"""
    ra, ca, rmin, cmin = npy(res.row_arg), npy(res.col_arg), npy(res.row_min), npy(res.col_min)
    ram, cam = npy(res.row_argmax), npy(res.col_argmax)
    # the arg-maxes the backward routes the max gradients through are the first maxima of the fp32 minima
    assert np.array_equal(ram, rmin.argmax(1)) and np.array_equal(cam, cmin.argmax(1))
    R, C, taps = t64(rows), t64(cols), []
    v_row, v_col = F64.nn1_surrogates64(R, C, ra, ca, rmin, cmin, swap, transform, taps)
    stat = {"row_min": v_row, "col_min": v_col,
            "row_sum": float(np.float32(row_scale)) * v_row.sum(1), "col_sum": float(np.float32(col_scale)) * v_col.sum(1),
            "row_max": v_row.gather(1, torch.from_numpy(ram.astype(np.int64))[:, None])[:, 0],
            "col_max": v_col.gather(1, torch.from_numpy(cam.astype(np.int64))[:, None])[:, 0]}
    sum(_reduce(stat[name], w) for name, w in terms).backward()
    return (R.grad.numpy(), bound(R, taps)), (C.grad.numpy(), bound(C, taps))


def run_nn1(rows, cols, form, norm, swap, transform, terms, kinds=(0, 0), need=(True, True), scales=(1.0, 1.0), what=""):
    tr, tc = layout(rows, kinds[0], need[0]), layout(cols, kinds[1], need[1])
    res = F.nn1(tr, tc, form, norm, swap_norms=swap, transform=transform, row_sum_scale=scales[0], col_sum_scale=scales[1],
                cache=False)
    rmin = npy(res.row_min).astype(np.float64)
    assert (np.abs(npy(res.row_sum) - np.float32(scales[0]) * rmin.sum(1)) <= 2e-6 * abs(scales[0]) * np.abs(rmin).sum(1)).all()
    assert np.array_equal(npy(res.row_max), npy(res.row_min).max(1))
    gpu_loss(res, terms).backward()
    (gr, br), (gc, bc) = nn1_ref(rows, cols, res, swap, transform, terms, *scales)
    if need[0]:
        assert_grad(npy(tr.grad), gr, br, what + " rows")
    if need[1]:
        assert_grad(npy(tc.grad), gc, bc, what + " cols")
    return res, tr, tc


SIZES = [1, 2, 31, 33, 127, 500, 1025, 2500]


@pytest.mark.parametrize("seed", range(48))
def test_nn1_backward_random(seed):
    rs = np.random.RandomState(4000 + seed)
    B = int(rs.randint(1, 5))
    N = int(rs.choice(SIZES))
    swap = seed % 4 < 2                                  # swapped norms need N == M
    M = N if swap else int(rs.choice(SIZES))
    transform = [F.VALUE_SQUARED, F.VALUE_SQRT_CLAMP][seed % 2]
    form, norm = FORMS[(seed // 4) % 3]
    need = [(True, True), (True, False), (False, True)][int(rs.randint(0, 3))]
    mix = ["point", "sum", "weights", "all"][(seed // 2) % 4]
    cols = fp32(rs.randn(B, M, 3))
    rows = fp32(cols[:, rs.randint(0, M, N)] + 0.05 * rs.randn(B, N, 3)) if seed % 3 == 0 else fp32(rs.randn(B, N, 3))
    scales = (1.0 / N, 1.0 / M) if seed % 5 else (0.37, 1.0)
    run_nn1(rows, cols, form, norm, swap, transform, upstream_terms(rs, mix, B, N, M),
            kinds=(int(rs.randint(0, 3)), int(rs.randint(0, 3))), need=need, scales=scales,
            what=f"B={B} N={N} M={M} swap={swap} t={transform} mix={mix}")


@pytest.mark.parametrize("transform", [F.VALUE_SQUARED, F.VALUE_SQRT_CLAMP])
def test_nn1_backward_swapped_norms(transform):
    """swap_norms: the two norm terms land on the other index and take that minimum's chain factor (g / v under sqrt)."""
    rs = np.random.RandomState(41)
    cols = fp32(rs.rand(2, 300, 3))
    rows = fp32(cols + 0.02 * rs.randn(2, 300, 3))
    for mix in ("point", "weights", "all"):
        run_nn1(rows, cols, F.FORM_COL_ROW, F.NORM_MULSUM, True, transform, upstream_terms(rs, mix, 2, 300, 300), what=mix)


def test_nn1_backward_memset_path():
    """B*N*3 not a multiple of 4: the forward does not clear the gradient buffers, the backward memsets them."""
    rs = np.random.RandomState(42)
    rows, cols = fp32(rs.randn(1, 33, 3)), fp32(rs.randn(1, 127, 3))
    assert (33 * 3) % 4 and (127 * 3) % 4
    for transform in (F.VALUE_SQUARED, F.VALUE_SQRT_CLAMP):
        run_nn1(rows, cols, F.FORM_SUM_FIRST, F.NORM_FMA, False, transform, upstream_terms(rs, "all", 1, 33, 127))


def test_nn1_backward_unstaged_clouds():
    """> 17 K points: the fix-up re-scans global memory and its zero fill of the gradient buffers is the unstaged one."""
    rs = np.random.RandomState(43)
    cols = fp32(rs.rand(1, 17408, 3) - 0.5)
    rows = fp32(cols[:, :17200] + 0.002 * rs.randn(1, 17200, 3))
    run_nn1(rows, cols, F.FORM_SUM_FIRST, F.NORM_FMA, False, F.VALUE_SQUARED, upstream_terms(rs, "all", 1, 17200, 17408),
            scales=(1 / 17200, 1 / 17408))


def test_nn1_backward_exact_copies_under_sqrt():
    """Rows that are exact copies of columns have minimum 0: under sqrt their gradient is 0, not NaN."""
    rs = np.random.RandomState(44)
    cols = fp32(rs.randn(2, 500, 3))
    perm = rs.permutation(500)[:400]
    rows = cols[:, perm].copy()
    rows[:, 200:] += fp32(0.01 * rs.randn(2, 200, 3))
    zeros = 0
    for form, norm in FORMS:
        res, _, _ = run_nn1(rows, cols, form, norm, False, F.VALUE_SQRT_CLAMP, upstream_terms(rs, "all", 2, 400, 500))
        assert (npy(res.row_arg)[:, :200] == perm[:200]).all()
        zeros += int((npy(res.row_min)[:, :200] == 0).sum())
    assert zeros > 0                                                     # the v == 0 branch of the chain factor ran


def test_nn1_backward_hub():
    """4096 rows whose nearest column is one point: 4096 atomic contributions onto that column."""
    rs = np.random.RandomState(45)
    far = rs.randn(2, 1023, 3)
    cols = fp32(np.concatenate([np.zeros((2, 1, 3)), 5 * far / np.linalg.norm(far, axis=-1, keepdims=True)], 1))
    rows = fp32(0.01 * rs.randn(2, 4096, 3))
    for transform in (F.VALUE_SQUARED, F.VALUE_SQRT_CLAMP):
        res, _, _ = run_nn1(rows, cols, F.FORM_ROW_COL, F.NORM_MULSUM, False, transform, upstream_terms(rs, "all", 2, 4096, 1024))
        assert (npy(res.row_arg) == 0).all()


def test_nn1_backward_tied_maxima():
    """Every minimum equal (a lattice shifted by an exact offset): all of the max gradient goes to the first index."""
    g = np.stack(np.meshgrid(np.arange(6), np.arange(6), np.arange(6), indexing="ij"), -1).reshape(1, -1, 3) * 0.25
    cols = fp32(np.concatenate([g, g + 3.0]))
    rows = fp32(cols + np.array([0.0625, 0.0, 0.0]))
    rs = np.random.RandomState(46)
    for form, norm in FORMS:
        res, _, _ = run_nn1(rows, cols, form, norm, False, F.VALUE_SQUARED, upstream_terms(rs, "weights", 2, 216, 216))
        assert (npy(res.row_min) == 0.0625 ** 2).all() and (npy(res.row_argmax) == 0).all() and (npy(res.col_argmax) == 0).all()


def test_nn1_backward_chamfer_and_hausdorff_share_one_sweep():
    """distance.chamfer + distance.hausdorff on the same tensors: one cached sweep, all four weights in one backward."""
    rs = np.random.RandomState(47)
    gts = fp32(rs.rand(3, 1000, 3))
    preds = fp32(gts[:, rs.randint(0, 1000, 900)] + 0.01 * rs.randn(3, 900, 3))
    p, t = cu(preds).requires_grad_(True), cu(gts)
    w = [fp32(rs.rand(3)) for _ in range(4)]
    F.clear_cache()
    n0 = F.launches()
    c1, c2 = pcd.distance.chamfer(p, t)
    h1, h2 = pcd.distance.hausdorff(p, t)
    assert F.launches() - n0 == 3                          # one forward chain served both
    ((c1 * cu(w[0])).sum() + (c2 * cu(w[1])).sum() + (h1 * cu(w[2])).sum() + (h2 * cu(w[3])).sum()).backward()
    res = F.nn1(t, p.detach(), F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    terms = [("col_sum", w[0]), ("row_sum", w[1]), ("col_max", w[2]), ("row_max", w[3])]
    _, (gc, bc) = nn1_ref(gts, preds, res, False, F.VALUE_SQUARED, terms, 1 / 1000, 1 / 900)
    assert_grad(npy(p.grad), gc, bc)
    F.clear_cache()


# ------------------------------------------------------------------------------------ NN-1, C ABI
def _cloud(t):
    return [None, 0, 0, 0] if t is None else [t.data_ptr(), t.stride(0), t.stride(1), t.stride(2)]


def nan_grad(B, P, strided):
    """a NaN-filled gradient buffer [B,P,3]: dense, or a channel-first view"""
    if strided:
        return torch.full((B, 3, P), NAN, device="cuda").transpose(1, 2)
    return torch.full((B, P, 3), NAN, device="cuda")


@pytest.mark.parametrize("case", ["two_pass", "memset", "rows_only", "cols_only", "w_strides", "two_pass_swap_sqrt"])
def test_nn1_backward_c_abi(case):
    """pcd_nn1_backward on buffers it must write in full (grads_prezeroed = 0): channel-first views (the two-pass scheme),
    dense buffers (memset + atomics), one gradient pointer NULL, and w arrays read with element strides 2, 3, 0 and 1."""
    lib = pcd._lib.load()
    rs = np.random.RandomState(["two_pass", "memset", "rows_only", "cols_only", "w_strides", "two_pass_swap_sqrt"].index(case) + 50)
    B, N = 3, 700
    swap = case == "two_pass_swap_sqrt"
    M = N if swap else 900
    transform = F.VALUE_SQRT_CLAMP if swap or case == "memset" else F.VALUE_SQUARED
    form, norm = (F.FORM_COL_ROW, F.NORM_MULSUM) if swap else (F.FORM_SUM_FIRST, F.NORM_FMA)
    cols = fp32(rs.randn(B, M, 3))
    rows = fp32(cols[:, :N] + 0.1 * rs.randn(B, N, 3))
    tr, tc = layout(rows, 1), layout(cols, 2)
    res = F.nn1(tr, tc, form, norm, swap_norms=swap, transform=transform, cache=False)
    g_row, g_col = fp32(rs.randn(B, N)), fp32(rs.randn(B, M))
    g_row[:, ::7] = 0
    stride = [2, 3, 0, 1] if case == "w_strides" else [1, 1, 1, 1]
    w_dev, w_ref = [], []
    for s in stride:
        full = fp32(rs.randn(max(1, (B - 1) * s + 1)))
        w_dev.append(cu(full))
        w_ref.append(full[np.arange(B) * s])
    scales = (0.5, 0.25)
    strided = case not in ("memset",)
    gr = None if case == "cols_only" else nan_grad(B, N, strided)
    gc = None if case == "rows_only" else nan_grad(B, M, strided)
    dg_r, dg_c = cu(g_row), cu(g_col)
    st = lib.pcd_nn1_backward(*_cloud(tr), *_cloud(tc), B, N, M, int(swap), transform,
                              res.row_arg.data_ptr(), res.col_arg.data_ptr(), res.row_min.data_ptr(), res.col_min.data_ptr(),
                              dg_r.data_ptr(), dg_c.data_ptr(),
                              w_dev[0].data_ptr(), w_dev[1].data_ptr(), res.row_argmax.data_ptr(),
                              w_dev[2].data_ptr(), w_dev[3].data_ptr(), res.col_argmax.data_ptr(),
                              (ctypes.c_int64 * 4)(*stride), scales[0], scales[1], *_cloud(gr), *_cloud(gc), 0,
                              F._stream())
    pcd._lib.check(st, "pcd_nn1_backward")
    torch.cuda.synchronize()
    terms = [("row_min", g_row), ("col_min", g_col)] + list(zip(STATS, w_ref))
    (ref_r, br), (ref_c, bc) = nn1_ref(rows, cols, res, swap, transform, terms, *scales)
    if gr is not None:
        assert_grad(npy(gr), ref_r, br, case + " rows")
    if gc is not None:
        assert_grad(npy(gc), ref_c, bc, case + " cols")


# ------------------------------------------------------------------------------------------- k-NN
def knn_ref(rows, cols, idx, g, swap, same=False):
    R, taps = t64(rows), []
    C = R if same else t64(cols)
    (F64.knn_pairs64(R, C, idx, swap, taps) * torch.from_numpy(np.asarray(g, np.float64))).sum().backward()
    return (R.grad.numpy(), bound(R, taps)), (C.grad.numpy(), bound(C, taps))


KNN_CASES = ([("swap", K) for K in (2, 3, 17, 20, 33, 64)] + [("plain", K) for K in (2, 3, 17, 20, 33, 64)]
             + [("self_swap", 20), ("self_plain", 17), ("duplicates", 33), ("hub", 8), ("hub", 64)])


@pytest.mark.parametrize("kind,K", KNN_CASES)
def test_knn_backward(kind, K):
    rs = np.random.RandomState(5000 + K + 100 * [c[0] for c in KNN_CASES].index(kind))
    B = 2
    swap = kind in ("swap", "self_swap")
    same = kind.startswith("self")
    N, M = (500, 500) if swap else (300, 1100)
    cols = fp32(rs.randn(B, M, 3))
    rows = fp32(rs.randn(B, N, 3))
    if kind == "duplicates":
        cols[:, M // 2:] = cols[:, :M - M // 2]                     # every candidate exists twice: lowest-index ties
    if kind == "hub":                                                # K columns at the origin's doorstep, every row near it
        far = rs.randn(B, M, 3)
        cols = fp32(4 * far / np.linalg.norm(far, axis=-1, keepdims=True))
        cols[:, 100:100 + K] = fp32(0.05 * rs.randn(B, K, 3))
        N, rows = 2048, fp32(0.01 * rs.randn(B, 2048, 3))
    if same:
        rows = cols = fp32(rs.rand(B, 700, 3))
        N = M = 700
    kr, kc = int(rs.randint(0, 3)), int(rs.randint(0, 3))
    tr = layout(rows, kr, True)
    tc = tr if same else layout(cols, kc, True)
    d, idx = F.knn(tr, tc, K, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM, swap_norms=swap)
    if kind == "hub":
        assert (np.sort(npy(idx), 2) == np.arange(100, 100 + K)).all()
    g = fp32(rs.randn(B, N, K))
    g[rs.rand(B, N, K) < 0.3] = 0
    (d * cu(g)).sum().backward()
    (gr, br), (gc, bc) = knn_ref(rows, cols, npy(idx), g, swap, same)
    if same:
        assert_grad(npy(tr.grad), gr, br, kind)
    else:
        assert_grad(npy(tr.grad), gr, br, kind + " rows")
        assert_grad(npy(tc.grad), gc, bc, kind + " cols")


@pytest.mark.parametrize("swap", [False, True])
def test_knn_backward_c_abi_nan_buffers(swap):
    """pcd_knn_backward writes both gradients in full: NaN-filled dense and channel-first buffers come back finite and right."""
    lib = pcd._lib.load()
    rs = np.random.RandomState(60 + swap)
    B, N, K = 2, 400, 12
    M = N if swap else 650
    rows, cols = fp32(rs.randn(B, N, 3)), fp32(rs.randn(B, M, 3))
    tr, tc = layout(rows, 0), layout(cols, 1)
    _, idx = F.knn(tr, tc, K, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM, swap_norms=swap)
    g = fp32(rs.randn(B, N, K))
    dg = cu(g)
    (ref_r, br), (ref_c, bc) = knn_ref(rows, cols, npy(idx), g, swap)
    for strided in (False, True):
        gr, gc = nan_grad(B, N, strided), nan_grad(B, M, not strided)
        st = lib.pcd_knn_backward(*_cloud(tr), *_cloud(tc), B, N, M, K, int(swap), idx.data_ptr(), dg.data_ptr(),
                                  *_cloud(gr), *_cloud(gc), F._stream())
        pcd._lib.check(st, "pcd_knn_backward")
        torch.cuda.synchronize()
        assert_grad(npy(gr), ref_r, br, "rows")
        assert_grad(npy(gc), ref_c, bc, "cols")


# ------------------------------------------------------------------------------ k-NN outlier loss
OUTLIER_CASES = [(N, k) for N in (2, 33, 1023, 1024, 1025, 4096, 5000) for k in (1, 5, 16, 63) if k + 1 <= N]


def outlier_check(pc, k, alpha, swap, loss, value, mask, thr, grad, gB):
    B, N, _ = pc.shape
    x = cu(pc)
    dists, idx = F.knn(x, x, k + 1, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM, swap_norms=swap)
    d64 = npy(dists).astype(np.float64)[:, :, 1:]
    v64 = d64.mean(-1)
    thr64 = v64.mean(-1) + alpha * v64.std(-1, ddof=1)
    value, mask, thr = npy(value), npy(mask), npy(thr)
    assert rel_inf(value, v64) < RTOL
    assert rel_inf(thr, thr64) < RTOL
    assert np.array_equal(mask, (value > thr[:, None]).astype(np.float32))
    assert rel_inf(npy(loss), (v64 * mask).mean(1)) < RTOL
    l64, m64, g64 = F64.knn_outlier_loss_grad64(pc, npy(dists), npy(idx), alpha, gB)
    assert np.array_equal(m64, mask)
    assert_grad(grad, g64, what=f"N={N} k={k} alpha={alpha}")


@pytest.mark.parametrize("N,k", OUTLIER_CASES)
def test_knn_outlier_loss_backward(N, k):
    """F.knn_outlier_loss summed (upstream stride 0), KNNDist with weights and batch_avg=False (stride 1) and
    kNN_smoothing_loss averaged (stride 0, swapped norms), each with a retain_graph second backward (not pre-zeroed)."""
    rs = np.random.RandomState(N * 100 + k)
    B = 2
    pc = fp32(rs.rand(B, N, 3))
    pc[:, :max(1, N // 20)] += fp32(rs.rand(B, max(1, N // 20), 3))       # a few outliers
    w = fp32(rs.rand(B) + 0.5)
    for alpha in (0.0, 1.05, 3.0):
        for variant in ("sum", "weights", "smoothing"):
            kind = int(rs.randint(0, 3))
            if variant == "smoothing":
                x = cu(pc.transpose(0, 2, 1)).requires_grad_(True)
                loss = pcd.loss_utils.kNN_smoothing_loss(x, k, alpha)
                total, gB, swap = loss.mean(), np.full(B, 1.0 / B), True
            else:
                x = layout(pc, kind, True)
                if variant == "sum":
                    loss = F.knn_outlier_loss(x, k, alpha)[0]
                    total, gB, swap = loss.sum(), np.ones(B), False
                else:
                    loss = pcd.dist_utils.KNNDist(k=k, alpha=alpha)(x, weights=w, batch_avg=False)
                    total, gB, swap = (loss * cu(w)).sum(), w.astype(np.float64) ** 2, False
            g1, = torch.autograd.grad(total, x, retain_graph=True)
            g1 = npy(g1).copy()
            g2, = torch.autograd.grad(total, x)
            if variant == "smoothing":
                g1, g2 = g1.transpose(0, 2, 1), npy(g2).transpose(0, 2, 1)
            else:
                g2 = npy(g2)
            x_pm = x.detach().transpose(1, 2) if variant == "smoothing" else x.detach()
            l, value, mask, thr = F.knn_outlier_loss(x_pm, k, alpha, swap_norms=swap)
            if variant == "weights":
                np.testing.assert_array_equal(npy(loss), npy(l) * w)
            else:
                np.testing.assert_array_equal(npy(loss), npy(l))
            outlier_check(pc, k, alpha, swap, l, value, mask, thr, g1, gB)
            assert_grad(g2, g1.astype(np.float64), what="retain_graph")


# ------------------------------------------------------------------------------------------- kappa
@pytest.mark.parametrize("k", [1, 2, 8, 16, 31])
@pytest.mark.parametrize("use_nidx", [False, True])
def test_kappa_backward(k, use_nidx):
    """Batch 0 random; batch 1 with exact duplicate neighbours (r = 0); batch 2 with neighbours 1e-13 away (below the
    1e-12 clamp of the unit vector); batch 3 with offsets exactly in the tangent plane (the subgradient of |s| at 0 is 0).
    Values and gradients are compared per sample: the clamp branch's 1e12 gradients would hide the others."""
    rs = np.random.RandomState(70 + k + 1000 * use_nidx)
    B, N = 4, 333
    pc = rs.rand(B, N, 3)
    nrm = rs.randn(B, N, 3)
    pc[1, 1::2] = pc[1, 0:-1:2]                                           # exact duplicates
    pc[2, :20] *= 1e-9                                                    # 20 points around the origin ...
    pc[2, 20:40] = pc[2, :20] + np.array([1e-13, 0.0, 0.0])               # ... each with a twin 1e-13 away
    pc[3, :, 2] = 0.5                                                     # a plane z = 0.5 ...
    flat = rs.rand(N) < 0.5
    nrm[3, flat] = [0.0, 0.0, 1.0]                                        # ... half of it with the plane's normal
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    pc, nrm = fp32(pc), fp32(nrm)
    x = layout(pc, 1 + k % 2, True)
    n = layout(nrm, 2 - k % 2)
    _, idx = F.knn(x.detach(), x.detach(), k + 1, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM, swap_norms=True)
    nidx = torch.from_numpy(rs.randint(0, N, (B, N)).astype(np.int64)).cuda() if use_nidx else None
    kap = F.kappa(x, n, idx, nidx=nidx)
    gk = fp32(rs.randn(B, N))
    (kap * cu(gk)).sum().backward()
    a = t64(pc)
    k64 = F64.kappa64(a, t64(nrm, False), npy(idx), None if nidx is None else npy(nidx))
    (k64 * torch.from_numpy(gk.astype(np.float64))).sum().backward()
    ours_v, ours_g, ref_v, ref_g = npy(kap), npy(x.grad), k64.detach().numpy(), a.grad.numpy()
    assert np.isfinite(ours_g).all()
    for b in range(B):
        assert rel_inf(ours_v[b], ref_v[b]) < RTOL, b
        assert_grad(ours_g[b], ref_g[b], what=f"sample {b}")
    assert np.abs(ref_g[2]).max() > 1e9                                  # the clamp branch was reached
    # the 40 points at the origin are each other's neighbours: every other point of sample 2 is held to the bar on its own
    assert (npy(idx)[2, :40] < 40).all()
    assert_grad(ours_g[2][40:], ref_g[2][40:], what="sample 2 away from the origin")


# ---------------------------------------------------------------------------- three-NN interpolation
@pytest.mark.parametrize("seed", range(4))
def test_three_nn_interpolation_backward(seed):
    rs = np.random.RandomState(80 + seed)
    B = int(rs.randint(1, 4))
    N, S = [(1000, 250), (64, 700), (2048, 513), (300, 3)][seed]
    D = [1, 7, 64, 128][seed]
    x1, x2, f2 = fp32(rs.rand(B, N, 3)), fp32(rs.rand(B, S, 3)), fp32(rs.randn(B, S, D))
    t1, t2, tf = layout(x1, seed % 3, True), layout(x2, (seed + 1) % 3, True), layout(f2, seed % 2, True)
    out = pcd.pointnet2_utils.three_nn_interpolate(t1, t2, tf)
    gw = fp32(rs.randn(B, N, D))
    (out * cu(gw)).sum().backward()
    d32, i3 = F.knn(t1.detach(), t2.detach(), 3, form=F.FORM_ROW_COL, norm=F.NORM_MULSUM)
    o64, g1, g2, gf = F64.three_nn_interpolate_grad64(x1, x2, f2, npy(i3), gw, npy(d32))
    assert rel_inf(npy(out), o64) < RTOL
    assert_grad(npy(t1.grad), g1, what="xyz1")
    assert_grad(npy(t2.grad), g2, what="xyz2")
    assert_grad(npy(tf.grad), gf, what="feat2")


# ------------------------------------------------------------------ the forward's zero fill
def poison_allocator():
    """Fill the caching allocator's free blocks with NaN: one >= 256 MB block (large pool) and many 1 MB ones (small pool)."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    big = torch.full((64 << 20,), NAN, device="cuda")
    small = [torch.full((1 << 18,), NAN, device="cuda") for _ in range(96)]
    torch.cuda.synchronize()
    del big, small


@pytest.mark.parametrize("case", ["raw", "packed", "unstaged", "outlier"])
def test_forward_zero_fill_under_poisoned_allocator(case):
    """The NN-1 fix-up and the outlier forward clear the gradient buffers their backward only adds into.  With the
    allocator's free memory NaN, a missing or partial fill shows as NaN or a wrong gradient."""
    rs = np.random.RandomState(90 + len(case))
    if case == "outlier":
        B, N = 2, 2048
    else:
        B, N, M = {"raw": (2, 1024, 2048), "packed": (3, 1000, 1500), "unstaged": (1, 17408, 17408)}[case]
    pc = fp32(rs.rand(B, N, 3))
    poison_allocator()
    probe = torch.empty((B, N, 3), device="cuda")
    assert probe.isnan().all(), "the poison did not take"
    del probe
    if case == "outlier":
        x = cu(pc).requires_grad_(True)
        loss, value, mask, thr = F.knn_outlier_loss(x, 16, 1.05)
        loss.sum().backward()
        outlier_check(pc, 16, 1.05, False, loss, value, mask, thr, npy(x.grad), np.ones(B))
        return
    cols = fp32(rs.rand(B, M, 3))
    kinds = (2, 0) if case == "packed" else (0, 0)
    terms = upstream_terms(rs, "all", B, N, M)
    run_nn1(pc, cols, F.FORM_SUM_FIRST, F.NORM_FMA, False, F.VALUE_SQUARED, terms, kinds=kinds, scales=(1 / N, 1 / M))


# ------------------------------------------------------ self-exclusion of the brute-force k-NN losses
def _direct_knn64(pm, k):
    """the reference's ranking: direct-form squared distances (d(i,i) = 0 exactly), self first -> (idx [B,N,k], ambiguous [B,N])
    with `ambiguous` where the k-th and (k+1)-th distances lie within the expansion form's fp32 rounding of each other"""
    d = ((pm[:, :, None].astype(np.float64) - pm[:, None]) ** 2).sum(-1)
    order = np.argsort(d, axis=2, kind="stable")
    srt = np.take_along_axis(d, order, 2)
    n2 = (pm.astype(np.float64) ** 2).sum(-1)
    tol = 16 * 2.0 ** -24 * (n2 + n2.max(1, keepdims=True))
    return order[:, :, 1:k + 1], srt[:, :, k + 1] - srt[:, :, k] <= tol


def _loss64(name, adv_pm, ori_pm, idx):
    a = t64(adv_pm)
    ii = torch.from_numpy(idx.astype(np.int64))
    nb = F64._gather_pm(a, ii)                                            # [B,N,k,3]
    if name == "displacement_loss":
        theta = ((a - torch.from_numpy(ori_pm.astype(np.float64))) ** 2).sum(-1)
        v = ((torch.gather(theta, 1, ii.reshape(ii.shape[0], -1)).view(ii.shape) - theta[:, :, None]) ** 2).mean(2)
    elif name == "repulsion_loss":
        dis = ((nb - a[:, :, None]) ** 2).sum(-1)
        v = -(dis * torch.exp(-(dis ** 2) / 0.03 ** 2)).mean(2)
    else:
        dis = ((a[:, :, None] - nb + 1e-12) ** 2).sum(-1).sqrt()
        dm = dis.mean(-1)
        v = (dm[:, :, None] - torch.gather(dm, 1, ii.reshape(ii.shape[0], -1)).view(ii.shape)).abs().mean(-1)
    return a, v


@pytest.mark.parametrize("name,k", [("displacement_loss", 16), ("repulsion_loss", 4), ("distance_kmean_loss", 8)])
def test_knn_losses_drop_self_next_to_near_duplicates(name, k):
    """Pairs 1e-5 .. 3e-4 apart in a unit cloud: in the expansion form the twin can rank before the point itself.  The
    losses must still drop self and keep the k nearest others, as the reference's direct-form ranking does.  Points
    whose neighbour set is decided by a near tie within fp32 rounding get no upstream weight."""
    rs = np.random.RandomState(95 + k)
    B, N = 2, 1024
    ori = rs.rand(B, N, 3)
    for b in range(B):
        src, dst = rs.permutation(N)[:128].reshape(2, 64)
        u = rs.randn(64, 3)
        ori[b, dst] = ori[b, src] + u / np.linalg.norm(u, axis=1, keepdims=True) * np.exp(rs.uniform(np.log(1e-5), np.log(3e-4), (64, 1)))
    ori = fp32(ori)
    adv = fp32(ori + 0.01 * rs.randn(B, N, 3)) if name == "displacement_loss" else ori
    idx, amb = _direct_knn64(ori, k)
    a, v64 = _loss64(name, adv, ori, idx)
    excl = amb.copy()
    if name == "distance_kmean_loss":                                     # the loss reads the neighbours' own means, and
        dis = np.sqrt(((adv[:, :, None].astype(np.float64) - adv[np.arange(B)[:, None, None], idx]) ** 2).sum(-1))
        dm = dis.mean(-1)                                                 # |.| has a kink where two means agree to fp32 rounding
        kink = (np.abs(dm[:, :, None] - np.take_along_axis(dm, idx.reshape(B, -1), 1).reshape(B, N, k)) < 1e-6 * dm.max()).any(-1)
        excl = amb | kink | np.take_along_axis(amb, idx.reshape(B, -1), 1).reshape(B, N, k).any(-1)
    assert excl.mean() < 0.3                                             # most points are held to the bar
    gN = fp32(rs.randn(B, N))
    gN[excl] = 0
    (v64 * torch.from_numpy(gN.astype(np.float64))).sum().backward()
    x = cu(adv.transpose(0, 2, 1)).requires_grad_(True)
    LU = pcd.loss_utils
    if name == "displacement_loss":
        v = LU.displacement_loss(x, cu(ori.transpose(0, 2, 1)), k=k)
    elif name == "repulsion_loss":
        v = LU.repulsion_loss(x, k=k, h=0.03)
    else:
        v = LU.distance_kmean_loss(x, k)
    (v * cu(gN)).sum().backward()
    ref = v64.detach().numpy()
    bad = np.abs(npy(v) - ref) > RTOL * np.abs(ref).max()
    assert not (bad & ~excl).any(), (name, int((bad & ~excl).sum()))
    assert_grad(npy(x.grad).transpose(0, 2, 1), a.grad.numpy(), what=name)
