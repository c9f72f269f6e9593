"""GPU: the float64 nearest-neighbour distances (functional.nn_dist64, metrics.chamfer64 / hausdorff64) against the
numpy brute force of the contract (bit-identical per-point minima and arg-minima, exact maxima, means within the
summation bound) across data kinds, shapes and ragged lengths; batch, layout and column-split invariance; non-finite
input; scipy per sample; SOR-kept clouds scored with their lengths."""
import importlib
import math

import numpy as np
import pytest
import torch
from scipy.spatial import distance

from oracle import nn_dist64_oracle as O

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F = pcd.functional
M64 = pcd.metrics


def make_cloud(kind, B, N, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "uniform":
        return torch.rand((B, N, 3), generator=g) * 2 - 1
    if kind == "lattice":                       # exact ties everywhere: a shuffled 1/8-pitch grid
        side = int(np.ceil(N ** (1 / 3)))
        grid = torch.stack(torch.meshgrid(*[torch.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3).float() * 0.125
        return torch.stack([grid[torch.randperm(grid.shape[0], generator=g)[:N]] for _ in range(B)])
    pc = synth.face_clouds(B, N, seed=seed)
    if kind == "duplicates":                    # a third of the points repeat others exactly
        n = N // 3
        if n:
            pc[:, N - n:] = pc[:, :n]
        return pc
    return pc + float(kind) * torch.randn(pc.shape, generator=g)      # face clouds + noise at sigma = kind


def make_pair(kind, B, N, M, seed):
    a = make_cloud(kind, B, N, seed)
    if kind in ("uniform", "lattice", "duplicates"):
        return a, make_cloud(kind, B, M, seed + 1)
    # b: the same face cloud at M points, moved by the noise; sigma = 1e-7 leaves many exactly equal coordinates
    b = synth.face_clouds(B, M, seed=seed) + float(kind) * torch.randn((B, M, 3), generator=torch.Generator().manual_seed(seed + 1))
    return a, b


def lengths_for(mode, B, n, seed):
    if mode == "full":
        return None
    rng = np.random.default_rng(seed)
    if mode == "zero_one":
        v = np.array([0, 1, n, rng.integers(0, n + 1)] * B)[:B]
    else:
        v = rng.integers(0, n + 1, B)
    return torch.from_numpy(v.astype(np.int64))


def mean_bound(v, mean):
    n = len(v)
    return (n - 1) * 2.0 ** -53 * math.fsum(np.abs(v)) / n + 2.0 ** -53 * abs(mean)


def to_np(r):
    return type(r)(*[t.cpu().numpy() for t in r])


def check_against_oracle(r, o, la, lb):
    assert np.array_equal(r.a_min, o.a_min, equal_nan=True) and np.array_equal(r.a_arg, o.a_arg)
    assert np.array_equal(r.b_min, o.b_min, equal_nan=True) and np.array_equal(r.b_arg, o.b_arg)
    B = r.a_min.shape[0]
    for pre, pts, lens in (("a", o.a_min, la), ("b", o.b_min, lb)):
        for i in range(B):
            v = pts[i, :lens[i]]
            for name in ("max_sq", "max", "argmax"):
                got, want = getattr(r, f"{pre}_{name}")[i], getattr(o, f"{pre}_{name}")[i]
                assert np.array_equal(got, want, equal_nan=True), (pre, name, i, got, want)
            for name, x in (("mean_sq", v), ("mean", np.sqrt(v))):
                got, want = getattr(r, f"{pre}_{name}")[i], getattr(o, f"{pre}_{name}")[i]
                if len(x) == 0 or not np.isfinite(want):
                    assert np.array_equal(got, want, equal_nan=True), (pre, name, i, got, want)
                else:
                    exact = math.fsum(x) / len(x)
                    assert abs(got - exact) <= mean_bound(x, exact), (pre, name, i, got, exact)


def run(a, b, la=None, lb=None, **kw):
    r = F.nn_dist64(a.cuda(), b.cuda(), None if la is None else la.cuda(), None if lb is None else lb.cuda(), **kw)
    B, N, M = a.shape[0], a.shape[1], b.shape[1]
    o = O.nn_dist64(a.numpy(), b.numpy(), None if la is None else la.numpy(), None if lb is None else lb.numpy())
    lens_a = np.full(B, N) if la is None else np.clip(la.numpy(), 0, N)
    lens_b = np.full(B, M) if lb is None else np.clip(lb.numpy(), 0, M)
    return r, to_np(r), o, lens_a, lens_b


CASES = [   # kind, B, N, M, length mode
    ("0.01", 1, 1, 1, "full"),
    ("0.01", 2, 1, 700, "full"),
    ("1e-07", 3, 513, 129, "random"),
    ("0.001", 8, 1000, 1025, "zero_one"),
    ("0.01", 3, 4000, 5000, "full"),
    ("0.01", 2, 4000, 5000, "random"),
    ("1e-07", 1, 4096, 4096, "full"),
    ("0.001", 1, 16384, 16384, "full"),
    ("0.01", 1, 16384, 3, "zero_one"),
    ("uniform", 8, 2048, 1500, "random"),
    ("uniform", 5, 777, 6001, "full"),
    ("lattice", 4, 1000, 1331, "full"),
    ("lattice", 2, 4096, 700, "random"),
    ("duplicates", 6, 1537, 1024, "zero_one"),
    ("duplicates", 1, 5000, 4000, "full"),
]


@pytest.mark.parametrize("kind,B,N,M,mode", CASES)
def test_nn_dist64_matches_float64_brute_force(kind, B, N, M, mode):
    a, b = make_pair(kind, B, N, M, seed=N + 7 * M + B)
    la, lb = lengths_for(mode, B, N, seed=1), lengths_for(mode, B, M, seed=2)
    r, rn, o, lens_a, lens_b = run(a, b, la, lb)
    check_against_oracle(rn, o, lens_a, lens_b)
    assert r.a_min.dtype == torch.float64 and r.a_arg.dtype == torch.int64 and r.a_mean.shape == (B,)


def test_non_finite_coordinates():
    a, b = make_pair("0.01", 4, 900, 1100, seed=3)
    a[0, 10, 0] = float("nan")                  # a NaN row
    b[1, 20, 2] = float("nan")                  # a NaN column: every a row of sample 1 takes it
    a[2, 30, 1] = float("inf")                  # inf - inf = NaN against the +inf column below
    b[2, 40, 1] = float("inf")
    b[2, 41, 0] = float("-inf")
    a[3, :, :] = float("inf")                   # every distance of sample 3 is +inf or NaN
    b[3, 5, 0] = 1.0
    for la, lb in ((None, None), (torch.tensor([900, 15, 31, 0]), torch.tensor([1100, 21, 40, 900]))):
        r, rn, o, lens_a, lens_b = run(a, b, la, lb)
        check_against_oracle(rn, o, lens_a, lens_b)


def same_bits(x, y):
    return torch.equal(x.view(torch.int64), y.view(torch.int64)) if x.dtype == torch.float64 else torch.equal(x, y)


def test_batch_layout_and_split_invariance():
    B, N, M = 5, 2100, 1700
    a, b = make_pair("0.001", B, N, M, seed=31)
    a[2, 100, 0] = float("nan")
    la, lb = torch.tensor([2100, 0, 1, 1999, 640]).cuda(), torch.tensor([1700, 5, 0, 1700, 1000]).cuda()
    a, b = a.cuda(), b.cuda()
    ref = F.nn_dist64(a, b, la, lb)
    a_cf = a.transpose(1, 2).contiguous().transpose(1, 2)        # a [B,3,N] cloud passed as its transposed view
    b_strided = torch.full((B, 2 * M, 3), float("nan"), device="cuda")
    b_strided[:, ::2] = b
    for kw in ({"col_split": 0}, {"col_split": 1}, {"col_split": 2}, {"col_split": 7}):
        for x, y in ((a, b), (a_cf, b_strided[:, ::2])):
            r = F.nn_dist64(x, y, la, lb, **kw)
            for u, v in zip(r, ref):
                assert same_bits(u, v)
    for i in range(B):
        r = F.nn_dist64(a[i:i + 1], b[i:i + 1], la[i:i + 1], lb[i:i + 1])
        for u, v in zip(r, ref):
            assert same_bits(u[0], v[i])
    r = F.nn_dist64(a, b, la.long().cpu(), (lb + (1 << 33)).long())  # int64 lengths past 2^31 clamp, never wrap
    full_b = F.nn_dist64(a, b, la, torch.full_like(lb, M))
    for u, v in zip(r, full_b):
        assert same_bits(u, v)


def test_launch_count_no_grad_and_validation():
    a = make_cloud("0.01", 2, 64, 1).cuda().requires_grad_(True)
    b = make_cloud("0.01", 2, 48, 2).cuda()
    before = F.launches()
    r = F.nn_dist64(a, b)
    assert F.launches() - before == 2
    assert not any(t.requires_grad for t in r)
    with pytest.raises(ValueError):
        F.nn_dist64(a, b, torch.ones(3, dtype=torch.int32))
    with pytest.raises(ValueError):
        F.nn_dist64(a, b, torch.ones(2))
    with pytest.raises(ValueError):
        F.nn_dist64(a, b[:1])
    with pytest.raises(TypeError):
        F.nn_dist64(a.double(), b)


def check_metric(chamfer, hausdorff, m, squared):
    """m: scipy's Euclidean nearest-neighbour distances of the valid points.  The Euclidean metrics are sqrt(s) exactly,
    so the mean is within the summation bound and the maximum is equal; squaring scipy's distances does not give s back
    exactly, so the squared metrics agree to a few units in the last place."""
    if squared:
        np.testing.assert_allclose(chamfer, math.fsum(m * m) / len(m), rtol=1e-14, atol=0)
        np.testing.assert_allclose(hausdorff, m.max() ** 2, rtol=1e-15, atol=0)
    else:
        exact = math.fsum(m) / len(m)
        assert abs(chamfer - exact) <= mean_bound(m, exact)
        assert hausdorff == m.max()


@pytest.mark.parametrize("squared", [False, True])
def test_metrics_agree_with_scipy_per_sample(squared):
    B = 4
    a, b = make_pair("0.01", B, 4000, 5000, seed=41)
    la, lb = torch.tensor([4000, 3500, 1, 4000]), torch.tensor([5000, 5000, 4999, 17])
    cd = M64.chamfer64(a.cuda(), b.cuda(), la.cuda(), lb.cuda(), squared=squared)
    hd = M64.hausdorff64(a.cuda(), b.cuda(), la.cuda(), lb.cuda(), squared=squared)
    for i in range(B):
        d = distance.cdist(a[i, :la[i]].double().numpy(), b[i, :lb[i]].double().numpy(), "euclidean")
        for direction, m in ((0, d.min(1)), (1, d.min(0))):
            check_metric(cd[direction][i].item(), hd[direction][i].item(), m, squared)


def test_sor_kept_clouds_scored_with_lengths():
    B, N = 4, 2048
    ori = synth.face_clouds(B, N, seed=51)
    x = ori + 0.01 * torch.randn(ori.shape, generator=torch.Generator().manual_seed(52))
    x[:, :40] = (torch.rand((B, 40, 3), generator=torch.Generator().manual_seed(53)) * 2 - 1) * 3     # outliers
    xg, og = x.cuda(), ori.cuda()
    s = F.sor(xg, 2, 1.1)
    kept = torch.gather(xg, 1, s.kept_idx.clamp_min(0)[..., None].expand(-1, -1, 3))
    for squared in (False, True):
        cd = M64.chamfer64(kept, og, s.lengths, squared=squared)
        hd = M64.hausdorff64(kept, og, s.lengths, squared=squared)
        for i in range(B):
            keep = s.keep[i].cpu().numpy()
            d = distance.cdist(x[i].numpy()[keep].astype(np.float64), ori[i].double().numpy(), "euclidean")
            for direction, m in ((0, d.min(1)), (1, d.min(0))):
                check_metric(cd[direction][i].item(), hd[direction][i].item(), m, squared)
