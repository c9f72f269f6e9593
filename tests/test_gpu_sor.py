"""GPU: the float64 SOR kernels (functional.sor, defense.SORDefense) against the brute force of the contract
(bit-identical values), across data kinds, shapes, k and alpha; layout and batch invariance; the defence's
list, gradient and resampling; non-finite input; the reference's torch formulation on the same GPU."""
import importlib

import numpy as np
import pytest
import torch

from oracle import sor_oracle as O

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F = pcd.functional

BAND = 1e-12
ALPHAS = (0.0, 1.1, 3.0)


def make_cloud(kind, B, N, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "uniform":
        return torch.rand((B, N, 3), generator=g) * 2 - 1
    if kind == "lattice":                       # exact ties everywhere: a shuffled 1/8-pitch grid
        side = int(np.ceil(N ** (1 / 3)))
        grid = torch.stack(torch.meshgrid(*[torch.arange(side)] * 3, indexing="ij"), -1).reshape(-1, 3).float() * 0.125
        return torch.stack([grid[torch.randperm(grid.shape[0], generator=g)[:N]] for _ in range(B)])
    pc = synth.face_clouds(B, N, seed=seed)
    pc = pc + 0.01 * torch.randn(pc.shape, generator=g)
    if kind == "outliers":                      # a few far points
        n = max(1, N // 50)
        pc[:, :n] = (torch.rand((B, n, 3), generator=g) * 2 - 1) * 3
    elif kind == "duplicates":                  # a third of the points repeat others exactly
        n = N // 3
        if n:
            pc[:, N - n:] = pc[:, :n]
    return pc


def check_consistent(keep, kept_idx, lengths):
    for b in range(keep.shape[0]):
        idx = np.flatnonzero(keep[b])
        assert lengths[b] == idx.size
        assert np.array_equal(kept_idx[b, :idx.size], idx)
        assert (kept_idx[b, idx.size:] == -1).all()


KINDS = ("face", "outliers", "duplicates", "lattice", "uniform")
NS = ("k+1", 17, 1000, 1024, 4096, 5000)
KS = (1, 2, 4, 8, 15)
CASES = []
for ci, (kind, n) in enumerate([(kd, n) for kd in KINDS for n in NS]):
    k = KS[ci % len(KS)]
    N = k + 1 if n == "k+1" else n
    B = (1, 3, 8)[ci % 3] if N < 4096 else (1, 3)[ci % 2]
    CASES.append((kind, B, N, k))


@pytest.mark.parametrize("kind,B,N,k", CASES)
def test_sor_matches_float64_brute_force(kind, B, N, k):
    pc = make_cloud(kind, B, N, seed=100 + N + k)
    o = O.sor64(pc.numpy(), k, ALPHAS[0])
    x = pc.cuda()
    for alpha in ALPHAS:
        r = F.sor(x, k, alpha)
        value, thr, keep = r.value.cpu().numpy(), r.threshold.cpu().numpy(), r.keep.cpu().numpy()
        othr, okeep = O.sor64_threshold(o.value, alpha)
        assert np.array_equal(value, o.value)
        assert (np.abs(thr - othr) <= BAND * np.abs(othr)).all(), (thr, othr)
        band = np.abs(o.value - othr[:, None]) <= BAND * np.abs(othr[:, None])
        print(f"{kind} B={B} N={N} k={k} alpha={alpha}: {int(band.sum())} of {band.size} points inside the band")
        assert np.array_equal(keep[~band], okeep[~band])
        if kind not in ("lattice", "duplicates") and N > 2:     # two points share one distance: both sit on the threshold
            assert not band.any()
        check_consistent(keep, r.kept_idx.cpu().numpy(), r.lengths.cpu().numpy())
        assert r.value.dtype == torch.float64 and r.keep.dtype == torch.bool
        assert r.kept_idx.dtype == torch.int64 and r.lengths.dtype == torch.int64


def test_sor_launch_count():
    before = F.launches()
    F.sor(make_cloud("face", 2, 64, 1).cuda())
    assert F.launches() - before == 2


@pytest.mark.parametrize("k", [2, 8, 15])
def test_sor_layout_and_batch_invariance(k):
    pc = make_cloud("outliers", 8, 1500, seed=5).cuda()
    ref = F.sor(pc, k, 1.1)
    cf = pc.transpose(1, 2).contiguous().transpose(1, 2)
    strided = torch.full((8, 3000, 3), float("nan"), device="cuda")
    strided[:, ::2] = pc
    views = [cf, strided[:, ::2]]
    for v in views:
        r = F.sor(v, k, 1.1)
        for a, b in zip(r, ref):
            assert torch.equal(a, b)
    for b in range(8):
        r = F.sor(pc[b:b + 1], k, 1.1)
        for a, full in zip(r, ref):
            assert torch.equal(a[0], full[b])


def test_outlier_removal_list_and_gradient():
    x = make_cloud("outliers", 4, 1024, seed=9).cuda().requires_grad_(True)
    d = pcd.defense.SORDefense(k=2, alpha=1.1)
    sel = d.outlier_removal(x)
    keep = F.sor(x, 2, 1.1).keep
    assert len(sel) == 4
    for b in range(4):
        assert torch.equal(sel[b], x[b][keep[b]])
    sum(s.sum() for s in sel).backward()
    assert torch.equal(x.grad, keep[..., None].expand_as(x).float())


def test_forward_equals_process_data_of_outlier_removal():
    pc = make_cloud("outliers", 6, 1024, seed=13)
    x = pc.cuda()
    o = O.sor64(pc.numpy(), 2, 1.1)
    lengths = o.keep.sum(1)
    # N_i above, equal to and below npoint (with and without a remainder) across the batch and the calls
    for npoint in (int(lengths.min()) - 40, int(lengths[0]), int(lengths.max()) + 1, 2 * int(lengths[1]), 3000):
        d = pcd.defense.SORDefense(k=2, alpha=1.1, npoint=npoint)
        np.random.seed(77)
        out = d(x)
        np.random.seed(77)
        via_list = d.process_data(d.outlier_removal(x))
        np.random.seed(77)
        ref = O.sor_process_data([pc.numpy()[b][o.keep[b]] for b in range(6)], npoint)
        assert out.shape == (6, npoint, 3)
        assert torch.equal(out, via_list)
        assert np.array_equal(out.cpu().numpy(), ref)


def test_non_finite_points_do_not_fault():
    pc = make_cloud("face", 3, 1000, seed=17)
    pc[1, 10, 0] = float("nan")
    pc[2, 20, 2] = float("inf")
    x = pc.cuda()
    r = F.sor(x, 4, 1.1)
    torch.cuda.synchronize()
    clean = F.sor(x[:1], 4, 1.1)
    for a, c in zip(r, clean):
        assert torch.equal(a[:1], c)
    lengths, kept = r.lengths.cpu().numpy(), r.kept_idx.cpu().numpy()
    assert ((lengths >= 0) & (lengths <= 1000)).all()
    assert ((kept >= -1) & (kept < 1000)).all()
    check_consistent(r.keep.cpu().numpy(), kept, lengths)


@pytest.mark.parametrize("B,N,k", [(4, 1024, 2), (2, 4096, 2), (3, 2000, 8)])
def test_sor_agrees_with_reference_torch_formulation_on_gpu(B, N, k):
    x = make_cloud("outliers", B, N, seed=23 + N).cuda()
    r = F.sor(x, k, 1.1)
    _, mask, value, thr = O.sor_outlier_removal(x, k, 1.1)
    np.testing.assert_allclose(r.value.cpu().numpy(), value.cpu().numpy(), rtol=1e-10, atol=0)
    np.testing.assert_allclose(r.threshold.cpu().numpy(), thr.cpu().numpy(), rtol=1e-10, atol=0)
    t = thr.cpu().numpy()[:, None]
    outside = np.abs(value.cpu().numpy() - t) > 1e-9 * np.abs(t)
    print(f"B={B} N={N} k={k}: {int((~outside).sum())} points inside the band")
    assert np.array_equal(r.keep.cpu().numpy()[outside], mask.cpu().numpy()[outside])
