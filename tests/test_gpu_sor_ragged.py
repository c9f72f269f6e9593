"""GPU: SOR on ragged batches (functional.sor with lengths, pcd_sor_forward_len).  Every sample with a statistic is
bit-identical to the unsplit path on its truncated cloud, whatever the rest of the batch, the padding, the layout or
the column split; short samples and padding rows are filled as the contract says; chains with a second SOR pass, the
float64 metrics and the defence work without a loop over samples."""
import ctypes
import importlib

import numpy as np
import pytest
import torch

from oracle import sor_oracle as O
from sor_ragged_oracle import sor64_ragged
from test_gpu_sor import BAND, KINDS, check_consistent, make_cloud

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
F = pcd.functional


def same(a, c):
    """bit-for-bit equality; float64 outputs compare as their bits, so the NaN of padding rows equals itself"""
    if a.dtype == torch.float64:
        a, c = a.view(torch.int64), c.view(torch.int64)
    return torch.equal(a, c)


def ragged_lengths(N, k, seed):
    """0, 1, k, k + 1, N and one random length in [k + 1, N]"""
    rng = np.random.default_rng(seed)
    return [0, 1, k, k + 1, N, int(rng.integers(k + 1, N + 1))]


def assert_sample_equals_alone(r, pc, b, n, k, alpha):
    """every output of sample b of the ragged result r against F.sor on pc[b:b+1, :n] (n >= k + 1), bit for bit"""
    one = F.sor(pc[b:b + 1, :n], k, alpha)
    assert same(r.value[b, :n], one.value[0])
    assert same(r.threshold[b], one.threshold[0])
    assert same(r.keep[b, :n], one.keep[0])
    assert same(r.kept_idx[b, :n], one.kept_idx[0]) and (r.kept_idx[b, n:] == -1).all()
    assert same(r.lengths[b], one.lengths[0])


def assert_padding(r, b, n, k):
    if n < k + 1:
        assert torch.isnan(r.value[b]).all() and torch.isnan(r.threshold[b])
        assert not r.keep[b].any() and (r.kept_idx[b] == -1).all() and r.lengths[b] == 0
    assert torch.isnan(r.value[b, n:]).all() and not r.keep[b, n:].any()


CASES = []
for ci, kind in enumerate(KINDS):
    for N in ((300, 10000) if ci % 2 else (2000, 5000)):
        CASES.append((kind, N, (1, 2, 8, 15)[(ci + N) % 4]))


@pytest.mark.parametrize("kind,N,k", CASES)
def test_ragged_samples_equal_their_truncated_clouds(kind, N, k):
    lengths = ragged_lengths(N, k, seed=N + k)
    pc = make_cloud(kind, len(lengths), N, seed=200 + N + k)
    for b, n in enumerate(lengths):
        pc[b, n:] = float("nan")                                # padding is never read into a result
    x = pc.cuda()
    r = F.sor(x, k, 1.1, lengths=torch.tensor(lengths, device="cuda"))
    o = sor64_ragged(pc.numpy(), lengths, k, 1.1)
    value, thr, keep = r.value.cpu().numpy(), r.threshold.cpu().numpy(), r.keep.cpu().numpy()
    assert np.array_equal(value, o.value, equal_nan=True)
    for b, n in enumerate(lengths):
        assert_padding(r, b, n, k)
        if n < k + 1:
            continue
        assert_sample_equals_alone(r, x, b, n, k, 1.1)
        assert abs(thr[b] - o.threshold[b]) <= BAND * abs(o.threshold[b])
        band = np.abs(o.value[b, :n] - o.threshold[b]) <= BAND * abs(o.threshold[b])
        assert np.array_equal(keep[b, :n][~band], o.keep[b, :n][~band])
    check_consistent(keep, r.kept_idx.cpu().numpy(), r.lengths.cpu().numpy())


def test_padding_values_change_nothing():
    pc = make_cloud("outliers", 4, 3000, seed=31).cuda()
    lengths = torch.tensor([3000, 1200, 2, 2999], device="cuda")
    ref = F.sor(pc, 2, 1.1, lengths=lengths)
    for fill in (float("nan"), float("inf"), -float("inf"), 1e30):
        p = pc.clone()
        for b, n in enumerate(lengths.tolist()):
            p[b, n:] = fill
        for a, c in zip(F.sor(p, 2, 1.1, lengths=lengths), ref):
            assert same(a, c)


def test_lengths_dtypes_and_clamping():
    pc = make_cloud("face", 4, 1000, seed=37).cuda()
    ref = F.sor(pc, 4, 1.1, lengths=torch.tensor([1000, 0, 500, 1000], dtype=torch.int32, device="cuda"))
    for lengths in (torch.tensor([1000, 0, 500, 1000], dtype=torch.int64, device="cuda"),
                    torch.tensor([5000, -3, 500, 2 ** 40], dtype=torch.int64, device="cuda"),
                    torch.tensor([1000, 0, 500, 1000], dtype=torch.int64)):          # a host tensor is moved
        for a, c in zip(F.sor(pc, 4, 1.1, lengths=lengths), ref):
            assert same(a, c)
    full = F.sor(pc, 4, 1.1)
    for a, c in zip(full, ref):
        assert same(a[0], c[0]) and same(a[3], c[3])
    clamped = F.sor(pc, 4, 1.1, lengths=torch.tensor([2 ** 31 - 1, -(2 ** 31), 500, 1000], dtype=torch.int32, device="cuda"))
    for a, c in zip(clamped, ref):
        assert same(a, c)
    with pytest.raises(ValueError, match="lengths"):
        F.sor(pc, 4, 1.1, lengths=torch.tensor([1.0, 2.0, 3.0, 4.0], device="cuda"))
    with pytest.raises(ValueError, match="lengths"):
        F.sor(pc, 4, 1.1, lengths=torch.tensor([1, 2, 3], device="cuda"))


@pytest.mark.parametrize("B,N,k", [(1, 4096, 2), (1, 10000, 8), (3, 2500, 15), (5, 700, 1)])
def test_split_invariance(B, N, k):
    pc = make_cloud("outliers", B, N, seed=41 + N).cuda()
    lengths = torch.tensor([N, N - 1, N // 2, 3, N // 3][:B], device="cuda")
    max_split = (N + 63) // 64                                  # one 64-column tile per range
    for lens in (None, lengths):
        ref = F.sor(pc, k, 1.1, lengths=lens, col_split=1)
        for split in (0, 2, 7, max_split, max_split + 5):
            for a, c in zip(F.sor(pc, k, 1.1, lengths=lens, col_split=split), ref):
                assert same(a, c)


def test_launch_counts():
    before = F.launches()
    F.sor(make_cloud("face", 1, 4096, 1).cuda())               # B = 1: split columns, merge
    assert F.launches() - before == 3
    before = F.launches()
    F.sor(make_cloud("face", 2, 64, 1).cuda(), lengths=torch.tensor([64, 30], device="cuda"))
    assert F.launches() - before == 2


@pytest.mark.parametrize("k", [2, 8, 15])
def test_layout_invariance(k):
    pc = make_cloud("duplicates", 5, 2000, seed=43).cuda()
    lengths = torch.tensor([2000, 1500, 0, 700, 17], device="cuda")
    ref = F.sor(pc, k, 1.1, lengths=lengths)
    cf = pc.transpose(1, 2).contiguous().transpose(1, 2)
    strided = torch.full((5, 4000, 3), float("nan"), device="cuda")
    strided[:, ::2] = pc
    for v in (cf, strided[:, ::2]):
        for a, c in zip(F.sor(v, k, 1.1, lengths=lengths), ref):
            assert same(a, c)


@pytest.mark.parametrize("B,N,k", [(2, 64, 2), (1, 4096, 2), (3, 1500, 8), (32, 1024, 15)])
def test_unsplit_calls_equal_the_fixed_size_entry(B, N, k):
    pc = make_cloud("uniform", B, N, seed=47).cuda()
    lib = pcd._lib.load()
    value = torch.empty((B, N), dtype=torch.float64, device="cuda")
    thr = torch.empty((B,), dtype=torch.float64, device="cuda")
    keep = torch.empty((B, N), dtype=torch.uint8, device="cuda")
    kept = torch.empty((B, N), dtype=torch.int32, device="cuda")
    lengths = torch.empty((B,), dtype=torch.int32, device="cuda")
    st = lib.pcd_sor_forward(pc.data_ptr(), pc.stride(0), pc.stride(1), pc.stride(2), B, N, k, ctypes.c_double(1.1),
                             value.data_ptr(), thr.data_ptr(), keep.data_ptr(), kept.data_ptr(), lengths.data_ptr(),
                             torch.cuda.current_stream().cuda_stream)
    assert st == 0
    r = F.sor(pc, k, 1.1)
    assert same(r.value, value) and same(r.threshold, thr)
    assert same(r.keep, keep.bool()) and same(r.kept_idx, kept.long()) and same(r.lengths, lengths.long())


def test_two_passes_and_float64_metrics_on_the_kept_clouds():
    from oracle import nn_dist64_oracle
    pc = make_cloud("outliers", 6, 2048, seed=53)
    x = pc.cuda()
    lengths = [2048, 1500, 1024, 3, 2047, 800]
    r1 = F.sor(x, 2, 1.1, lengths=torch.tensor(lengths, device="cuda"))
    kept1 = torch.gather(x, 1, r1.kept_idx.clamp_min(0)[..., None].expand(-1, -1, 3))
    r2 = F.sor(kept1, 2, 1.1, lengths=r1.lengths)
    kept2 = torch.gather(kept1, 1, r2.kept_idx.clamp_min(0)[..., None].expand(-1, -1, 3))
    n1, n2 = r1.lengths.cpu().numpy(), r2.lengths.cpu().numpy()
    k1, k2 = kept1.cpu().numpy(), kept2.cpu().numpy()
    for b, n in enumerate(lengths):
        if n < 3:
            assert n1[b] == 0 and n2[b] == 0
            continue
        o1 = O.sor64(pc.numpy()[b:b + 1, :n], 2, 1.1)
        assert np.array_equal(r1.value[b, :n].cpu().numpy(), o1.value[0])
        assert np.array_equal(k1[b, :n1[b]], pc.numpy()[b, :n][r1.keep[b, :n].cpu().numpy()])
        if n1[b] < 3:
            assert n2[b] == 0
            continue
        o2 = O.sor64(k1[b:b + 1, :n1[b]], 2, 1.1)
        assert np.array_equal(r2.value[b, :n1[b]].cpu().numpy(), o2.value[0])
        t = o2.threshold[0]
        outside = np.abs(o2.value[0] - t) > BAND * abs(t)
        assert np.array_equal(r2.keep[b, :n1[b]].cpu().numpy()[outside], o2.keep[0][outside])
        assert n2[b] <= n1[b] <= n
    nd = F.nn_dist64(kept2, x, r2.lengths, torch.tensor(lengths, device="cuda"))
    ond = nn_dist64_oracle.nn_dist64(k2, pc.numpy(), n2, lengths)
    assert np.array_equal(nd.a_min.cpu().numpy(), ond.a_min, equal_nan=True)
    assert np.array_equal(nd.a_arg.cpu().numpy(), ond.a_arg)
    assert np.array_equal(nd.b_min.cpu().numpy(), ond.b_min, equal_nan=True)
    assert np.array_equal(nd.a_max.cpu().numpy(), ond.a_max, equal_nan=True)


def test_defense_with_lengths_equals_a_loop_over_samples():
    pc = make_cloud("outliers", 5, 1500, seed=59).cuda()
    lengths = torch.tensor([1500, 1000, 1499, 600, 1200], device="cuda")
    d = pcd.defense.SORDefense(k=2, alpha=1.1, npoint=1024)
    sel = d.outlier_removal(pc, lengths)
    for b, n in enumerate(lengths.tolist()):
        (one,) = d.outlier_removal(pc[b:b + 1, :n])
        assert same(sel[b], one)
    np.random.seed(5)
    out = d(pc, lengths)
    np.random.seed(5)
    loop = torch.cat([d(pc[b:b + 1, :n]) for b, n in enumerate(lengths.tolist())])
    assert same(out, loop)
    with pytest.raises(ValueError, match="sample 1"):
        d(pc, torch.tensor([1500, 2, 1499, 600, 1200], device="cuda"))


def test_non_finite_points_inside_the_valid_range_do_not_fault():
    pc = make_cloud("face", 4, 1000, seed=61)
    pc[1, 10, 0] = float("nan")
    pc[2, 20, 2] = float("inf")
    pc[3, :] = float("nan")
    x = pc.cuda()
    lengths = torch.tensor([900, 800, 700, 600], device="cuda")
    for split in (0, 1, 3):
        r = F.sor(x, 4, 1.1, lengths=lengths, col_split=split)
        torch.cuda.synchronize()
        assert_sample_equals_alone(r, x, 0, 900, 4, 1.1)
        n, kept = r.lengths.cpu().numpy(), r.kept_idx.cpu().numpy()
        assert ((n >= 0) & (n <= lengths.cpu().numpy())).all()
        assert ((kept >= -1) & (kept < 1000)).all()
        check_consistent(r.keep.cpu().numpy(), kept, n)
