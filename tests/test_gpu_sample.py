"""GPU: the device point sampler (functional.sample_points, pcd_sample_points) and the defences built on it.  The draws
equal the numpy oracle bit for bit, whatever the batch, the padding or the sharding; the counter advances once per call,
in eager runs and graph replays alike; the draws are uniform; the device-sampled SOR and SRS defences are the oracle on
the kernels' own kept indices and carry the gradient to exactly the drawn points; attacks run through a defended victim,
eager and captured."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from oracle import sample_oracle as S
from test_sample_cpu import chi_square_over_tuples

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F, D, CL = pcd.functional, pcd.defense, pcd.cw_loop
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tiny_victim  # noqa: E402

NS = [0, 1, 2, 5, 1000, 1023, 1024, 1025, 4096, 10000, 16384]
NPOINTS = [1, 3, 524, 1024, 4096]
SEED = 0x9E3779B97F4A7C15


def counter(sampler):
    return int(sampler.counter.item())


def draw(lengths, N, npoint, sampler, table=None):
    """sample_points on the device and the oracle from the counter before the call -> (device, oracle) as numpy"""
    c = counter(sampler)
    n = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    out = F.sample_points(n, N, npoint, sampler, table=None if table is None else torch.from_numpy(table).cuda())
    ref = S.sample_points([min(max(v, 0), N) for v in lengths], npoint, sampler.seed, c, sampler.first_sample, table)
    return out.cpu().numpy(), ref


def random_table(B, N, seed):
    rng = np.random.default_rng(seed)
    return np.stack([rng.permutation(N) for _ in range(B)]).astype(np.int32)


@pytest.mark.parametrize("npoint", NPOINTS)
@pytest.mark.parametrize("with_table", [False, True])
def test_equals_the_oracle_bit_for_bit(npoint, with_table):
    s = F.PointSampler(SEED, device="cuda")
    # every n in one padded batch (the largest size class) ...
    N = max(NS)
    out, ref = draw(NS, N, npoint, s, random_table(len(NS), N, 1) if with_table else None)
    assert np.array_equal(out, ref)
    # ... and every n alone at N = n, the smallest size class that holds it
    for n in NS:
        Nn = max(n, 1)
        out, ref = draw([n], Nn, npoint, s, random_table(1, Nn, n) if with_table else None)
        assert np.array_equal(out, ref), n
    assert counter(s) == 1 + len(NS)


def test_lengths_none_and_clamping():
    s = F.PointSampler(3, device="cuda")
    c = counter(s)
    out = F.sample_points(None, 2000, 1024, s, table=torch.zeros(4, 2000, dtype=torch.int64, device="cuda")
                          + torch.arange(2000, device="cuda"))
    assert np.array_equal(out.cpu().numpy(), S.sample_points([2000] * 4, 1024, 3, c))
    for dtype in (torch.int64, torch.int32):
        c = counter(s)
        out = F.sample_points(torch.tensor([-5, 3000, 700], dtype=dtype, device="cuda"), 2000, 1024, s)
        assert np.array_equal(out.cpu().numpy(), S.sample_points([0, 2000, 700], 1024, 3, c))


def test_counter_advances_once_per_call_and_draws_differ():
    s = F.PointSampler(5, device="cuda")
    n = torch.full((64,), 1000, dtype=torch.int32, device="cuda")
    outs = []
    for call in range(4):
        assert counter(s) == call and int(s.state[1]) == 0
        outs.append(F.sample_points(n, 1024, 512, s))
    assert counter(s) == 4
    for a in range(4):
        for b in range(a + 1, 4):
            assert not torch.equal(outs[a], outs[b])
    s.reset(2)
    assert torch.equal(F.sample_points(n, 1024, 512, s), outs[2])
    s.reset(2 ** 40 + 7)                  # the counter's high word takes part
    c = counter(s)
    out = F.sample_points(n[:2], 1024, 512, s)
    assert c == 2 ** 40 + 7 and np.array_equal(out.cpu().numpy(), S.sample_points([1000] * 2, 512, 5, c))


def test_draws_do_not_depend_on_the_batch_padding_or_sharding():
    lengths = [900, 1000, 37, 1024, 0, 513, 1000, 4]
    npoint = 700
    s = F.PointSampler(11, device="cuda")
    whole = F.sample_points(torch.tensor(lengths, device="cuda"), 1024, npoint, s)
    # sharded: two calls of four, with first_sample 0 and 4, from the same counter
    s0, s4 = F.PointSampler(11, 0, device="cuda"), F.PointSampler(11, 4, device="cuda")
    a = F.sample_points(torch.tensor(lengths[:4], device="cuda"), 1024, npoint, s0)
    b = F.sample_points(torch.tensor(lengths[4:], device="cuda"), 1024, npoint, s4)
    assert torch.equal(whole, torch.cat([a, b]))
    # padding: the same samples in a larger N (another size class)
    assert torch.equal(whole, F.sample_points(torch.tensor(lengths, device="cuda"), 16000, npoint, s.reset(0)))
    # batch position: sample 5 alone is sample 5 of the batch when its global id is 5
    one = F.sample_points(torch.tensor([lengths[5]], device="cuda"), 1024, npoint, F.PointSampler(11, 5, device="cuda"))
    assert torch.equal(one[0], whole[5])
    # B: the first three samples as a batch of three
    assert torch.equal(F.sample_points(torch.tensor(lengths[:3], device="cuda"), 1024, npoint, s.reset(0)), whole[:3])


def test_device_draws_are_uniform():
    s = F.PointSampler(12, device="cuda")
    out = F.sample_points(torch.full((60000,), 5, device="cuda"), 16, 3, s).cpu().numpy()
    assert chi_square_over_tuples(out, 5, 3) > 1e-4
    out = F.sample_points(torch.full((60000,), 5, device="cuda"), 5, 13, s).cpu().numpy()
    assert (out[:, :10] == np.tile(np.arange(5), 2)).all()
    assert chi_square_over_tuples(out[:, 10:], 5, 3) > 1e-4


def test_graph_replays_equal_eager_calls():
    lengths = torch.tensor([1000, 700, 1024, 3, 0, 999], device="cuda")
    s = F.PointSampler(13, device="cuda")
    F.sample_points(lengths, 1024, 1024, s)                   # opt-in and module load outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = F.sample_points(lengths, 1024, 1024, s)
    s.reset(0)
    replays = []
    for _ in range(3):
        g.replay()
        replays.append(out.clone())
    assert counter(s) == 3
    s.reset(0)
    for r in replays:
        assert torch.equal(r, F.sample_points(lengths, 1024, 1024, s))
    assert not torch.equal(replays[0], replays[1])


# ------------------------------------------------------------------------------------------------ defences
def noisy_faces(B, N, seed):
    pc = synth.face_clouds(B, N, seed=seed)
    return (pc + 0.01 * torch.randn(pc.shape, generator=torch.Generator().manual_seed(seed))).cuda()


def defended_reference(x, lengths, npoint, sampler, c):
    """the oracle's draws through functional.sor's kept indices, and the gathered points (NaN where nothing is kept)"""
    r = F.sor(x, 2, 1.1, lengths)
    idx = S.sample_points(r.lengths.cpu().tolist(), npoint, sampler.seed, c, sampler.first_sample,
                          r.kept_idx.cpu().numpy())
    xs = x.detach().cpu().numpy()
    pts = np.where((idx < 0)[..., None], np.nan, np.take_along_axis(xs, np.maximum(idx, 0)[..., None], 1))
    return idx, pts, r


@pytest.mark.parametrize("B, N, lengths", [(4, 1024, None), (4, 1024, [1024, 700, 2, 513]), (3, 4096, [4096, 1500, 10])])
def test_sor_defense_equals_the_oracle_on_the_kept_indices(B, N, lengths):
    x = noisy_faces(B, N, seed=B + N)
    lt = None if lengths is None else torch.tensor(lengths, device="cuda")
    s = F.PointSampler(17, device="cuda")
    c = counter(s)
    y = D.SORDefense(npoint=1024, sampler=s)(x, lt)
    idx, pts, r = defended_reference(x, lt, 1024, s, c)
    assert y.shape == (B, 1024, 3) and counter(s) == c + 1
    assert np.array_equal(y.cpu().numpy(), pts, equal_nan=True)
    for b in range(B):
        if int(r.lengths[b]) == 0:
            assert torch.isnan(y[b]).all()
        else:
            assert torch.isfinite(y[b]).all()


def test_gradient_reaches_exactly_the_drawn_points():
    B, N, npoint = 4, 1024, 1024
    x = noisy_faces(B, N, seed=21).requires_grad_(True)
    lt = torch.tensor([1024, 900, 2, 1024], device="cuda")
    s = F.PointSampler(19, device="cuda")
    c = counter(s)
    y = D.SORDefense(npoint=npoint, sampler=s)(x, lt)
    up = torch.randn(y.shape, generator=torch.Generator().manual_seed(0)).cuda()
    (torch.nan_to_num(y) * up).sum().backward()
    idx, _, r = defended_reference(x, lt, npoint, s, c)
    ref = np.zeros((B, N, 3))
    upn = up.cpu().numpy().astype(np.float64)
    for b in range(B):
        for j in range(npoint):
            if idx[b, j] >= 0:
                ref[b, idx[b, j]] += upn[b, j]
    g = x.grad.cpu().numpy()
    assert np.abs(g - ref).max() <= 1e-6 * np.abs(ref).max()
    removed = ~r.keep.cpu().numpy()
    assert (g[removed] == 0).all() and removed.any()
    assert (g[2] == 0).all()                                   # nothing kept: no gradient at all


def test_srs_defense_both_modes():
    x = noisy_faces(5, 1024, seed=23)
    # numpy mode: the published loop under np.random.seed
    np.random.seed(3)
    y = D.SRSDefense(drop_num=500)(x)
    np.random.seed(3)
    xs = x.cpu().numpy()
    ref = np.stack([xs[b][np.random.choice(1024, 524, replace=False)] for b in range(5)])
    assert np.array_equal(y.cpu().numpy(), ref)
    # device mode: the sampler with no table
    s = F.PointSampler(29, device="cuda")
    c = counter(s)
    xg = x.clone().requires_grad_(True)
    y = D.SRSDefense(drop_num=500, sampler=s)(xg)
    idx = S.sample_points([1024] * 5, 524, 29, c)
    assert np.array_equal(y.detach().cpu().numpy(), np.take_along_axis(xs, idx[..., None], 1))
    y.sum().backward()
    drawn = np.zeros((5, 1024), bool)
    np.put_along_axis(drawn, idx, True, 1)
    assert (xg.grad.cpu().numpy()[drawn] == 1).all() and (xg.grad.cpu().numpy()[~drawn] == 0).all()
    assert D.SRSDefense(drop_num=0, sampler=s)(x).shape == (5, 1024, 3)


# ------------------------------------------------------------------------------------------- attacks through SOR
def defended_tiny(seed, sampler):
    victim = tiny_victim.make(seed).cuda()
    for p in victim.parameters():
        p.requires_grad_(False)
    return D.DefendedVictim(victim, D.SORDefense(npoint=512, sampler=sampler))


def test_victim_gradient_is_zero_on_removed_points():
    s = F.PointSampler(31, device="cuda")
    model = defended_tiny(0, s)
    x = noisy_faces(3, 512, seed=31)
    adv = x.transpose(1, 2).contiguous().requires_grad_(True)
    c = counter(s)
    logits = model(adv)[0]
    CL.UntargetedLogitsAdvLoss(kappa=5.)(logits, torch.tensor([0, 1, 2], device="cuda")).backward()
    keep = F.sor(x, 2, 1.1).keep
    g = adv.grad.transpose(1, 2)
    assert (g[~keep] == 0).all() and (~keep).any()
    assert g.abs().sum() > 0 and counter(s) == c + 1


def test_captured_defended_step_equals_eager_steps():
    """one forward and backward of DefendedVictim captured; after a counter reset the replays equal eager calls: the
    same points reach the victim (the same gradient support), and the victim's float32 arithmetic agrees"""
    s = F.PointSampler(37, device="cuda")
    model = defended_tiny(1, s)
    x = noisy_faces(4, 512, seed=37).transpose(1, 2).contiguous()
    target = torch.tensor([0, 1, 2, 3], device="cuda")
    adv = x.clone().requires_grad_(True)
    loss_fn = CL.UntargetedLogitsAdvLoss(kappa=5.)

    def step():
        adv.grad = None if adv.grad is None else adv.grad.zero_()
        logits = model(adv)[0]
        loss = loss_fn(logits, target, reduce=False).sum()
        loss.backward()
        return logits.detach(), loss.detach()

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        logits_g, loss_g = step()
    s.reset(0)
    replays = []
    for _ in range(3):
        g.replay()
        replays.append((logits_g.clone(), adv.grad.clone()))
    assert counter(s) == 3
    s.reset(0)
    for lg, gg in replays:
        le, _ = step()
        assert torch.equal(gg != 0, adv.grad != 0)
        torch.testing.assert_close(lg, le, rtol=1e-6, atol=1e-6)
        torch.testing.assert_close(gg, adv.grad, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("use_graph", [False, True])
def test_cw_attack_through_sor(use_graph):
    s = F.PointSampler(41, device="cuda")
    model = defended_tiny(2, s)
    data = noisy_faces(4, 512, seed=41)
    target = torch.tensor([0, 1, 2, 3], device="cuda")
    atk = CL.CWAttack(model, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.ChamferDist(method="adv2ori"),
                      attack_lr=1e-2, binary_step=2, num_iter=10, clip_func=CL.ClipPointsLinf(0.1), use_graph=use_graph)
    dist, adv, ok = atk.attack(data, target)
    assert adv.shape == data.shape and torch.isfinite(adv).all() and torch.isfinite(dist).all()
    assert counter(s) >= 20


@pytest.mark.parametrize("use_graph", [False, True])
def test_knn_attack_through_sor(use_graph):
    s = F.PointSampler(43, device="cuda")
    model = defended_tiny(3, s)
    data = noisy_faces(4, 512, seed=43)
    target = torch.tensor([0, 1, 2, 3], device="cuda")
    atk = CL.KNNAttack(model, CL.UntargetedLogitsAdvLoss(kappa=15.), pcd.dist_utils.ChamferDist(method="adv2ori"),
                       CL.ProjectInnerClipLinf(0.1), attack_lr=1e-3, num_iter=10, use_graph=use_graph)
    losses = []
    orig = atk._iteration

    def tracked(st):
        orig(st)
        losses.append(st["loss"].clone())
    if not use_graph:
        atk._iteration = tracked
    adv, ok = atk.attack(data, target)
    assert adv.shape == data.shape and torch.isfinite(adv).all()
    assert all(torch.isfinite(v) for v in losses)
    assert counter(s) >= 10
