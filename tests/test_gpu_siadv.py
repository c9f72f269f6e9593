"""GPU: the SI-Adv step kernel (functional.shape_invariant_step_, pcd_si_step) equals the float32 oracle bit for bit on
every output, whatever the batch, the layout or the split; it agrees with the float64 oracle; samples are independent
of their batch and non-finite samples stay alone.  estimate_normals agrees with float64 normals, and SIAdvAttack runs,
eager and captured, with and without a device-sampled defence, at four library launches per iteration."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from oracle import siadv_oracle as O

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F, D = pcd.functional, pcd.defense
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tiny_victim  # noqa: E402

STEP, EPS, SCALE = 0.007, 0.16, float(np.sqrt(3 * 1024))


def unit(v):
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)


def inputs(kind, B, N, seed):
    """(pc, ori, normal, grad) [B,N,3] float32 numpy"""
    rng = np.random.default_rng(seed)
    if kind == "face" and N > 1:      # a one-point face is 0 / 0 after its scaling
        ori = synth.face_clouds(B, N, seed=seed).numpy()
    else:
        ori = rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    pc = (ori + 0.01 * rng.standard_normal((B, N, 3))).astype(np.float32)
    normal = unit(rng.standard_normal((B, N, 3)))
    if kind == "boundary":           # z = +-1 exactly, and |z^2 - 1| just under and just over 1e-4
        m = rng.integers(0, 4, (B, N))
        d = np.array([0.0, 0.0, 0.97e-4, 1.03e-4])[m]
        z = np.sqrt(1 - d) * np.where(rng.random((B, N)) < 0.5, -1, 1)
        phi = rng.uniform(0, 2 * np.pi, (B, N))
        r = np.sqrt(d)
        nb = np.stack([r * np.cos(phi), r * np.sin(phi), z], -1).astype(np.float32)
        normal = np.where((rng.random((B, N)) < 0.7)[..., None], nb, normal)
    # gradients of unequal scale per sample, sparse in places (a max-pooled victim's gradient is)
    grad = (rng.standard_normal((B, N, 3)) * 10.0 ** rng.uniform(-3, 1, (B, 1, 1))).astype(np.float32)
    grad[rng.random((B, N)) < 0.5] = 0
    return pc, ori, normal, grad


def same_bits(a, b):
    """bit-equal, except that any NaN equals any NaN (payloads differ between the GPU and numpy)"""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and (na == nb).all() and (a[~na].view(np.uint32) == b[~nb].view(np.uint32)).all()


def layout(x, channel_first):
    t = torch.from_numpy(x).cuda()
    return t.transpose(1, 2).contiguous().transpose(1, 2) if channel_first else t.contiguous()


def run(pc, ori, normal, grad, eps=EPS, split=0, channel_first=False, step=STEP):
    p = layout(pc, channel_first)
    g = F.shape_invariant_step_(p, layout(ori, channel_first), layout(normal, channel_first), layout(grad, channel_first),
                                step, eps, SCALE, split=split)
    return p.cpu().numpy(), g.cpu().numpy()


def splits(N):
    return [0] + [s for s in (1, 2, 4, 8, 16) if s * 2048 >= N]


@pytest.mark.parametrize("N", [1, 31, 1024, 4096, 16384])
@pytest.mark.parametrize("B", [1, 3, 32])
@pytest.mark.parametrize("kind", ["face", "uniform", "boundary"])
def test_equals_the_float32_oracle_bit_for_bit(kind, B, N):
    pc, ori, normal, grad = inputs(kind, B, N, seed=B * 7 + N)
    eps = EPS if kind != "uniform" else 1.0               # the clip active, and mostly not
    want, wnorm = O.si_step(pc, ori, normal, grad, STEP, eps, SCALE)
    for channel_first in (False, True):
        for split in splits(N):
            out, gnorm = run(pc, ori, normal, grad, eps, split, channel_first)
            assert same_bits(out, want), (channel_first, split)
            assert same_bits(gnorm, wnorm), (channel_first, split)


@pytest.mark.parametrize("kind", ["face", "uniform", "boundary"])
def test_agrees_with_the_float64_oracle(kind):
    """fp32 roundings only: within 1e-4 of the float64 steps on unit-scale clouds, the gradient norm within 1e-5.  The
    bound is set by normals near the poles: den = sqrt(1 - z*z) keeps few digits there, and the frame's error grows as
    one ulp / (1 - z*z), in the reference's formula as much as here (1.5e-5 is typical with random unit normals)."""
    pc, ori, normal, grad = inputs(kind, 3, 1024, seed=5)
    out, gnorm = run(pc, ori, normal, grad)
    want, wnorm = O.si_step(pc, ori, normal, grad, STEP, EPS, SCALE, dtype=np.float64)
    assert np.abs(out - want).max() < 1e-4
    assert np.abs(gnorm - wnorm).max() < 1e-5 * wnorm.max()


def test_sample_does_not_depend_on_its_batch():
    """B = 64 in one CTA per sample against each sample alone in a cluster"""
    pc, ori, normal, grad = inputs("face", 64, 1024, seed=9)
    for split in (1, 0):
        batch, bnorm = run(pc, ori, normal, grad, split=split)
        for b in (0, 17, 63):
            alone, anorm = run(pc[b:b + 1], ori[b:b + 1], normal[b:b + 1], grad[b:b + 1])
            assert same_bits(batch[b:b + 1], alone) and same_bits(bnorm[b:b + 1], anorm), (split, b)


def test_non_finite_samples_stay_alone_and_zero_gradient_moves_nothing():
    pc, ori, normal, grad = inputs("face", 5, 1024, seed=11)
    grad[1, 100, 0] = np.nan
    normal[2, 7] = [np.inf, 0, 0]
    grad[3] = 0
    pc[3] = ori[3]
    # sample 3's normals keep |z| <= 0.9: near the poles den = sqrt(1 - z*z) keeps few digits and the frame's round trip
    # (the explicit inverse transform of the contract) is exact only to about one ulp / (1 - z*z)
    rng = np.random.default_rng(3)
    z, phi = rng.uniform(-0.9, 0.9, 1024), rng.uniform(0, 2 * np.pi, 1024)
    normal[3] = np.stack([np.sqrt(1 - z * z) * np.cos(phi), np.sqrt(1 - z * z) * np.sin(phi), z], -1)
    out, gnorm = run(pc, ori, normal, grad)
    want, wnorm = O.si_step(pc, ori, normal, grad, STEP, EPS, SCALE)
    assert same_bits(out, want) and same_bits(gnorm, wnorm)
    assert np.isnan(out[1]).all() and np.isnan(out[2]).all() and np.isnan(gnorm[1:3]).all()
    assert np.isfinite(out[[0, 3, 4]]).all() and np.isfinite(gnorm[[0, 3, 4]]).all()
    # a zero gradient: zero norm and a zero step, bit for bit the same as no step at all ...
    still, snorm = run(pc, ori, normal, grad, step=0.0)
    assert gnorm[3] == 0 and snorm[3] == 0 and same_bits(out[3], still[3])
    # ... so the points move only by the rounding of the round trip through their frames
    assert np.abs(out[3] - pc[3]).max() < 2e-6


def test_empty_batch_is_a_no_op():
    x = torch.zeros(0, 16, 3, device="cuda")
    assert F.shape_invariant_step_(x, x.clone(), x.clone(), x.clone(), STEP, EPS).shape == (0,)


@pytest.mark.parametrize("channel_first", [False, True])
def test_estimate_normals_against_float64(channel_first):
    """|cos| >= 1 - 1e-4 wherever the 20th and 21st neighbours are apart and the patch has a well-defined normal"""
    pc = synth.face_clouds(2, 1024, seed=21).numpy()
    n = F.estimate_normals(layout(pc, channel_first), 20).cpu().numpy()
    ref, gap, w = O.normals64(pc, 20)
    ok = (gap > 1e-5 * w[..., 2]) & (w[..., 1] > 10 * w[..., 0])
    assert ok.mean() > 0.9
    cos = np.abs((n.astype(np.float64) * ref).sum(-1))
    assert cos[ok].min() >= 1 - 1e-4
    assert np.abs(np.linalg.norm(n, axis=-1) - 1).max() < 1e-5


# ---------------------------------------------------------------------------------------------------------- the loop
def victim_and_data(B, N=1024, seed=0):
    model = tiny_victim.make(seed).cuda()
    x = synth.face_clouds(B, N, seed=seed + 100).cuda()
    with torch.no_grad():
        label = model(x.transpose(1, 2))[0].argmax(1)
    return model, x, label


def margin(model, x, label):
    with torch.no_grad():
        return pcd.siadv.SIAdvAttack(model)._loss(model(x.transpose(1, 2))[0], label).item()


@pytest.mark.parametrize("eps, step_size, steps, must_succeed", [(0.16, 0.007, 50, False), (2.0, 0.05, 30, True)])
def test_attack_lowers_the_loss_and_mostly_succeeds(eps, step_size, steps, must_succeed):
    """The reference's budget (eps = 0.16 on each axis's norm over the whole cloud) lowers the margin of the tiny victim,
    whose weights are scaled up threefold, by about a tenth in 50 steps without flipping a label; a larger budget flips
    most of them."""
    model, x, label = victim_and_data(8)
    atk = pcd.siadv.SIAdvAttack(model, eps=eps, step_size=step_size, max_steps=steps)
    adv, pred, success = atk.attack(x, label)
    assert adv.shape == x.shape and torch.isfinite(adv).all()
    before, after = margin(model, x, label), margin(model, adv, label)
    assert after < before
    if must_succeed:
        assert after < 0.5 * before and success.float().mean().item() >= 0.5
    assert torch.equal(success, pred != label)
    d = (adv - x).norm(dim=1)                             # the per-axis clip: each axis's norm over the cloud <= eps
    assert d.max().item() <= eps * (1 + 1e-5)


def test_graph_replay_equals_eager_and_counts_launches():
    model, x, label = victim_and_data(4)
    n0 = F.launches()
    eager = pcd.siadv.SIAdvAttack(model, max_steps=10).attack(x, label)
    assert F.launches() - n0 == 3 + 4 * 10             # the initial normals, then step + k-NN (2) + frames per iteration
    with_normals = torch.cat([x, torch.from_numpy(O.normals64(x.cpu().numpy(), 20)[0]).float().cuda() * 2], -1)
    n0 = F.launches()
    pcd.siadv.SIAdvAttack(model, max_steps=10).attack(with_normals, label)
    assert F.launches() - n0 == 4 * 10                 # given normals: no initial estimate
    graph = pcd.siadv.SIAdvAttack(model, max_steps=10, use_graph=True).attack(x, label)
    assert torch.equal(eager[0], graph[0]) and torch.equal(eager[1], graph[1])


def test_samples_are_independent_of_the_batch():
    model, x, label = victim_and_data(4)
    adv, pred, _ = pcd.siadv.SIAdvAttack(model, max_steps=10).attack(x, label)
    for b in range(4):
        a1, p1, _ = pcd.siadv.SIAdvAttack(model, max_steps=10).attack(x[b:b + 1], label[b:b + 1])
        assert torch.equal(a1[0], adv[b]) and p1[0] == pred[b], b


@pytest.mark.parametrize("defence", ["srs", "sor"])
def test_attack_through_a_device_sampled_defence(defence):
    model, x, label = victim_and_data(4)
    runs = []
    for use_graph in (False, True):
        sampler = F.PointSampler(1234, device="cuda")
        pre = D.SRSDefense(200, sampler=sampler) if defence == "srs" else D.SORDefense(2, 1.1, 1024, sampler=sampler)
        atk = pcd.siadv.SIAdvAttack(D.DefendedVictim(model, pre), max_steps=6, eval_model=model, use_graph=use_graph)
        adv, pred, success = atk.attack(x, label)
        assert torch.isfinite(adv).all() and torch.equal(success, pred != label)
        assert int(sampler.counter.item()) == 6          # one draw per iteration; warm-up and capture leave no trace
        runs.append((adv, pred))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
