"""GPU: AOF's low-frequency projection (functional.low_pass, pcd_low_pass) equals the float32 oracle bit for bit whatever
the batch, the layout or the split, agrees with float64, passes gradcheck, keeps samples apart; low_frequency_basis is
orthonormal; AOFAttack equals the reference-shaped host loop at B = 1, replays as a graph what it runs eagerly, keeps
samples apart, launches the projection twice per iteration, is CWAttack at gamma = 0, and flips the tiny victim."""
import importlib
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from oracle import aof_oracle as O

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F, CL = pcd.functional, pcd.cw_loop
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tiny_victim  # noqa: E402


def same_bits(a, b):
    """bit-equal, except that any NaN equals any NaN (payloads differ between the GPU and numpy)"""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and (na == nb).all() and (a[~na].view(np.uint32) == b[~nb].view(np.uint32)).all()


def orthonormal_basis(B, Kl, N, seed):
    rng = np.random.default_rng(seed)
    q = np.linalg.qr(rng.standard_normal((B, N, Kl)))[0]
    return np.ascontiguousarray(np.swapaxes(q, 1, 2)).astype(np.float32)


def gaussian_basis(B, Kl, N, seed):
    """rows of unit expected norm with entries spread over six decades: the bits, not the geometry, are under test"""
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((B, Kl, N)) * 10.0 ** rng.uniform(-3, 3, (B, Kl, 1)) / np.sqrt(N)).astype(np.float32)


def layout(x, channel_first):
    t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return t.transpose(1, 2).contiguous().transpose(1, 2) if channel_first else t.contiguous()


def run(V, x, channel_first=False, split=None):
    y = F.low_pass(layout(x, channel_first), torch.from_numpy(V).cuda(), split=split)
    assert y.stride() == layout(x, channel_first).stride()          # x's layout
    return y.cpu().numpy()


@pytest.mark.parametrize("N", [256, 1024, 16384])
@pytest.mark.parametrize("B", [1, 3, 32])
@pytest.mark.parametrize("Kl", [1, 100, "N"])
def test_equals_the_float32_oracle_bit_for_bit(Kl, B, N):
    if Kl == "N":
        if N > 1024:
            pytest.skip("a full basis only up to N = 1024")
        Kl = N
    V = gaussian_basis(B, Kl, N, seed=B + N + Kl)
    x = np.random.default_rng(N).uniform(-1, 1, (B, N, 3)).astype(np.float32)
    want = O.low_pass(V, x)
    for channel_first in (False, True):
        for split in (None, 1, 2, 4, 8, 16):
            assert same_bits(run(V, x, channel_first, split), want), (channel_first, split)


def test_agrees_with_float64_and_passes_gradcheck():
    V = orthonormal_basis(3, 100, 1024, seed=1)
    x = synth.face_clouds(3, 1024, seed=5).numpy()
    y = run(V, x)
    y64 = O.low_pass(V, x, dtype=np.float64)
    assert np.abs(y - y64).max() <= 1e-5 * np.abs(y64).max()
    # the backward is the same projection of the incoming gradient, to the bit
    xc = torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 1))).cuda().requires_grad_(True)    # [B,3,N]
    g = torch.randn(x.shape, device="cuda")
    F.low_pass(xc.transpose(1, 2), torch.from_numpy(V).cuda()).backward(g)
    assert same_bits(xc.grad.transpose(1, 2).cpu().numpy(), O.low_pass(V, g.cpu().numpy()))
    # gradcheck in float64 around the fp32 kernel: the map is linear, so a wide step is exact up to fp32 rounding
    Vs = torch.from_numpy(orthonormal_basis(2, 8, 64, seed=2)).cuda()
    x64 = torch.randn(2, 64, 3, dtype=torch.float64, device="cuda", requires_grad=True)
    assert torch.autograd.gradcheck(lambda t: F.low_pass(t.float(), Vs).double(), (x64,), eps=1e-2, atol=1e-4, rtol=1e-3)


def test_samples_are_independent_and_nan_stays_alone():
    B, Kl, N = 32, 100, 1024
    V = gaussian_basis(B, Kl, N, seed=7)
    x = np.random.default_rng(8).uniform(-1, 1, (B, N, 3)).astype(np.float32)
    batch = run(V, x)
    for b in (0, 13, 31):
        assert same_bits(run(V[b:b + 1], x[b:b + 1]), batch[b:b + 1]), b
    xn, Vn = x.copy(), V.copy()
    xn[4, 100, 1] = np.nan
    Vn[9, 50, 7] = np.inf
    out = run(Vn, xn)
    assert np.isnan(out[4]).any() and not np.isfinite(out[9]).all()
    assert same_bits(out, O.low_pass(Vn, xn))
    keep = [b for b in range(B) if b not in (4, 9)]
    assert same_bits(out[keep], batch[keep])
    # a basis shared over the batch through a stride-0 view
    shared = torch.from_numpy(V[:1]).cuda().expand(B, -1, -1)
    got = F.low_pass(layout(x, False), shared).cpu().numpy()
    assert same_bits(got, O.low_pass(np.broadcast_to(V[:1], V.shape), x))


def test_one_eigenvector_gives_the_centroid():
    ori = synth.face_clouds(2, 1024, seed=3).cuda()
    L = pcd.taof.laplacian_from_pc(ori.transpose(1, 2), 30).double()
    assert (torch.linalg.eigvalsh(L)[:, 1] > 1e-6).all()               # the 30-NN graph is connected
    V = pcd.taof.low_frequency_basis(ori.transpose(1, 2), 1)
    y = F.low_pass(ori, V)
    centroid = ori.double().mean(1, keepdim=True)
    assert (y.double() - centroid).abs().max().item() <= 1e-5


def test_low_frequency_basis_is_orthonormal():
    ori = synth.face_clouds(2, 1024, seed=4).cuda()
    V = pcd.taof.low_frequency_basis(ori.transpose(1, 2), 100)
    assert V.shape == (2, 100, 1024) and V.dtype == torch.float32 and V.is_contiguous()
    gram = V.double() @ V.double().transpose(1, 2)
    assert (gram - torch.eye(100, dtype=torch.float64, device="cuda")).abs().max().item() <= 1e-6
    with pytest.raises(ValueError):
        pcd.taof.low_frequency_basis(ori.transpose(1, 2), 1025)


# ---------------------------------------------------------------------------------------------------------- the loop
N_LOOP, KL_LOOP = 512, 100


def victim_and_data(B, seed=0):
    model = tiny_victim.make(seed).cuda()
    x = synth.face_clouds(B, N_LOOP, seed=seed + 100).cuda()
    with torch.no_grad():
        label = model(x.transpose(1, 2))[0].argmax(1)
    return model, x, label


def make(model, gamma=0.25, use_graph=False, cls=None, **kw):
    args = dict(gamma=gamma, low_pass=KL_LOOP, attack_lr=1e-2, init_weight=10., max_weight=80., binary_step=2,
                num_iter=20, clip_func=CL.ClipPointsLinf(0.18), use_graph=use_graph)
    args.update(kw)
    return (cls or pcd.taof.AOFAttack)(model, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.L2Dist(), **args)


def test_device_loop_equals_the_host_loop():
    model, x, label = victim_and_data(1)
    V = torch.from_numpy(orthonormal_basis(1, KL_LOOP, N_LOOP, seed=11)).cuda()
    noise = torch.randn((2, 1, 3, N_LOOP), generator=torch.Generator().manual_seed(12))
    atk = make(model)
    dist, adv, ok = atk.attack(x, label, basis=V, init_noise=noise)
    hd, ha, hok = O.host_loop(model, F.low_pass, x, label, V, CL.UntargetedLogitsAdvLoss(kappa=5.),
                              pcd.dist_utils.L2Dist(), 0.25, noise, binary_step=2, num_iter=20,
                              clip_func=CL.ClipPointsLinf(0.18))
    assert same_bits(dist.cpu().numpy(), hd) and same_bits(adv.cpu().numpy(), ha)
    assert np.array_equal(ok.cpu().numpy(), hok)
    assert float((adv - x).abs().max()) > 1e-3                      # the cloud did move


class _EagerCapturable(pcd.taof.AOFAttack):
    """the graph path's state and optimiser (capturable Adam), with every iteration run eagerly instead of replayed"""

    def _capture(self, st, warmup=3):
        return types.SimpleNamespace(replay=lambda: self._iteration(st))


def test_graph_replay_equals_eager():
    """the graph path uses capturable Adam, which rounds its bias corrections on the device; the plain eager path does
    not, so the graph is compared with eager iterations of the same optimiser"""
    model, x, label = victim_and_data(4)
    V = torch.from_numpy(orthonormal_basis(4, KL_LOOP, N_LOOP, seed=13)).cuda()
    graph = make(model, use_graph=True).attack(x, label, basis=V, seed=5)
    eager = make(model, use_graph=True, cls=_EagerCapturable).attack(x, label, basis=V, seed=5)
    for g, e in zip(graph, eager):
        assert torch.equal(g, e)


def test_samples_are_independent_of_the_batch():
    """The projection is batch-invariant to the bit (test_samples_are_independent_and_nan_stays_alone).  The victim and
    L2Dist are torch ops whose kernels and reduction orders may change with the batch size, so a sample alone is
    compared with the batch within rounding, as CWAttack's graph and eager runs are."""
    model, x, label = victim_and_data(4)
    V = torch.from_numpy(orthonormal_basis(4, KL_LOOP, N_LOOP, seed=14)).cuda()
    dist, adv, ok = make(model).attack(x, label, basis=V, seed=7)
    for b in range(4):
        d1, a1, o1 = make(model).attack(x[b:b + 1], label[b:b + 1], basis=V[b:b + 1], seed=7, first_sample=b)
        assert o1[0] == ok[b] and torch.allclose(d1[0], dist[b], rtol=1e-4), b
        assert (a1[0] - adv[b]).abs().max().item() < 1e-4, b


_COUNT = r"""
import importlib, os, sys
import numpy as np, torch
from torch.profiler import ProfilerActivity, profile
sys.path.insert(0, "."); sys.path.insert(0, "tests")
pcd = importlib.import_module("3dpointcloudattack_b200"); synth = importlib.import_module("3dpointcloudattack_b200.synth")
import tiny_victim
CL = pcd.cw_loop
model = tiny_victim.make(0).cuda()
x = synth.face_clouds(2, 512, seed=100).cuda()
label = torch.tensor([0, 1], device="cuda")
q = np.linalg.qr(np.random.default_rng(15).standard_normal((2, 512, 100)))[0]
V = torch.from_numpy(np.ascontiguousarray(q.transpose(0, 2, 1)).astype(np.float32)).cuda()
atk = pcd.taof.AOFAttack(model, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.L2Dist(), low_pass=100,
                         binary_step=1, num_iter=int(sys.argv[1]), clip_func=CL.ClipPointsLinf(0.18))
atk.attack(x, label, basis=V); torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    atk.attack(x, label, basis=V); torch.cuda.synchronize()
print(sum("low_pass_kernel" in e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA))
"""


def test_two_low_pass_launches_per_iteration():
    """profiled in a fresh process (a profiler session leaves state behind in the one it ran in)"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-s", "-c", _COUNT, "6"], cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert int(r.stdout.split()[-1]) == 2 * 6


def test_gamma_zero_is_cw_bit_for_bit():
    model, x, label = victim_and_data(4)
    kw = dict(attack_lr=1e-2, init_weight=10., max_weight=80., binary_step=2, num_iter=10,
              clip_func=CL.ClipPointsLinf(0.18))
    n0 = F.launches()
    aof = make(model, gamma=0., **kw).attack(x, label, seed=9)
    n_aof = F.launches() - n0
    n0 = F.launches()
    cw = CL.CWAttack(model, CL.UntargetedLogitsAdvLoss(kappa=5.), pcd.dist_utils.L2Dist(), **kw).attack(x, label, seed=9)
    assert F.launches() - n0 == n_aof == 2 * 10                   # the clip only: no basis, no projection
    for a, c in zip(aof, cw):
        assert torch.equal(a, c)


def test_large_budget_flips_most_labels():
    model, x, label = victim_and_data(8)
    atk = make(model, attack_lr=2e-2, init_weight=0.01, max_weight=10., binary_step=1, num_iter=100, clip_func=None)
    dist, adv, ok = atk.attack(x, label)                            # the basis from the eigensolver
    assert ok.float().mean().item() >= 0.75
    assert (dist[ok] < 1e10).all() and (dist[~ok] == 1e10).all() and torch.isfinite(adv).all()
