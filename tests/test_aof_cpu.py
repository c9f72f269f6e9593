"""AOF without a GPU: the float32 order of pcd_low_pass against float64, the projector's idempotence and symmetry, the
full basis giving x back, the argument errors of pcd_low_pass that come before any CUDA call, the attack's argument
checks, and dist_utils.L2Dist against its formula."""
import ctypes
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from oracle import aof_oracle as O

pcd = importlib.import_module("3dpointcloudattack_b200")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tiny_victim  # noqa: E402


def orthonormal_basis(B, Kl, N, seed):
    """[B,Kl,N] float32 with orthonormal rows (float64 QR of a Gaussian matrix)"""
    rng = np.random.default_rng(seed)
    q = np.linalg.qr(rng.standard_normal((B, N, Kl)))[0]
    return np.ascontiguousarray(np.swapaxes(q, 1, 2)).astype(np.float32)


def cloud(B, N, seed):
    return np.random.default_rng(seed).uniform(-1, 1, (B, N, 3)).astype(np.float32)


@pytest.mark.parametrize("B, Kl, N", [(2, 1, 37), (3, 10, 256), (1, 100, 1024), (1, 64, 64)])
def test_float32_order_agrees_with_float64(B, Kl, N):
    V, x = orthonormal_basis(B, Kl, N, seed=N + Kl), cloud(B, N, seed=Kl)
    y32 = O.low_pass(V, x)
    y64 = O.low_pass(V, x, dtype=np.float64)
    assert y32.dtype == np.float32 and y32.shape == x.shape
    assert np.abs(y32 - y64).max() <= 1e-5 * np.abs(y64).max()


def test_lane_order_is_the_stated_one():
    """one row, one channel, written out: lane sums in ascending n, then the xor butterfly"""
    N = 100
    rng = np.random.default_rng(4)
    V = (rng.standard_normal((1, 1, N)) * 10.0 ** rng.uniform(-3, 3, N)).astype(np.float32)
    x = (rng.standard_normal((1, N, 3)) * 10.0 ** rng.uniform(-3, 3, (N, 1))).astype(np.float32)
    lanes = np.zeros(32, np.float32)
    for n in range(N):
        lanes[n % 32] = lanes[n % 32] + V[0, 0, n] * x[0, n, 1]
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[np.arange(32) ^ o]
    assert (lanes == lanes[0]).all()                     # every lane ends with the same total
    want = np.float32(0) + V[0, 0] * lanes[0]
    assert np.array_equal(O.low_pass(V, x)[0, :, 1].view(np.uint32), want.view(np.uint32))


def test_projector_is_idempotent_and_symmetric():
    B, Kl, N = 2, 100, 512
    V = orthonormal_basis(B, Kl, N, seed=1)
    x, z = cloud(B, N, seed=2), cloud(B, N, seed=3)
    px = O.low_pass(V, x)
    ppx = O.low_pass(V, px)
    assert np.abs(ppx - px).max() <= 1e-5 * np.abs(px).max()
    lhs = (px.astype(np.float64) * z).sum(axis=1)                                  # <P x, z> per channel
    rhs = (x.astype(np.float64) * O.low_pass(V, z)).sum(axis=1)                    # <x, P z>
    assert np.abs(lhs - rhs).max() <= 1e-5 * np.abs(lhs).max()


@pytest.mark.parametrize("N", [1, 33, 256])
def test_full_basis_gives_x_back(N):
    V, x = orthonormal_basis(2, N, N, seed=N), cloud(2, N, seed=N + 1)
    assert np.abs(O.low_pass(V, x) - x).max() <= 1e-5


def test_low_pass_argument_errors():
    lib = pcd._lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every call below fails its argument check

    def call(basis=fake, b_sb=16 * 4, Kl=4, x=fake, B=2, N=16, y=fake, split=0):
        return lib.pcd_low_pass(basis, b_sb, Kl, x, 48, 3, 1, B, N, y, 48, 3, 1, split, None)

    assert call(basis=None) == 1
    assert call(x=None) == 1
    assert call(y=None) == 1
    assert call(N=0) == 1
    assert call(B=-1) == 1
    assert call(Kl=0) == 1 and call(Kl=17) == 1                               # 1 <= Kl <= N
    assert call(b_sb=-1) == 1
    assert call(split=3) == 1 and call(split=32) == 1 and call(split=-1) == 1
    assert b"pcd_low_pass" in lib.pcd_last_error()
    assert call(N=16385, Kl=100) == 4                                         # PCD_ERR_UNSUPPORTED
    assert b"16384" in lib.pcd_last_error()
    assert call(B=0) == 0 and call(B=0, basis=None, x=None, y=None) == 0     # an empty batch is a no-op


def test_attack_checks_its_arguments():
    CL = pcd.cw_loop
    model = tiny_victim.make(0)
    adv_func, dist = CL.UntargetedLogitsAdvLoss(kappa=0.), pcd.dist_utils.L2Dist()
    for gamma in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            pcd.taof.AOFAttack(model, adv_func, dist, gamma=gamma)
    with pytest.raises(ValueError):
        pcd.taof.AOFAttack(model, adv_func, dist, low_pass=0)
    atk = pcd.taof.AOFAttack(model, adv_func, dist)
    assert atk.gamma == 0.25 and atk.low_pass == 100
    with pytest.raises(RuntimeError, match="CUDA"):
        atk.attack(torch.zeros(1, 128, 3), torch.zeros(1, dtype=torch.long))


def test_l2dist_is_its_formula():
    rng = np.random.default_rng(5)
    a, o = rng.standard_normal((4, 50, 3)), rng.standard_normal((4, 50, 3))
    w = np.array([1., 2., 0.5, 3.])
    want = np.sqrt(((a - o) ** 2).sum(axis=(1, 2))) * w
    L2 = pcd.dist_utils.L2Dist()
    at, ot = torch.from_numpy(a).float(), torch.from_numpy(o).float()
    got = L2(at, ot, torch.from_numpy(w), batch_avg=False)
    assert got.shape == (4,) and np.allclose(got.numpy(), want, rtol=1e-6)
    assert np.isclose(L2(at, ot, torch.from_numpy(w)).item(), want.mean(), rtol=1e-6)
    assert np.allclose(L2(at, ot, batch_avg=False).numpy(), want / w, rtol=1e-6)    # no weights: ones
    assert np.allclose(L2(at.transpose(1, 2), ot.transpose(1, 2), batch_avg=False).numpy(), want / w, rtol=1e-6)
