"""SOR defence without a GPU: the float64 brute force against two independent formulations, the resampling draws
against a literal transcription of the reference's loop, argument errors of the C ABI, and the CUDA-only guard."""
import ctypes
import importlib

import numpy as np
import pytest
import torch

from oracle import sor_oracle as O

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")


def noisy_faces(B, N, seed):
    pc = synth.face_clouds(B, N, seed=seed)
    return (pc + 0.01 * torch.randn(pc.shape, generator=torch.Generator().manual_seed(seed))).numpy()


def direct_sor64(pc, k, alpha):
    """(a - b)^2 summed per channel, a different rounding path from the contract's expansion form."""
    p = pc.astype(np.float64)
    d = ((p[:, :, None, :] - p[:, None, :, :]) ** 2).sum(-1)
    value = np.sort(d, axis=-1)[..., 1:k + 1].mean(-1)
    return value, *O.sor64_threshold(value, alpha)


def assert_sor_agrees(value, threshold, keep, ref_value, ref_threshold, ref_keep, band):
    np.testing.assert_allclose(value, ref_value, rtol=1e-10, atol=0)
    np.testing.assert_allclose(threshold, ref_threshold, rtol=1e-10, atol=0)
    outside = np.abs(ref_value - ref_threshold[:, None]) > band * np.abs(ref_threshold[:, None])
    assert np.array_equal(keep[outside], ref_keep[outside])
    assert outside.mean() > 0.99


@pytest.mark.parametrize("k,alpha", [(1, 0.0), (2, 1.1), (4, 3.0), (15, 1.1)])
def test_sor64_matches_direct_form(k, alpha):
    pc = noisy_faces(2, 600, seed=7 + k)
    o = O.sor64(pc, k, alpha, row_block=128)
    assert_sor_agrees(o.value, o.threshold, o.keep, *direct_sor64(pc, k, alpha), band=1e-9)
    assert 0 < o.keep.mean() < 1


@pytest.mark.parametrize("k,alpha", [(2, 1.1), (5, 0.5)])
def test_sor64_matches_reference_torch_formulation(k, alpha):
    pc = noisy_faces(3, 700, seed=21)
    o = O.sor64(pc, k, alpha)
    sel, mask, value, thr = O.sor_outlier_removal(torch.from_numpy(pc), k, alpha)
    assert_sor_agrees(o.value, o.threshold, o.keep, value.numpy(), thr.numpy(), mask.numpy(), band=1e-9)
    for b in range(3):
        assert torch.equal(sel[b], torch.from_numpy(pc[b][mask[b].numpy()]))


@pytest.mark.parametrize("sizes,npoint", [([1500, 1024, 700, 512, 1, 3000], 1024),   # above, equal, below, 1024 % 512 == 0
                                          ([5, 7, 9], 10), ([10, 10], 10), ([33], 1024), ([1024, 2048, 256], 1024)])
def test_draw_indices_match_the_transcribed_loop(sizes, npoint):
    rng = np.random.default_rng(3)
    pcs = [rng.standard_normal((n, 3)) for n in sizes]
    np.random.seed(1234)
    ref = O.sor_process_data(pcs, npoint)
    after_ref = np.random.random()
    np.random.seed(1234)
    idx = pcd.defense.draw_indices(sizes, npoint)
    assert np.random.random() == after_ref                  # the same number of draws from the global generator
    assert idx.shape == (len(sizes), npoint) and idx.dtype == np.int64
    assert np.array_equal(np.stack([p[i] for p, i in zip(pcs, idx)]), ref)


def test_draw_indices_reject_an_empty_sample():
    with pytest.raises(ValueError, match="sample 1"):
        pcd.defense.draw_indices([4, 0, 4], 8)


def test_sor_forward_argument_errors():
    lib = pcd._lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every call below fails its argument check

    def call(B=2, N=16, k=2, alpha=1.1, value=fake):
        return lib.pcd_sor_forward(fake, 48, 3, 1, B, N, k, alpha, value, fake, fake, fake, fake, None)

    assert call(k=0) == 1
    assert call(k=16) == 1
    assert call(N=5, k=5) == 1
    assert call(value=None) == 1
    assert call(alpha=float("nan")) == 1
    assert call(alpha=float("inf")) == 1
    assert call(B=0) == 1
    assert b"pcd_sor_forward" in lib.pcd_last_error()


def test_sor_is_cuda_only():
    a = torch.zeros(2, 16, 3)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.functional.sor(a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.defense.SORDefense()(a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.defense.SORDefense().outlier_removal(a)
