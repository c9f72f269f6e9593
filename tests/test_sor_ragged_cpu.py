"""SOR on ragged batches without a GPU: the ragged reference against per-sample sor64, argument errors and workspace
size of pcd_sor_forward_len, and the Python argument checks that run before any device work."""
import ctypes
import importlib

import numpy as np
import pytest
import torch

from oracle import sor_oracle as O
from sor_ragged_oracle import sor64_ragged

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")


def noisy_faces(B, N, seed):
    pc = synth.face_clouds(B, N, seed=seed)
    return (pc + 0.01 * torch.randn(pc.shape, generator=torch.Generator().manual_seed(seed))).numpy()


@pytest.mark.parametrize("k", [1, 2, 8])
def test_sor64_ragged_is_sor64_per_truncated_sample(k):
    pc = noisy_faces(6, 300, seed=3 + k)
    pc[2, 200:] = np.nan                     # padding never reaches a result
    lengths = [300, 0, 200, k, k + 1, 1000]  # full, empty, padded, short, the smallest with a statistic, clamped
    o = sor64_ragged(pc, lengths, k, 1.1)
    for b, n in enumerate(lengths):
        n = min(n, 300)
        if n >= k + 1:
            ref = O.sor64(pc[b:b + 1, :n], k, 1.1)
            assert np.array_equal(o.value[b, :n], ref.value[0])
            assert o.threshold[b] == ref.threshold[0] and np.array_equal(o.keep[b, :n], ref.keep[0])
        else:
            assert np.isnan(o.value[b]).all() and np.isnan(o.threshold[b]) and not o.keep[b].any()
        assert np.isnan(o.value[b, n:]).all() and not o.keep[b, n:].any()
    assert np.isfinite(o.value[2, :200]).all()


def test_sor_forward_len_argument_errors():
    lib = pcd._lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every call below fails its argument check

    def call(B=2, N=16, k=2, alpha=1.1, col_split=0, value=fake, lengths=fake, ws=fake, ws_bytes=1 << 30):
        return lib.pcd_sor_forward_len(fake, 48, 3, 1, B, N, k, alpha, None, col_split, value, fake, fake, fake, lengths,
                                       ws, ws_bytes, None)

    assert call(k=0) == 1
    assert call(k=16) == 1
    assert call(value=None) == 1
    assert call(lengths=None) == 1
    assert call(alpha=float("nan")) == 1
    assert call(alpha=float("-inf")) == 1
    assert call(B=0) == 1
    assert call(N=0) == 1
    assert call(col_split=-1) == 1
    assert b"pcd_sor_forward_len" in lib.pcd_last_error()
    need = lib.pcd_sor_workspace_bytes(1, 4096, 2, 0)
    assert need > 0
    assert call(B=1, N=4096, ws_bytes=need - 1) == 2                        # PCD_ERR_WORKSPACE
    assert call(B=1, N=4096, ws=None) == 2
    assert call(B=2, N=16, col_split=3, ws_bytes=0) == 2
    assert b"workspace" in lib.pcd_last_error()


def test_sor_workspace_size_without_gpu():
    ws = pcd._lib.load().pcd_sor_workspace_bytes
    assert ws(0, 16, 2, 0) == 0 and ws(2, 0, 2, 0) == 0 and ws(2, 16, 0, 0) == 0 and ws(2, 16, 16, 0) == 0
    assert ws(2, 16, 2, -1) == 0
    assert ws(2, 64, 2, 0) == 0                                             # one 64-column tile: one range, no workspace
    assert ws(3, 1000, 4, 1) == 0
    assert ws(3, 1000, 4, 7) == 7 * 3 * 5 * 1000 * 8                        # k + 1 doubles per row and range
    assert ws(1, 4096, 2, 0) > 0                                            # a small batch splits its columns
    assert ws(1, 100, 2, 0) == 2 * 3 * 100 * 8                              # never below one tile per range
    assert ws(512, 4096, 2, 0) == 0                                         # a large one does not


def test_sor_lengths_checks_before_the_device():
    a = torch.zeros(2, 16, 3)
    F = pcd.functional
    with pytest.raises(RuntimeError, match="CUDA only"):
        F.sor(a, lengths=torch.tensor([3, 16]))
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.defense.SORDefense()(a, lengths=torch.tensor([3, 16]))
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.defense.SORDefense().outlier_removal(a, lengths=torch.tensor([3, 16]))
