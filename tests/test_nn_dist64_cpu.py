"""Float64 nearest-neighbour distances without a GPU: the numpy brute force against scipy's Euclidean distance matrix
(bit for bit) and its reductions against math.fsum, argument errors of the C ABI, the workspace size, and the
CUDA-only guard."""
import ctypes
import importlib
import math
import warnings

import numpy as np
import pytest
import torch
from scipy.spatial import distance, distance_matrix

from oracle import nn_dist64_oracle as O

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")


def face_pair(N, M, sigma, seed):
    a = synth.face_clouds(1, N, seed=seed)[0]
    b = synth.face_clouds(1, M, seed=seed + 1)[0]
    g = torch.Generator().manual_seed(seed)
    return a.numpy(), (b + sigma * torch.randn(b.shape, generator=g)).numpy()


def mean_bound(v, mean):
    """|mean - exact| allowed: the recursive-summation bound (n-1) * 2^-53 * sum|v| over n, plus the division's
    rounding."""
    n = len(v)
    return (n - 1) * 2.0 ** -53 * math.fsum(np.abs(v)) / n + 2.0 ** -53 * abs(mean)


@pytest.mark.parametrize("N,M,sigma", [(700, 1100, 1e-3), (1000, 513, 0.01), (64, 64, 1e-7)])
def test_pair_s64_is_scipy_euclidean_bit_for_bit(N, M, sigma):
    a, b = face_pair(N, M, sigma, seed=N + M)
    s = O.pair_s64(a, b)
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    assert np.array_equal(np.sqrt(s), distance.cdist(a64, b64, "euclidean"))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)         # distance_matrix is deprecated from SciPy 1.18
        assert np.array_equal(np.sqrt(s), distance_matrix(a64, b64))
    o = O.nn_dist64(a[None], b[None], row_block=256)
    d = distance.cdist(a64, b64, "euclidean")
    assert np.array_equal(np.sqrt(o.a_min[0]), d.min(1)) and np.array_equal(np.sqrt(o.b_min[0]), d.min(0))
    assert np.array_equal(o.a_arg[0], s.argmin(1)) and np.array_equal(o.b_arg[0], s.argmin(0))


def test_pair_s64_with_exact_duplicates():
    a, b = face_pair(500, 400, 0.01, seed=3)
    b[:200] = a[100:300]                 # exact duplicates: distance 0 at the duplicated points
    a[300:320] = a[0]                    # repeated rows: equal minima, the lowest index wins
    s = O.pair_s64(a, b)
    assert np.array_equal(np.sqrt(s), distance.cdist(a.astype(np.float64), b.astype(np.float64)))
    o = O.nn_dist64(a[None], b[None])
    assert (o.a_min[0, 100:300] == 0).all() and np.array_equal(o.a_arg[0, 100:300], np.arange(200))
    assert np.array_equal(o.b_arg[0], s.argmin(0))


def test_reductions_within_the_summation_bound():
    a, b = face_pair(3000, 2500, 1e-3, seed=11)
    o = O.nn_dist64(a[None], b[None], a_lengths=[2900], b_lengths=[2500])
    for v, mean_sq, mean, max_sq, max_, argmax in ((o.a_min[0, :2900], o.a_mean_sq, o.a_mean, o.a_max_sq, o.a_max, o.a_argmax),
                                                   (o.b_min[0], o.b_mean_sq, o.b_mean, o.b_max_sq, o.b_max, o.b_argmax)):
        for got, x in ((mean_sq[0], v), (mean[0], np.sqrt(v))):
            exact = math.fsum(x) / len(x)
            assert abs(got - exact) <= mean_bound(x, exact)
        assert max_sq[0] == v.max() and max_[0] == np.sqrt(v.max()) and argmax[0] == v.argmax()
    assert np.isnan(o.a_min[0, 2900:]).all() and (o.a_arg[0, 2900:] == -1).all()


def test_lengths_zero_and_nan_follow_numpy():
    a, b = face_pair(40, 30, 0.01, seed=5)
    a[7, 1] = np.nan
    o = O.nn_dist64(np.stack([a, a]), np.stack([b, b]), a_lengths=[40, 0], b_lengths=[30, 30])
    assert np.isnan(o.a_min[0, 7]) and o.a_arg[0, 7] == 0                   # a NaN row: the first NaN column
    assert np.isnan(o.b_min[0]).all() and (o.b_arg[0] == 7).all()            # a NaN column wins every row
    assert np.isnan(o.b_max_sq[0]) and o.b_argmax[0] == 0
    assert np.isnan(o.a_mean_sq[1]) and o.a_argmax[1] == -1                  # no valid row
    assert np.isnan(o.b_min[1]).all() and (o.b_arg[1] == -1).all()          # the other side is empty
    assert np.isnan(o.b_mean[1]) and o.b_argmax[1] == 0


def test_nn_dist64_forward_argument_errors():
    lib = pcd._lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every call below fails its argument check

    def call(B=2, N=16, M=8, col_split=0, out=fake, ws=fake, ws_bytes=1 << 30):
        return lib.pcd_nn_dist64_forward(fake, 48, 3, 1, fake, 24, 3, 1, B, N, M, None, None, col_split,
                                         out, fake, fake, fake, fake, fake, ws, ws_bytes, None)

    assert call(B=0) == 1
    assert call(B=-1) == 1
    assert call(N=0) == 1
    assert call(M=0) == 1
    assert call(col_split=-1) == 1
    assert call(out=None) == 1
    assert b"pcd_nn_dist64_forward" in lib.pcd_last_error()
    need = lib.pcd_nn_dist64_workspace_bytes(2, 16, 8, 0)
    assert call(ws_bytes=need - 1) == 2                                     # PCD_ERR_WORKSPACE
    assert call(ws=None) == 2
    assert b"workspace" in lib.pcd_last_error()


def test_workspace_size_without_gpu():
    ws = pcd._lib.load().pcd_nn_dist64_workspace_bytes
    assert ws(0, 16, 16, 0) == 0 and ws(2, 0, 16, 0) == 0 and ws(2, 16, 16, -1) == 0
    assert ws(3, 1000, 700, 1) == 3 * 1700 * 12                             # one (f64, i32) partial per row
    assert ws(3, 1000, 700, 7) == 7 * ws(3, 1000, 700, 1)
    assert ws(1, 4096, 4096, 0) > ws(1, 4096, 4096, 1)                      # a small batch splits its columns
    assert ws(512, 4096, 4096, 0) == ws(512, 4096, 4096, 1)                 # a large one does not


def test_nn_dist64_is_cuda_only():
    a = torch.zeros(2, 16, 3)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.functional.nn_dist64(a, a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.metrics.chamfer64(a, a)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pcd.metrics.hausdorff64(a, a)
