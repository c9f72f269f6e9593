"""The device point sampler's reference without a GPU: Random123's known answers for Philox4x32-10, the structure of the
three draw cases, chi-square uniformity over ordered tuples, the table composition, and the argument errors of
pcd_sample_points and of the Python wrappers that run before any device work."""
import ctypes
import importlib
import itertools

import numpy as np
import pytest
import torch
from scipy import stats

from oracle import sample_oracle as S

pcd = importlib.import_module("3dpointcloudattack_b200")


@pytest.mark.parametrize("ctr, key, want", [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
])
def test_philox_known_answers(ctr, key, want):
    assert S.philox4x32_10(ctr, key).tolist() == want
    # vectorised: the same block at every position of a batch
    assert (S.philox4x32_10(np.tile(ctr, (3, 2, 1)), np.tile(key, (3, 2, 1))) == np.array(want, np.uint32)).all()


def test_keys_are_distinct_and_carry_the_index():
    k = S.point_keys(seed=7, g=[0, 1, 2], counter=3, n=S.MAX_N)
    assert k.shape == (3, S.MAX_N) and k.dtype == np.uint64
    assert ((k & np.uint64(S.MAX_N - 1)) == np.arange(S.MAX_N, dtype=np.uint64)).all()
    assert all(len(np.unique(row)) == S.MAX_N for row in k)
    # a key is a function of (seed, g, counter, i) alone: a shorter cloud has the same leading keys
    assert (S.point_keys(7, [1], 3, 100)[0] == k[1, :100]).all()
    assert not (S.point_keys(8, [1], 3, 100)[0] == k[1, :100]).all()
    assert not (S.point_keys(7, [1], 4, 100)[0] == k[1, :100]).all()
    assert not (S.point_keys(7, [1], 3 + (1 << 32), 100)[0] == k[1, :100]).all()      # the counter's high word counts


@pytest.mark.parametrize("n, npoint", [(1000, 524), (1025, 1024), (5, 3), (16384, 4096)])
def test_more_points_than_drawn_gives_distinct_points(n, npoint):
    out = S.sample_points([n, n, n], npoint, seed=1, counter=0)
    for row in out:
        assert len(np.unique(row)) == npoint and row.min() >= 0 and row.max() < n
    assert not np.array_equal(out[0], out[1])                                        # samples draw independently
    assert not np.array_equal(np.sort(out[0]), np.arange(npoint))


@pytest.mark.parametrize("n, npoint", [(1, 3), (2, 3), (5, 13), (1000, 1024), (1023, 4096), (3, 524)])
def test_fewer_points_than_drawn_tiles_the_cloud(n, npoint):
    out = S.sample_points([n, n], npoint, seed=2, counter=5)
    whole = npoint // n * n
    for row in out:
        assert np.array_equal(row[:whole], np.tile(np.arange(n), npoint // n))
        rest = row[whole:]
        assert len(rest) == npoint % n and len(np.unique(rest)) == len(rest) and (rest < n).all()


def test_equal_and_empty_samples():
    out = S.sample_points([4, 0, 4], 4, seed=3, counter=0)
    assert np.array_equal(out[0], np.arange(4)) and (out[1] == -1).all() and np.array_equal(out[2], np.arange(4))


def test_table_maps_every_drawn_value():
    rng = np.random.default_rng(0)
    table = np.stack([rng.permutation(50) for _ in range(3)]).astype(np.int32)
    lengths, npoint = [40, 7, 0], 20
    plain = S.sample_points(lengths, npoint, seed=4, counter=9)
    mapped = S.sample_points(lengths, npoint, seed=4, counter=9, table=table)
    for b in range(2):
        assert np.array_equal(mapped[b], table[b][plain[b]])
    assert (mapped[2] == -1).all()


def test_first_sample_shards_the_draws():
    whole = S.sample_points([30] * 8, 10, seed=5, counter=2)
    a = S.sample_points([30] * 4, 10, seed=5, counter=2, first_sample=0)
    b = S.sample_points([30] * 4, 10, seed=5, counter=2, first_sample=4)
    assert np.array_equal(whole, np.concatenate([a, b]))


def chi_square_over_tuples(rows, n, r):
    """p-value of the counts of ordered r-tuples of distinct values < n among rows against the uniform distribution"""
    tuples = list(itertools.permutations(range(n), r))
    index = {t: m for m, t in enumerate(tuples)}
    counts = np.bincount([index[tuple(t)] for t in rows.tolist()], minlength=len(tuples))
    assert counts.sum() == len(rows)
    return stats.chisquare(counts).pvalue


def test_draws_are_uniform_over_ordered_tuples():
    """n = 5, npoint = 3: the 60 ordered tuples, 60 000 samples of distinct g"""
    g = np.arange(60000)
    perm = S.permutation(seed=11, g=g, counter=0, n=5)
    assert chi_square_over_tuples(perm[:, :3], 5, 3) > 1e-4
    # the sampler itself on a batch of 60 000 samples at another counter
    out = S.sample_points([5] * 60000, 3, seed=11, counter=1)
    assert chi_square_over_tuples(out, 5, 3) > 1e-4


def test_remainder_is_uniform_over_ordered_tuples():
    """n = 5, npoint = 13: two whole copies, then 3 distinct points -- the same 60 tuples"""
    out = S.sample_points([5] * 60000, 13, seed=12, counter=0)
    assert (out[:, :10] == np.tile(np.arange(5), 2)).all()
    assert chi_square_over_tuples(out[:, 10:], 5, 3) > 1e-4


# ------------------------------------------------------------------------------------------- C ABI without a GPU
def test_sample_points_argument_errors():
    lib = pcd._lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every call below fails its argument check

    def call(B=2, N=16, npoint=8, len_=None, table=None, ts=0, first=0, counter=fake, out=fake):
        return lib.pcd_sample_points(B, N, npoint, len_, table, ts, 1, first, counter, out, None)

    assert call(npoint=0) == 1
    assert call(npoint=-3) == 1
    assert call(B=0) == 1
    assert call(N=0) == 1
    assert call(counter=None) == 1
    assert call(out=None) == 1
    assert call(first=-1) == 1
    assert call(table=fake, ts=15) == 1                                     # a row stride below N
    assert b"pcd_sample_points" in lib.pcd_last_error()
    assert call(N=S.MAX_N + 1) == 4                                         # PCD_ERR_UNSUPPORTED
    assert call(N=100000, npoint=1024) == 4
    assert b"16384" in lib.pcd_last_error()


def test_python_checks_before_the_device():
    F, D = pcd.functional, pcd.defense
    with pytest.raises(RuntimeError, match="CUDA only"):
        F.PointSampler(0, device="cpu")
    with pytest.raises(ValueError):
        F.PointSampler(-1, device="cuda")
    with pytest.raises(ValueError):
        F.PointSampler(0, first_sample=-1, device="cuda")
    with pytest.raises(TypeError):
        F.sample_points(None, 16, 4, sampler=object(), table=torch.zeros(2, 16, dtype=torch.int32))
    with pytest.raises(ValueError, match="drop_num"):
        D.SRSDefense(drop_num=16)(torch.zeros(2, 16, 3))
    with pytest.raises(ValueError, match="drop_num"):
        D.SRSDefense(drop_num=-1)(torch.zeros(2, 16, 3))


def test_srs_numpy_mode_is_the_published_loop():
    """SRSDefense without a sampler: np.random.choice(K, K - drop_num, replace=False) per sample, in batch order"""
    x = torch.randn(3, 40, 3, generator=torch.Generator().manual_seed(0))
    np.random.seed(7)
    y = pcd.defense.SRSDefense(drop_num=15)(x)
    np.random.seed(7)
    ref = np.stack([x.numpy()[b][np.random.choice(40, 25, replace=False)] for b in range(3)])
    assert y.shape == (3, 25, 3) and np.array_equal(y.numpy(), ref)
