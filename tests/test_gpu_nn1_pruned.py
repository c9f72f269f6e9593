"""The pruned NN-1 chain (nn1_bucket -> nn1_pruned_sweep -> fix-up) against the oracle, bit for bit on minima and
lowest-index arg-mins, on the inputs that stress its pruning, its cross-chunk tie flag and its permutation.  The chain serves
dense clouds of 4096 to 16384 points per side in batches of 16 or more."""
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from oracle import pcd_oracle as O

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F = pcd.functional

FORMS = [(F.FORM_ROW_COL, F.NORM_MULSUM, O.FORM_ROW_COL, O.NORM_MULSUM),
         (F.FORM_COL_ROW, F.NORM_MULSUM, O.FORM_COL_ROW, O.NORM_MULSUM),
         (F.FORM_SUM_FIRST, F.NORM_FMA, O.FORM_SUM_FIRST, O.NORM_FMA),
         (F.FORM_ROW_COL, F.NORM_FMA, O.FORM_ROW_COL, O.NORM_FMA),
         (F.FORM_COL_ROW, F.NORM_FMA, O.FORM_COL_ROW, O.NORM_FMA),
         (F.FORM_SUM_FIRST, F.NORM_MULSUM, O.FORM_SUM_FIRST, O.NORM_MULSUM)]


B = 16          # the smallest batch the chain serves


def tile(x):
    return np.ascontiguousarray(np.broadcast_to(x, (B,) + x.shape[1:]) if x.shape[0] == 1 else x, np.float32)


def check(rows, cols, forms=FORMS, samples=2):
    """The batch runs on the GPU; its first `samples` samples are compared with the oracle."""
    rows, cols = tile(rows), tile(cols)
    r_, c_ = rows[:samples], cols[:samples]
    for form, norm, oform, onorm in forms:
        r = F.nn1(torch.from_numpy(rows).cuda(), torch.from_numpy(cols).cuda(), form, norm, cache=False)
        o = O.nn1(oform, r_, c_, O.norms(onorm, r_), O.norms(onorm, c_))
        got = [t[:samples].cpu().numpy() for t in (r.row_min, r.row_arg, r.col_min, r.col_arg)]
        for g, want in zip(got, o):
            assert np.array_equal(g, want)


def face_pair(B, n, seed=5):
    ori = synth.face_clouds(B, n, seed=seed)
    return synth.perturb(ori, 0.01, seed=seed + 1).numpy(), ori.numpy()


_NAMES = r"""
import importlib, sys
import numpy as np, torch
from torch.profiler import ProfilerActivity, profile
sys.path.insert(0, ".")
pcd = importlib.import_module("3dpointcloudattack_b200"); F = pcd.functional
synth = importlib.import_module("3dpointcloudattack_b200.synth")
B, n, R, mt = (int(x) for x in sys.argv[1:5])
o = synth.face_clouds(B, n, seed=5).cuda(); a = o + 0.01 * torch.randn_like(o)
F.force_tiling(R, mt)
F.nn1(a, o, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False); torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    F.nn1(a, o, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False); torch.cuda.synchronize()
print(" ".join(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA))
"""


def kernel_names(B, n, tiling=(0, 0)):
    """Kernels of one nn1 call, profiled in a fresh process (a profiler session leaves state behind in the one it ran in)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-s", "-c", _NAMES, str(B), str(n), *map(str, tiling)], cwd=root,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return r.stdout


def test_the_pruned_chain_serves_large_dense_batches_only():
    s = kernel_names(16, 4096)
    assert "nn1_pruned_sweep_kernel" in s and "nn1_sweep_kernel" not in s
    assert "nn1_pruned_sweep_kernel" not in kernel_names(16, 2048)      # small clouds
    assert "nn1_pruned_sweep_kernel" not in kernel_names(8, 4096)       # small batches
    s = kernel_names(16, 4096, (16, 256))                                 # an explicit tiling keeps the full sweep
    assert "nn1_sweep_kernel" in s and "nn1_pruned_sweep_kernel" not in s


def test_exact_ties_across_chunks_on_a_lattice():
    """Columns on an 18^3 lattice, rows at cell centres: every row has 8 equidistant nearest columns (exact in fp32), spread
    over different Morton chunks, so only the exact-tie pass gives the lowest index."""
    rs = np.random.RandomState(3)
    g = lambda idx: np.stack(np.meshgrid(idx, idx, idx, indexing="ij"), -1).reshape(-1, 3).astype(np.float32) * 0.25
    cols = g(np.arange(18) - 8.5)[rs.permutation(18 ** 3)][None]
    rows = g(np.arange(17) - 8.0)[rs.permutation(17 ** 3)[:4912]][None]
    check(rows, cols, FORMS[:3])


def test_duplicates_at_far_indices():
    """Every column exists twice, at indices far apart: equal Morton codes, so the copies sit in one chunk or straddle a
    chunk boundary (a cross-chunk tie)."""
    adv, ori = face_pair(B, 4096, seed=11)
    ori[:, 2048:] = ori[:, :2048][:, ::-1]
    check(adv, ori, FORMS[:3])
    check(ori, ori, FORMS[2:3])


def test_near_equidistant_neighbours_at_chunk_boundaries():
    """Columns on a grid of step h, rows half a step off by a relative 1e-6: two almost equidistant candidates per row whose
    values differ by far less than the pruning margin, often in different chunks."""
    rs = np.random.RandomState(4)
    h = 0.02
    cols = np.stack(np.meshgrid(np.arange(16) * h, np.arange(16) * h, np.arange(16) * h, indexing="ij"), -1)
    cols = cols.reshape(1, -1, 3).astype(np.float32)
    rows = cols.copy()
    rows[..., 0] += np.float32(h / 2) * (1 + 1e-6 * rs.choice([-1, 1], size=rows.shape[:2])).astype(np.float32)
    check(rows, cols[:, rs.permutation(cols.shape[1])], FORMS[:3])


def test_two_separated_clusters():
    adv, ori = face_pair(B, 4096, seed=21)
    ori[:, 2048:] += np.float32(50.0)
    adv[:, 2048:] += np.float32(50.0)
    check(adv, ori, FORMS[:3])


def test_nan_and_inf_points_in_face_clouds():
    adv, ori = face_pair(B, 4096, seed=31)
    adv[0, 17] = np.nan; adv[0, 1500, 2] = np.inf; ori[0, 999, 0] = -np.inf; ori[1, 5:40] = np.nan
    for form, norm, oform, onorm in FORMS[:3]:
        r = F.nn1(torch.from_numpy(adv).cuda(), torch.from_numpy(ori).cuda(), form, norm, cache=False)
        ra, ca = r.row_arg.cpu().numpy(), r.col_arg.cpu().numpy()
        assert ra.min() >= 0 and ra.max() < 4096 and ca.min() >= 0 and ca.max() < 4096
        ok_r = np.isfinite(adv).all(-1); ok_c = np.isfinite(ori).all(-1)
        for b in range(2):
            o = O.nn1(oform, adv[b:b + 1, ok_r[b]], ori[b:b + 1, ok_c[b]], O.norms(onorm, adv[b:b + 1, ok_r[b]]),
                      O.norms(onorm, ori[b:b + 1, ok_c[b]]))
            assert np.array_equal(r.row_min.cpu().numpy()[b, ok_r[b]], o.row_min[0])
            assert np.array_equal(r.col_min.cpu().numpy()[b, ok_c[b]], o.col_min[0])
            assert np.array_equal(np.flatnonzero(ok_c[b])[o.row_arg[0]], ra[b, ok_r[b]])
            assert np.array_equal(np.flatnonzero(ok_r[b])[o.col_arg[0]], ca[b, ok_c[b]])


@pytest.mark.parametrize("N,M", [(4100, 4104), (4096, 4228), (8204, 4100), (4116, 16384)])
def test_sizes_that_are_not_whole_chunks(N, M):
    rs = np.random.RandomState(N + M)
    cols = rs.rand(B, M, 3).astype(np.float32)
    rows = (cols[:, rs.randint(0, M, N)] + 0.01 * rs.randn(B, N, 3)).astype(np.float32)
    check(rows, cols, FORMS[:3])


@pytest.mark.parametrize("n", [4096, 16384])
def test_every_form_and_norm_kind_on_face_clouds(n):
    adv, ori = face_pair(B, n, seed=41)
    check(adv, ori, samples=2 if n == 4096 else 1)


def test_unrelated_uniform_clouds():
    rs = np.random.RandomState(9)
    check(rs.rand(B, 4096, 3).astype(np.float32), rs.rand(B, 4608, 3).astype(np.float32), FORMS[:3])
