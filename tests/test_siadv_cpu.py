"""The SI-Adv step's reference without a GPU: the spin-axis frames, the step's geometry before the clip, the per-axis
clip, the fixed tree sum, the float64 normals, and the argument errors of pcd_si_step that come before any CUDA call."""
import ctypes
import importlib

import numpy as np
import pytest

from oracle import siadv_oracle as O

pcd = importlib.import_module("3dpointcloudattack_b200")


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def normals_around_the_boundary(rng):
    """unit normals with z = +-1, |z^2 - 1| just under and just over 1e-4, and random ones"""
    zs = [1.0, -1.0, np.sqrt(1 - 0.9e-4), -np.sqrt(1 - 0.99e-4), np.sqrt(1 - 1.01e-4), -np.sqrt(1 - 1.2e-4), 0.0, 0.5]
    out = []
    for z in zs:
        phi = rng.uniform(0, 2 * np.pi)
        r = np.sqrt(max(1 - z * z, 0.0))
        out.append([r * np.cos(phi), r * np.sin(phi), z])
    return np.concatenate([np.array(out), unit(rng.standard_normal((200, 3)))])


def test_spin_axis_rows_are_orthonormal():
    n = normals_around_the_boundary(np.random.default_rng(0))
    u = O.spin_axis(n, np.float64)
    edge = np.abs(n[:, 2] ** 2 - 1) < O.BOUNDARY
    assert edge[:4].all() and not edge[4:].any()
    err = np.abs(u @ np.swapaxes(u, -1, -2) - np.eye(3)).max(axis=(-1, -2))
    # the boundary frame's last two rows have length |z|, within 1e-4 of 1 there; elsewhere the frame is exact
    assert err[edge].max() < 1e-4 and err[~edge].max() < 1e-12
    assert np.allclose(u[~edge, 2], n[~edge], atol=0)                          # u2 is the normal itself
    # float32: the boundary constants are fp32(1/sqrt 2) and fp32(sqrt 2), and the frame stays orthonormal to rounding
    assert np.float32(1 / np.sqrt(2)) == np.float32(0.70710677) and np.float32(np.sqrt(2)) == np.float32(1.41421354)
    u32 = O.spin_axis(n.astype(np.float32), np.float32).astype(np.float64)
    err32 = np.abs(u32 @ np.swapaxes(u32, -1, -2) - np.eye(3)).max(axis=(-1, -2))
    assert err32[edge].max() < 2e-4 and err32[np.abs(n[:, 2]) < 0.9].max() < 1e-6


def test_step_before_the_clip_is_the_tangent_gradient_step():
    """p_new = p - a (g - (g.n) n) / ||g - (g.n) n||, the norm over the whole sample; each point moves in its plane"""
    rng = np.random.default_rng(1)
    B, N = 3, 257
    pc = rng.standard_normal((B, N, 3)).astype(np.float32)
    n = unit(rng.standard_normal((B, N, 3)) * [1, 1, 0.3]).astype(np.float32)   # away from the boundary case
    g = rng.standard_normal((B, N, 3)).astype(np.float32)
    step_size, scale = 0.007, np.sqrt(3 * 1024)
    pn, norm = O.si_step(pc, pc, n, g, step_size, 0.16, scale, dtype=np.float64, clip=False)
    p, nn, gg = (x.astype(np.float64) for x in (pc, n, g))
    proj = gg - (gg * nn).sum(-1, keepdims=True) * nn
    pnorm = np.sqrt((proj ** 2).sum(axis=(1, 2)))
    assert np.allclose(norm, pnorm, rtol=1e-6)
    want = p - step_size * scale * proj / (pnorm[:, None, None] + 1e-9)
    assert np.abs(pn - want).max() < 1e-5 * np.abs(want).max()
    # a zero gradient gives a zero step: the point moves only by its round trip through the frame, which is exact up to
    # the fp32 rounding of the unit normal (|n|^2 - 1 ~ 1e-7)
    still, zn = O.si_step(pc, pc, n, np.zeros_like(g), step_size, 0.16, scale, dtype=np.float64, clip=False)
    assert (zn == 0).all() and np.abs(still - p).max() < 1e-6 * np.abs(p).max()
    # the step itself lies in every point's tangent plane
    step = pn - still
    assert np.abs((step * nn).sum(-1)).max() < 1e-6 * np.abs(step).max()


@pytest.mark.parametrize("dtype, tol", [(np.float64, 1e-12), (np.float32, 1e-6)])
def test_clip_bounds_every_axis_norm_by_eps(dtype, tol):
    rng = np.random.default_rng(2)
    B, N, eps = 4, 1000, 0.05
    ori = rng.standard_normal((B, N, 3)).astype(np.float32)
    pc = (ori + 0.01 * rng.standard_normal((B, N, 3))).astype(np.float32)
    n = unit(rng.standard_normal((B, N, 3))).astype(np.float32)
    g = rng.standard_normal((B, N, 3)).astype(np.float32)
    out, _ = O.si_step(pc, ori, n, g, 0.5, eps, dtype=dtype)
    axis_norm = np.sqrt(((out.astype(np.float64) - ori) ** 2).sum(axis=1))     # [B, 3]: over the N points of each axis
    assert axis_norm.max() <= eps * (1 + tol) + tol and axis_norm.max() > 0.9 * eps     # the clip is active ...
    free, _ = O.si_step(pc, ori, n, g, 1e-6, 10.0, dtype=dtype)                  # ... and leaves a small step alone
    pn, _ = O.si_step(pc, ori, n, g, 1e-6, 10.0, dtype=dtype, clip=False)
    assert np.abs(free - pn).max() <= 4 * np.finfo(dtype).eps * np.abs(pn).max()


def tree_by_definition(v):
    """a node covering the aligned block [k 2^l, min((k+1) 2^l, N)) is left + right, or left when the right half is
    empty; the leaves are the values in order"""
    N = len(v)

    def node(k, level):
        if level == 0:
            return v[k]
        left = node(2 * k, level - 1)
        if (2 * k + 1) << (level - 1) >= N:
            return left
        return left + node(2 * k + 1, level - 1)

    level = 0
    while (1 << level) < N:
        level += 1
    return node(0, level)


@pytest.mark.parametrize("N", [1, 2, 3, 5, 1000])
def test_tree_sum_is_its_definition(N):
    rng = np.random.default_rng(N)
    v = (rng.standard_normal(N) ** 2 * 10.0 ** rng.uniform(-6, 6, N)).astype(np.float32)
    want = tree_by_definition(v)
    got = O.tree_sum(v)
    assert got.dtype == np.float32 and got.view(np.uint32) == np.float32(want).view(np.uint32)
    # along the point axis of a batch, as the step uses it
    batch = np.stack([v, v[::-1]])[..., None].repeat(3, -1)
    t = O.tree_sum(batch, axis=1)
    assert t.shape == (2, 3) and (t[0] == want).all() and (t[1] == tree_by_definition(v[::-1])).all()


def test_normals64_of_a_plane():
    rng = np.random.default_rng(3)
    pc = np.concatenate([rng.uniform(-1, 1, (1, 300, 2)), np.zeros((1, 300, 1))], -1)
    n, gap, _ = O.normals64(pc, 20)
    assert np.allclose(np.abs(n[..., 2]), 1) and gap.shape == (1, 300) and (gap >= 0).all()


def test_si_step_argument_errors():
    lib = pcd._lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every call below fails its argument check

    def call(pc=fake, ori=fake, normal=fake, grad=fake, B=2, N=16, eps=0.1, split=0):
        return lib.pcd_si_step(pc, 48, 3, 1, ori, 48, 3, 1, normal, 48, 3, 1, grad, 48, 3, 1, B, N, 0.007, 55.4, eps,
                               split, None, None)

    assert call(pc=None) == 1
    assert call(ori=None) == 1
    assert call(normal=None) == 1
    assert call(grad=None) == 1
    assert call(N=0) == 1
    assert call(B=-1) == 1
    assert call(eps=-1e-3) == 1
    assert call(eps=float("nan")) == 1
    assert call(split=3) == 1 and call(split=32) == 1 and call(split=-1) == 1
    assert call(N=4096, split=1) == 1                                         # 4096 points in one CTA
    assert b"pcd_si_step" in lib.pcd_last_error()
    assert call(N=16385) == 4                                                 # PCD_ERR_UNSUPPORTED
    assert b"16384" in lib.pcd_last_error()
    assert call(B=0) == 0 and call(B=0, pc=None, grad=None) == 0             # an empty batch is a no-op
