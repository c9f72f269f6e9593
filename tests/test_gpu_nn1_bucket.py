"""The bucketed clouds that nn1_bucket writes for the pruned NN-1 chain, bit for bit against a numpy float32 restatement.

The chain's outputs do not depend on how the clouds are bucketed, so no other test looks at the layout; this one pins it: the
joint box of both clouds' finite points, cell = 32 / (hi - lo) per axis, the 15-bit Morton code of every point (non-finite
points 2^15), a stable sort by code, the pair records {x0,x1,y0,y1},{z0,z1,n0,n1} in sorted order with inert slots up to the
next multiple of 32, the permutation, and per chunk of 32 slots (lo xyz, largest norm), (hi xyz, never-prune flag)."""
import importlib

import numpy as np
import pytest
import torch

from oracle import pcd_oracle as O

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F = pcd.functional

B = 16          # the smallest batch the chain serves
BITS = 5


def round_up(v, a):
    return (v + a - 1) // a * a


def bucket_regions(ws, B, N, M):
    """(brec [B,2,bslots/2,8] f32, bbox [B,2,bslots/32,8] f32, bperm [B,2,bslots] i32): the last three regions of the nn1
    workspace, each 256-byte aligned, in the order brec, bbox, bperm."""
    bslots = round_up(max(N, M), 32)
    nb = B * 2 * bslots
    end = ws.numel()
    bperm0 = end - round_up(nb * 4, 256)
    bbox0 = bperm0 - round_up(nb, 256)
    brec0 = bbox0 - round_up(nb * 16, 256)
    host = ws.cpu().numpy()
    brec = host[brec0:brec0 + nb * 16].view(np.float32).reshape(B, 2, bslots // 2, 8)
    bbox = host[bbox0:bbox0 + nb].view(np.float32).reshape(B, 2, bslots // 32, 8)
    bperm = host[bperm0:bperm0 + nb * 4].view(np.int32).reshape(B, 2, bslots)
    return brec, bbox, bperm


def run_chain(rows, cols, norm, channel_major=False):
    """One pcd_nn1_forward on a workspace of our own; returns the workspace (after the whole chain)."""
    lib = pcd._lib.load()
    Bb, N, M = rows.shape[0], rows.shape[1], cols.shape[1]

    def dev(x):
        if channel_major:            # [B,3,n] storage seen as [B,n,3]
            return torch.from_numpy(np.ascontiguousarray(x.transpose(0, 2, 1))).cuda().transpose(1, 2)
        return torch.from_numpy(x).cuda()

    r, c = dev(rows), dev(cols)
    out = [torch.empty((Bb, N), dtype=torch.float32, device="cuda"), torch.empty((Bb, N), dtype=torch.int32, device="cuda"),
           torch.empty((Bb, M), dtype=torch.float32, device="cuda"), torch.empty((Bb, M), dtype=torch.int32, device="cuda"),
           torch.empty((4, Bb), dtype=torch.float32, device="cuda"), torch.empty((2, Bb), dtype=torch.int32, device="cuda")]
    ws_bytes = lib.pcd_nn1_workspace_bytes(Bb, N, M, 0)
    ws = torch.zeros((ws_bytes,), dtype=torch.uint8, device="cuda")
    st = lib.pcd_nn1_forward(r.data_ptr(), *r.stride(), c.data_ptr(), *c.stride(), Bb, N, M, F.FORM_SUM_FIRST, norm, 0, 0,
                             1.0, 1.0, *(t.data_ptr() for t in out), None, 0, None, 0, ws.data_ptr(), ws_bytes, 0, 0, 0,
                             None, None, torch._C._cuda_getCurrentRawStream(torch.cuda.current_device()))
    pcd._lib.check(st, "pcd_nn1_forward")
    torch.cuda.synchronize()
    return ws


def spread(v):
    out = np.zeros_like(v)
    for k in range(BITS):
        out |= ((v >> k) & 1) << (3 * k)
    return out


def expected(rows, cols, norm, side, bslots):
    """numpy float32 restatement of one (sample, side): records, chunk boxes, permutation."""
    pinf = np.float32(np.inf)
    fin = [np.isfinite(p).all(1) for p in (rows, cols)]
    both = np.concatenate([rows[fin[0]], cols[fin[1]]])
    lo, hi = both.min(0), both.max(0)
    with np.errstate(divide="ignore"):
        cell = np.where(hi > lo, np.float32(1 << BITS) / (hi - lo), np.float32(0)).astype(np.float32)
    pts, ok = (cols, fin[1]) if side else (rows, fin[0])
    n = pts.shape[0]
    with np.errstate(invalid="ignore"):
        q = np.clip((pts - lo) * cell, np.float32(0), np.float32((1 << BITS) - 1))
    q = np.where(ok[:, None], q, 0).astype(np.uint32)
    code = np.where(ok, spread(q[:, 0]) | (spread(q[:, 1]) << 1) | (spread(q[:, 2]) << 2), 1 << (3 * BITS))
    perm = np.argsort(code, kind="stable").astype(np.int32)
    nslots = round_up(n, 32)
    sp = np.zeros((nslots, 3), np.float32)
    sp[:n] = pts[perm]
    with np.errstate(invalid="ignore", over="ignore"):
        nrm = np.full(nslots, pinf, np.float32)
        nrm[:n] = O.norms(norm, pts[perm][None])[0]
    rec = np.zeros((bslots // 2, 8), np.float32)
    rec[:nslots // 2] = np.stack([sp[0::2, 0], sp[1::2, 0], sp[0::2, 1], sp[1::2, 1], sp[0::2, 2], sp[1::2, 2],
                                  nrm[0::2], nrm[1::2]], 1)
    sok = np.zeros(nslots, bool)
    sok[:n] = ok[perm]
    box = []
    for c in range(round_up(n, 32) // 32):
        s = slice(32 * c, min(32 * c + 32, n))
        f = sok[s]
        p = sp[s][f]
        box.append(np.concatenate([p.min(0) if len(p) else [pinf] * 3, [nrm[s][f].max() if len(p) else -pinf],
                                   p.max(0) if len(p) else [-pinf] * 3, [0.0 if f.all() else 1.0]]).astype(np.float32))
    return rec, np.array(box, np.float32), perm


def same_bits(got, want):
    """bit for bit; NaN only has to be NaN (a NaN norm's payload is the hardware's)"""
    g, w = np.asarray(got, np.float32), np.asarray(want, np.float32)
    nan = np.isnan(w)
    return np.array_equal(np.isnan(g), nan) and np.array_equal(g[~nan].view(np.uint32), w[~nan].view(np.uint32))


def check(rows, cols, norm=F.NORM_FMA, channel_major=False, samples=(0, 1, B - 1)):
    rows, cols = np.ascontiguousarray(rows, np.float32), np.ascontiguousarray(cols, np.float32)
    Bb, N, M = rows.shape[0], rows.shape[1], cols.shape[1]
    brec, bbox, bperm = bucket_regions(run_chain(rows, cols, norm, channel_major), Bb, N, M)
    bslots = brec.shape[2] * 2
    for b in samples:
        for side, n in ((0, N), (1, M)):
            rec, box, perm = expected(rows[b], cols[b], norm, side, bslots)
            assert np.array_equal(bperm[b, side, :n], perm), (b, side)
            assert same_bits(brec[b, side], rec), (b, side)
            assert same_bits(bbox[b, side, :len(box)], box), (b, side)


def face_pair(Bb, n, seed):
    ori = synth.face_clouds(Bb, n, seed=seed)
    return synth.perturb(ori, 0.01, seed=seed + 1).numpy(), ori.numpy()


@pytest.mark.parametrize("channel_major", [False, True])
@pytest.mark.parametrize("norm", [F.NORM_FMA, F.NORM_MULSUM])
def test_face_clouds(norm, channel_major):
    adv, ori = face_pair(B, 4096, seed=51)
    check(adv, ori, norm, channel_major)


@pytest.mark.parametrize("channel_major", [False, True])
def test_unequal_sizes_not_whole_chunks(channel_major):
    adv, _ = face_pair(B, 4096, seed=61)
    _, ori = face_pair(B, 5000, seed=62)
    check(adv, ori, channel_major=channel_major)
    check(ori, adv, F.NORM_MULSUM, channel_major)


def test_large_clouds():
    adv, ori = face_pair(B, 16384, seed=71)
    check(adv, ori, samples=(0, B - 1))


def test_nan_and_inf_points():
    adv, ori = face_pair(B, 4096, seed=81)
    adv[0, 17] = np.nan; adv[0, 1500, 2] = np.inf; ori[0, 999, 0] = -np.inf; ori[1, 5:40] = np.nan
    adv[B - 1, 4000:] = np.inf
    check(adv, ori)
    check(adv, ori, F.NORM_MULSUM, channel_major=True)


def test_all_identical_points():
    """every point of both clouds in one cell (hi == lo: cell 0), so the order is the index order"""
    same = np.full((B, 4096, 3), np.float32(0.3), np.float32)
    check(same, same.copy())
    adv, _ = face_pair(B, 4096, seed=91)
    check(adv, np.full((B, 4104, 3), np.float32(-1.5), np.float32))
