"""Reference for the device point sampler -- TEST / BENCH INFRASTRUCTURE ONLY (tests/, __graft_entry__.smoke(),
tools/defense_bench.py; the product never imports it).

A numpy restatement of the pcd_sample_points contract (include/pcdist.h):
  key[i]  = (r & ~0x3FFF) | i,  r = (w0 << 32) | w1,  (w0, w1, w2, w3) = Philox4x32-10((i, g, c_lo, c_hi), (s_lo, s_hi))
  the points ranked by ascending key (a stable argsort) are a random permutation P of 0 .. n-1;
  out[j] = P[j] (n > npoint), j % n then P (n < npoint), j (n == npoint), -1 (n == 0), each mapped through a table.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)
INDEX_BITS = 14
MAX_N = 1 << INDEX_BITS


def philox4x32_10(ctr, key):
    """ctr [..., 4], key [..., 2] (anything that converts to uint32) -> [..., 4] uint32, Random123's philox4x32-10."""
    ctr = np.asarray(ctr, np.uint64)
    key = np.asarray(key, np.uint64)
    c0, c1, c2, c3 = (ctr[..., m] for m in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2                       # 32 x 32 -> 64 bits, exact in uint64
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _LO, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _LO)
        k0, k1 = (k0 + np.uint64(_W0)) & _LO, (k1 + np.uint64(_W1)) & _LO
    return np.stack([c0, c1, c2, c3], -1).astype(np.uint32)


def point_keys(seed, g, counter, n):
    """The packed keys [len(g), n] uint64 of points 0 .. n-1 of the global samples g (an int or a sequence)."""
    g = np.atleast_1d(np.asarray(g, np.uint64)) & _LO
    seed, counter = int(seed) & (2 ** 64 - 1), int(counter) & (2 ** 64 - 1)
    i = np.arange(n, dtype=np.uint64)
    ctr = np.empty((len(g), n, 4), np.uint64)
    ctr[..., 0] = i[None, :]
    ctr[..., 1] = g[:, None]
    ctr[..., 2] = counter & 0xFFFFFFFF
    ctr[..., 3] = counter >> 32
    w = philox4x32_10(ctr, [seed & 0xFFFFFFFF, seed >> 32]).astype(np.uint64)
    r = (w[..., 0] << np.uint64(32)) | w[..., 1]
    return (r & ~np.uint64(MAX_N - 1)) | i[None, :]


def permutation(seed, g, counter, n):
    """[len(g), n] int64: the points of each sample ranked by ascending key"""
    return np.argsort(point_keys(seed, g, counter, n), axis=1, kind="stable").astype(np.int64)


def sample_points(lengths, npoint, seed, counter, first_sample=0, table=None):
    """lengths: per-sample n (already clamped to [0, N]) -> out_idx [B, npoint] int64 as pcd_sample_points writes it.
    table: None or [B, >= max n] integer array; every drawn value v becomes table[b, v]."""
    B = len(lengths)
    out = np.empty((B, npoint), np.int64)
    for b, n in enumerate(lengths):
        n = int(n)
        if n == 0:
            out[b] = -1
            continue
        if n == npoint:
            row = np.arange(n, dtype=np.int64)
        else:
            perm = permutation(seed, first_sample + b, counter, n)[0]
            if n > npoint:
                row = perm[:npoint]
            else:
                whole = npoint // n * n
                row = np.concatenate([np.arange(whole, dtype=np.int64) % n, perm[:npoint - whole]])
        out[b] = row if table is None else np.asarray(table[b], np.int64)[row]
    return out
