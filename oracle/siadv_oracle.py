"""Reference for the SI-Adv step and normals -- TEST / BENCH INFRASTRUCTURE ONLY (tests/, __graft_entry__.smoke(),
tools/siadv_bench.py; the product never imports it).

A numpy restatement of the pcd_si_step contract (include/pcdist.h), which restates SI-Adv's published
get_spin_axis_matrix / get_transformed_point_cloud / get_original_point_cloud / shape_invariant_ifgm:
  si_step(..., dtype=np.float32)  every operation of the kernel, in its order, each rounded to fp32 on its own (numpy
                                  never contracts a multiply and an add), the tree sums included: bit for bit
  si_step(..., dtype=np.float64)  the same steps in float64 (the accuracy yardstick)
  normals64                       the exact k-NN (squared distances in float64, self included) and the eigenvector of
                                  the smallest eigenvalue of the neighbourhood covariance (np.linalg.eigh)
"""
import numpy as np

BOUNDARY = 1e-4


def tree_sum(v, axis=-1):
    """Pairwise tree sum along axis: the aligned power-of-two tree of pcd_si_step, left + right at every node.  The
    values are zero-padded to a power of two; every summand here is a square, so a +0 leaf changes no node's bits."""
    v = np.moveaxis(np.asarray(v), axis, -1)
    n = v.shape[-1]
    m = 1
    while m < n:
        m *= 2
    t = np.concatenate([v, np.zeros(v.shape[:-1] + (m - n,), v.dtype)], -1)
    while t.shape[-1] > 1:
        t = t[..., 0::2] + t[..., 1::2]
    return t[..., 0]


def spin_axis(n, dtype=np.float32):
    """normal [..., 3] -> U [..., 3, 3] (rows u0, u1, u2), get_spin_axis_matrix with the boundary case"""
    n = np.asarray(n, dtype)
    x, y, z = n[..., 0], n[..., 1], n[..., 2]
    one = dtype(1)
    zz = z * z
    with np.errstate(all="ignore"):
        den = np.sqrt(one - zz)
        u = np.stack([np.stack([y / den, (-x) / den, np.zeros_like(z)], -1),
                      np.stack([(x * z) / den, (y * z) / den, -den], -1),
                      np.stack([x, y, z], -1)], -2)
        r, s2 = dtype(1 / np.sqrt(2)), dtype(np.sqrt(2))                 # fp32(1/sqrt 2), fp32(sqrt 2) in float32
        w = z / s2
        ub = np.stack([np.stack([np.full_like(z, r), np.full_like(z, -r), np.zeros_like(z)], -1),
                       np.stack([w, w, np.zeros_like(z)], -1),
                       np.stack([np.zeros_like(z), np.zeros_like(z), z], -1)], -2)
        edge = np.abs(zz - one) < dtype(BOUNDARY)
    return np.where(edge[..., None, None], ub, u)


def _rows(u, a):
    """(u_r0*a0 + u_r1*a1) + u_r2*a2 for r = 0, 1, 2"""
    return (u[..., 0] * a[..., None, 0] + u[..., 1] * a[..., None, 1]) + u[..., 2] * a[..., None, 2]


def _cols(u, a):
    """(u_0r*a0 + u_1r*a1) + u_2r*a2 for r = 0, 1, 2"""
    return (u[..., 0, :] * a[..., 0, None] + u[..., 1, :] * a[..., 1, None]) + u[..., 2, :] * a[..., 2, None]


def si_step(pc, ori, normal, grad, step_size, eps, step_scale=np.sqrt(3 * 1024), dtype=np.float32, clip=True):
    """pc, ori, normal, grad [B,N,3] -> (new pc [B,N,3], gnorm [B]) in dtype.  clip=False returns p_new of step 6."""
    pc, ori, normal, grad = (np.asarray(t, np.float32).astype(dtype) for t in (pc, ori, normal, grad))
    a = dtype(np.float32(float(step_size) * float(step_scale))) if dtype == np.float32 else dtype(step_size * step_scale)
    tiny = dtype(1e-9)
    with np.errstate(all="ignore"):
        c = (pc[..., 0] * normal[..., 0] + pc[..., 1] * normal[..., 1]) + pc[..., 2] * normal[..., 2]
        t = c[..., None] * normal
        q = pc + t
        u = spin_axis(normal, dtype)
        pp = _rows(u, q)
        g = _rows(u, grad)
        g[..., 2] = 0
        norm = np.sqrt(tree_sum(g[..., 0] * g[..., 0] + g[..., 1] * g[..., 1], axis=1))
        den = (norm + tiny)[:, None, None]
        p2 = pp - (a * g) / den
        pn = _cols(u, p2) - t
        if not clip:
            return pn, norm
        d = pn - ori
        nc = np.sqrt(tree_sum(d * d, axis=1))                            # [B, 3]
        s = dtype(eps) / (nc + tiny)
        s = np.where(s > 1, dtype(1), s)                                  # NaN stays NaN
        return ori + d * s[:, None, :], norm


def knn64(pc, k):
    """exact k-NN of every point of pc [B,N,3] among the same cloud, self included, by (squared distance, index) ->
    (idx [B,N,k], gap [B,N]: the (k+1)-th smallest squared distance minus the k-th, +inf when N == k)"""
    p = np.asarray(pc, np.float64)
    d = ((p[:, :, None, :] - p[:, None, :, :]) ** 2).sum(-1)
    order = np.argsort(d, axis=-1, kind="stable")
    idx = order[..., :k]
    ds = np.take_along_axis(d, order[..., :k + 1], -1)
    gap = ds[..., k] - ds[..., k - 1] if d.shape[-1] > k else np.full(d.shape[:2], np.inf)
    return idx, gap


def normals64(pc, k=20):
    """float64 unit normals [B,N,3] (sign arbitrary) of the k-NN patches, self included, the neighbour gaps [B,N] and the
    covariance eigenvalues [B,N,3] (ascending)"""
    p = np.asarray(pc, np.float64)
    idx, gap = knn64(p, k)
    nb = p[np.arange(p.shape[0])[:, None, None], idx]
    cen = nb - nb.mean(-2, keepdims=True)
    cov = np.einsum("bnki,bnkj->bnij", cen, cen)
    w, v = np.linalg.eigh(cov)
    return v[..., :, 0], gap, w
