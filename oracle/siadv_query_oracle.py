"""Reference for SI-Adv's query-based attack -- TEST / BENCH INFRASTRUCTURE ONLY (tests/, tools/siadv_query_bench.py;
the product never imports it).

  sensitivity, query_round, trial   numpy float32 restatements of pcd_si_sensitivity and pcd_si_query_round
                                    (include/pcdist.h): every operation in the kernels' order, each rounded to fp32 on
                                    its own, the frames, products and tree sum of siadv_oracle: bit for bit
  run                               the whole attack loop over query_round, for a numpy black box
  host_loop                         the reference's shape: one sample (B = 1) at a time, torch ops on the sample's
                                    device, the black box's logits copied to the host and one Python decision per query.
                                    Its arithmetic is the same contract, so its results are the device loop's bits.
"""
import numpy as np

from .siadv_oracle import _cols, _rows, spin_axis, tree_sum

ACTIVE, SUCCESS, FAILED = 0, 1, 2
SIGMA, CURSOR, QUERIES, STATUS = 0, 1, 2, 3
f32 = np.float32


def sensitivity(grad, normal):
    """grad, normal [B,N,3] -> (s [B,N], dir [B,N,2], order [B,N] int32: descending s, ties by the lower index)"""
    grad, normal = np.asarray(grad, f32), np.asarray(normal, f32)
    with np.errstate(all="ignore"):
        g = _rows(spin_axis(normal, f32), grad)
        s = np.sqrt(g[..., 0] * g[..., 0] + g[..., 1] * g[..., 1])
        d = g[..., :2] / (s + f32(1e-16))[..., None]
    bad = np.isnan(s)
    s = np.where(bad, f32(-1), s)
    d = np.where(bad[..., None], f32(0), d)
    order = np.argsort(-s.astype(np.float64), axis=1, kind="stable").astype(np.int32)
    return s, d, order


def score(row, y, targeted):
    """one logits row -> (valid, margin, success)"""
    row = np.asarray(row, f32)
    C = row.shape[0]
    if not 0 <= y < C:
        return False, f32(np.nan), False
    other = max(f32(-10000), max((row[j] for j in range(C) if j != y), default=f32(-np.inf)))
    with np.errstate(all="ignore"):
        margin = f32(other - row[y]) if targeted else f32(row[y] - other)
    valid = not np.isnan(row).any() and bool(np.isfinite(margin))
    arg = int(np.argmax(row))
    return valid, margin, valid and ((arg == y) if targeted else (arg != y))


def trial(cloud, ori, normal, dir, i, sigma, step_size, eps):
    """one sample's next trial [N,3]: point i (-1: none) moved by sigma * step_size along dir in its tangent plane,
    then the whole cloud clipped to eps"""
    p = np.array(cloud, f32)
    ori = np.asarray(ori, f32)
    with np.errstate(all="ignore"):
        if i >= 0:
            n = np.asarray(normal, f32)[i]
            q = p[i]
            c = (q[0] * n[0] + q[1] * n[1]) + q[2] * n[2]
            t = c * n
            u = spin_axis(n, f32)
            pp = _rows(u, q + t)
            sa = f32(sigma) * f32(step_size)
            pp[0] = pp[0] + sa * dir[i][0]
            pp[1] = pp[1] + sa * dir[i][1]
            p[i] = _cols(u, pp) - t
        d = p - ori
        s = f32(eps) / (np.sqrt(tree_sum(d * d, axis=0)) + f32(1e-9))
        s = np.where(s > 1, f32(1), s)                                  # NaN stays NaN
        return ori + d * s


def query_round(logits, target, ori, normal, order, dir, cloud, trial_, state, best, step_size, eps, max_query,
                targeted=False, active=None):
    """pcd_si_query_round on copies -> (cloud, trial, state, best, active)"""
    cloud, trial_, state, best = (np.array(x) for x in (cloud, trial_, state, best))
    logits = np.asarray(logits, f32)
    B, N = cloud.shape[:2]
    for b in range(B):
        st = state[b]
        if st[STATUS] != ACTIVE:
            continue
        valid, margin, success = score(logits[b], int(target[b]), targeted)
        st[QUERIES] += 1
        take = False
        if st[QUERIES] == 1:
            best[b] = margin
            if success:
                st[STATUS], take = SUCCESS, True
        elif success:
            st[STATUS], take = SUCCESS, True
        elif valid and margin < best[b]:
            best[b], take = margin, True
            st[CURSOR] += 1
            st[SIGMA] = -1
        elif st[SIGMA] == -1:
            st[SIGMA] = 1
        else:
            st[CURSOR] += 1
            st[SIGMA] = -1
        if st[STATUS] == ACTIVE and st[QUERIES] >= max_query:
            st[STATUS] = FAILED
        if take:
            cloud[b] = trial_[b]
        if st[STATUS] != ACTIVE:
            trial_[b] = cloud[b]
            if active is not None:
                active = active - 1
            continue
        i = int(order[b][st[CURSOR] % N])
        trial_[b] = trial(cloud[b], ori[b], normal[b], dir[b], i if 0 <= i < N else -1, st[SIGMA], step_size, eps)
    return cloud, trial_, state, best, active


def initial_state(B):
    return np.tile(np.array([-1, 0, 0, ACTIVE], np.int32), (B, 1))


def run(black_box, ori, normal, grad, target, step_size, eps, max_query, targeted=False):
    """the attack loop over query_round: black_box(clouds [B,N,3]) -> logits [B,C] float32 (the surrogate's gradient
    grad is given) -> (adv, queries, success, rounds)"""
    ori = np.asarray(ori, f32)
    _, dir, order = sensitivity(grad, normal)
    cloud, tr, state, best = ori.copy(), ori.copy(), initial_state(ori.shape[0]), np.zeros(ori.shape[0], f32)
    rounds = 0
    while rounds < max_query and (state[:, STATUS] == ACTIVE).any():
        cloud, tr, state, best, _ = query_round(black_box(tr), target, ori, normal, order, dir, cloud, tr, state, best,
                                                step_size, eps, max_query, targeted)
        rounds += 1
    return cloud, state[:, QUERIES].astype(np.int64), state[:, STATUS] == SUCCESS, rounds


# ---------------------------------------------------------------------------------------------- the reference's shape
def _full(x, v):
    """v as a tensor shaped like x: a CPU scalar operand would make torch divide by multiplying with its reciprocal"""
    import torch
    return torch.full_like(x, float(np.float32(v)))


def _spin_axis_torch(n):
    import torch
    x, y, z = n.unbind(-1)
    zero = torch.zeros_like(z)
    zz = z * z
    den = torch.sqrt(1 - zz)
    u = torch.stack([torch.stack([y / den, (-x) / den, zero], -1),
                     torch.stack([(x * z) / den, (y * z) / den, -den], -1),
                     torch.stack([x, y, z], -1)], -2)
    r = _full(z, 1 / np.sqrt(2))
    w = z / _full(z, np.sqrt(2))
    ub = torch.stack([torch.stack([r, -r, zero], -1), torch.stack([w, w, zero], -1), torch.stack([zero, zero, z], -1)], -2)
    return torch.where(((zz - 1).abs() < 1e-4)[..., None, None], ub, u)


def _tree_sum_torch(v):
    """tree_sum over dim 0 with torch adds"""
    import torch
    n = v.shape[0]
    m = 1
    while m < n:
        m *= 2
    t = torch.cat([v, torch.zeros((m - n,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)])
    while t.shape[0] > 1:
        t = t[0::2] + t[1::2]
    return t[0]


def margin_loss(logits, target, targeted):
    """the per-sample C&W margin without the clamp (SIAdvAttack._loss's terms), differentiable"""
    import torch
    one_hot = torch.zeros_like(logits).scatter_(1, target.view(-1, 1), 1.)
    real = torch.sum(one_hot * logits, dim=1)
    other = torch.max((1. - one_hot) * logits - one_hot * 10000., dim=1)[0]
    return other - real if targeted else real - other


def host_loop(model, ori, normal, target, eps=0.16, step_size=0.05, max_query=2000, targeted=False, surrogate=None):
    """One sample: ori, normal [N,3] (unit normals), target an int -> (adv [N,3], pred, success, queries).  The
    black box runs under no_grad, its logits go to the host after every query and Python decides."""
    import torch
    dev = ori.device
    surrogate = model if surrogate is None else surrogate
    x = ori[None].detach().clone().requires_grad_(True)
    tgt = torch.tensor([int(target)], device=dev)
    with torch.enable_grad():
        grad, = torch.autograd.grad(margin_loss(surrogate(x.transpose(1, 2))[0], tgt, targeted).sum(), x)
    g, n = grad[0], normal
    u = _spin_axis_torch(n)
    gr = (u[..., 0] * g[..., None, 0] + u[..., 1] * g[..., None, 1]) + u[..., 2] * g[..., None, 2]
    s = torch.sqrt(gr[:, 0] * gr[:, 0] + gr[:, 1] * gr[:, 1])
    d = gr[:, :2] / (s + 1e-16)[:, None]
    bad = torch.isnan(s)
    s = torch.where(bad, torch.full_like(s, -1.), s)
    d = torch.where(bad[:, None], torch.zeros_like(d), d)
    order = torch.sort(s, descending=True, stable=True)[1].tolist()
    N = ori.shape[0]
    a = np.float32(step_size)

    def make_trial(p, i, sigma):
        p = p.clone()
        q, nn = p[i], n[i]
        c = (q[0] * nn[0] + q[1] * nn[1]) + q[2] * nn[2]
        t = c * nn
        ui = u[i]
        pp = (ui[:, 0] * (q + t)[0] + ui[:, 1] * (q + t)[1]) + ui[:, 2] * (q + t)[2]
        sa = _full(pp[0], np.float32(sigma) * a)
        pp = torch.stack([pp[0] + sa * d[i, 0], pp[1] + sa * d[i, 1], pp[2]])
        p[i] = (ui[0, :] * pp[0] + ui[1, :] * pp[1]) + ui[2, :] * pp[2] - t
        dd = p - ori
        sc = _full(dd[0], eps) / (torch.sqrt(_tree_sum_torch(dd * dd)) + 1e-9)
        sc = torch.where(sc > 1, torch.ones_like(sc), sc)
        return ori + dd * sc

    def query(p):
        with torch.no_grad():
            return score(model(p[None].transpose(1, 2))[0][0].float().cpu().numpy(), int(target), targeted)

    P = ori.clone()
    valid, best, success = query(P)
    q, c, sigma = 1, 0, -1
    while not success and q < max_query:
        tr = make_trial(P, order[c % N], sigma)
        valid, margin, success = query(tr)
        q += 1
        if success:
            P = tr
        elif valid and margin < best:
            P, best, c, sigma = tr, margin, c + 1, -1
        elif sigma == -1:
            sigma = 1
        else:
            c, sigma = c + 1, -1
    with torch.no_grad():
        pred = int(model(P[None].transpose(1, 2))[0].argmax(1).item())
    return P, pred, success, q
