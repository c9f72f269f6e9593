"""Reference for AOF's low-frequency projection and loop -- TEST / BENCH INFRASTRUCTURE ONLY (tests/,
__graft_entry__.smoke(), tools/aof_bench.py; the product never imports it).

  low_pass(V, x, dtype=np.float32)  the pcd_low_pass contract (include/pcdist.h) in numpy: every product and sum of the
                                    kernel in its order, each rounded to fp32 on its own (numpy never contracts a multiply
                                    and an add): bit for bit
  low_pass(V, x, dtype=np.float64)  V^T (V x) in float64 (the accuracy yardstick)
  host_loop                         AOF at B = 1 in the reference's shape: torch on the device, the library's low_pass and
                                    one victim forward on the concatenated clouds, and the best-result tracking and
                                    binary search in numpy on the host after every iteration (CW_attack.py's loop body)
"""
import numpy as np
import torch

BUTTERFLY = (16, 8, 4, 2, 1)


def low_pass(V, x, dtype=np.float32):
    """V [B,Kl,N] (rows: the basis vectors), x [B,N,3] -> y = V^T (V x) [B,N,3] in dtype"""
    V, x = np.asarray(V, np.float32), np.asarray(x, np.float32)
    if dtype == np.float64:
        V, x = V.astype(np.float64), x.astype(np.float64)
        return np.einsum("bkn,bkc->bnc", V, np.einsum("bkn,bnc->bkc", V, x))
    B, Kl, N = V.shape
    M = (N + 31) // 32
    # phase 1: lane l sums n = l (mod 32) in ascending n from +0; zero padding adds +0 to a sum that is never -0
    Vp = np.zeros((B, Kl, 32 * M), np.float32)
    Vp[..., :N] = V
    xp = np.zeros((B, 32 * M, 3), np.float32)
    xp[:, :N] = x
    Vp, xp = Vp.reshape(B, Kl, M, 32), xp.reshape(B, M, 32, 3)
    lanes = np.zeros((B, Kl, 32, 3), np.float32)
    with np.errstate(all="ignore"):
        for m in range(M):
            lanes = lanes + Vp[:, :, m, :, None] * xp[:, None, m]
        for o in BUTTERFLY:
            lanes = lanes + lanes[:, :, np.arange(32) ^ o]
        c = lanes[:, :, 0]                                                   # [B,Kl,3]
        # phase 2: k ascending from +0
        y = np.zeros((B, N, 3), np.float32)
        for k in range(Kl):
            y = y + V[:, k, :, None] * c[:, k, None, :]
    return y


def host_loop(model, low_pass_fn, data, target, basis, adv_func, dist_func, gamma, init_noise, attack_lr=1e-2,
              init_weight=10., max_weight=80., binary_step=2, num_iter=20, clip_func=None):
    """AOF for one cloud: data [1,N,3], target [1] on the device, basis [1,Kl,N], init_noise [binary_step,1,3,N];
    low_pass_fn = functional.low_pass -> (o_bestdist [1] float32, o_bestattack [1,N,3] float32, success [1]) as numpy"""
    dev = data.device
    ori = data.float().transpose(1, 2).contiguous().detach()
    label_val = target.cpu().numpy()
    lower, upper = np.zeros(1, np.float32), np.full(1, max_weight, np.float32)
    weight = np.full(1, init_weight, np.float32)
    o_bestdist, o_bestscore = np.full(1, 1e10, np.float32), np.full(1, -1)
    o_bestattack = np.zeros((1, 3, ori.shape[2]), np.float32)
    input_val = None
    for step in range(binary_step):
        adv = (ori + init_noise[step].to(dev) * 1e-7).requires_grad_(True)
        opt = torch.optim.Adam([adv], lr=attack_lr, weight_decay=0.)
        bestdist, bestscore = np.full(1, 1e10, np.float32), np.full(1, -1)
        w = torch.from_numpy(weight).to(dev)
        for _ in range(num_iter):
            low = low_pass_fn(adv.transpose(1, 2), basis).transpose(1, 2)
            logits = model(torch.cat([adv, low]))[0]
            pred_val = torch.argmax(logits[:1], dim=1).cpu().numpy()
            dist_val = torch.sqrt(torch.sum((adv - ori) ** 2, dim=[1, 2])).detach().cpu().numpy()
            input_val = adv.detach().cpu().numpy()
            for e, (dist, pred, label) in enumerate(zip(dist_val, pred_val, label_val)):
                if dist < bestdist[e] and pred != label:
                    bestdist[e], bestscore[e] = dist, pred
                if dist < o_bestdist[e] and pred != label:
                    o_bestdist[e], o_bestscore[e], o_bestattack[e] = dist, pred, input_val[e]
            adv_loss = ((1. - gamma) * adv_func(logits[:1], target, reduce=False)
                        + gamma * adv_func(logits[1:], target, reduce=False)).mean()
            dist_loss = dist_func(adv.transpose(1, 2), ori.transpose(1, 2), w, batch_avg=False).mean()
            loss = adv_loss + dist_loss
            opt.zero_grad(set_to_none=False)          # the reference's torch zeroed the gradient
            loss.backward()
            opt.step()
            if clip_func is not None:
                clip_func(adv.data, ori)
        for e, label in enumerate(label_val):
            if bestscore[e] != label and bestscore[e] != -1 and bestdist[e] <= o_bestdist[e]:
                lower[e] = max(lower[e], weight[e])
            else:
                upper[e] = min(upper[e], weight[e])
            weight[e] = (lower[e] + upper[e]) / np.float32(2.)
    fail = lower == 0.
    o_bestattack[fail] = input_val[fail]
    return o_bestdist, o_bestattack.transpose(0, 2, 1), ~fail
