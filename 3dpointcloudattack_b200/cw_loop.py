"""Device-resident, batch-safe CW iteration loop (SURVEY.md section 8f-1, the caller of the path).

Same optimisation as attack/CW/CW_attack.py:57-260 (Adam on the cloud, per-sample binary search
of the distance weight, best-result tracking, clip/projection after every step) restated so that
it works for B > 1 and never leaves the GPU inside the loop:

  * the reference's per-iteration `.cpu().numpy()` copies and Python per-sample loop
    (CW_attack.py:129-153) become `torch.where` updates of device tensors;
  * `current_weight` / bounds are device tensors (the reference rebuilds a CPU tensor and
    `.cuda()`s it every iteration, CW_attack.py:161-163);
  * one whole iteration (victim forward+backward, distance forward+backward, Adam step, clip,
    tracking) can be captured into a CUDA graph and replayed (`use_graph=True`).

`dist_func(adv[B,K,3], ori[B,K,3], weights[B], batch_avg=False) -> [B]` is any of this package's
ChamferDist / HausdorffDist / ChamferkNNDist (or a sum of them); `model(x[B,3,K])` returns logits
first, as every victim of the reference does.
"""
import torch
import torch.nn as nn

from . import functional as F


class UntargetedLogitsAdvLoss(nn.Module):
    """attack/CW/CW_utils/adv_utils.py:52-78 without the hard-coded .cuda(); returns [B] when
    reduce=False."""

    def __init__(self, kappa=0.):
        super().__init__()
        self.kappa = kappa

    def forward(self, logits, targets, reduce=True):
        one_hot = torch.zeros_like(logits).scatter_(1, targets.view(-1, 1).long(), 1.)
        real = torch.sum(one_hot * logits, dim=1)
        other = torch.max((1. - one_hot) * logits - one_hot * 10000., dim=1)[0]
        loss = torch.clamp(real - other + self.kappa, min=0.)
        return loss.mean() if reduce else loss


class ClipPointsLinf(nn.Module):
    """attack/CW/CW_utils/clip_utils.py:32-56 (per-point L2 clip of the perturbation), IN PLACE, one launch
    (functional.clip_points_) instead of the reference's nine elementwise ops; bit-identical to that chain."""

    def __init__(self, budget):
        super().__init__()
        self.budget = budget

    @torch.no_grad()
    def forward(self, pc, ori_pc):
        return F.clip_points_(pc, ori_pc, self.budget, F.CLIP_LINF)


class ClipPointsL2(nn.Module):
    """attack/CW/CW_utils/clip_utils.py:5-29 (one scale per sample), IN PLACE, one launch."""

    def __init__(self, budget):
        super().__init__()
        self.budget = budget

    @torch.no_grad()
    def forward(self, pc, ori_pc):
        return F.clip_points_(pc, ori_pc, self.budget, F.CLIP_L2)


class ProjectInnerClipLinf(nn.Module):
    """attack/CW/CW_utils/clip_utils.py:59-136: points pushed inside the surface (negative offset
    along the normal) are projected back onto it, then the per-point L2 clip; IN PLACE, one launch, batch safe
    (the reference's dim-less torch.cross picks the wrong axis for B == 3).  normal=None: the clip alone."""

    def __init__(self, budget):
        super().__init__()
        self.budget = budget

    @torch.no_grad()
    def forward(self, pc, ori_pc, normal=None):
        if normal is None:
            return F.clip_points_(pc, ori_pc, self.budget, F.CLIP_LINF)
        return F.clip_points_(pc, ori_pc, self.budget, F.CLIP_PROJECT_LINF, normal=normal)


class CWAttack:
    def __init__(self, model, adv_func, dist_func, attack_lr=1e-2, init_weight=10., max_weight=80.,
                 binary_step=10, num_iter=500, clip_func=None, global_batch=None, use_graph=False,
                 attack_method="untarget"):
        if attack_method not in ("untarget", "target"):
            raise ValueError("attack_method must be 'untarget' or 'target' (CW_attack.py:28)")
        self.attack_method = attack_method
        self.model = model.eval()
        for p in self.model.parameters():
            p.requires_grad_(False)
        self.adv_func, self.dist_func, self.clip_func = adv_func, dist_func, clip_func
        self.attack_lr, self.init_weight, self.max_weight = attack_lr, init_weight, max_weight
        self.binary_step, self.num_iter = binary_step, num_iter
        self.global_batch = global_batch          # for 1/B_global gradient scaling when the batch is sharded
        self.use_graph = use_graph
        self.loop_ms = 0.0                        # device time spent in the iteration loops of the last attack()

    def _victim(self, adv, target):
        """the victim's forward: (logits of adv [B, classes], which tracking and success use; the adversarial term summed
        over the batch).  AOFAttack overrides it."""
        logits = self.model(adv)[0]
        return logits, self.adv_func(logits, target, reduce=False).sum()

    # one optimisation iteration on the state tensors (all updates in place -> graph capturable)
    def _iteration(self, st):
        adv, ori, target = st["adv"], st["ori"], st["target"]
        logits, adv_sum = self._victim(adv, target)
        pred = torch.argmax(logits, dim=1)
        with torch.no_grad():
            dist_val = torch.sqrt(torch.sum((adv - ori) ** 2, dim=[1, 2]))
            st["last_input"].copy_(adv)          # `input_val`: the iterate this iteration STARTS from (CW_attack.py:132)
            ok = (pred != target) if self.attack_method == "untarget" else (pred == target)   # CW_attack.py:136-153
            better = ok & (dist_val < st["bestdist"])
            st["bestdist"].copy_(torch.where(better, dist_val, st["bestdist"]))
            st["bestscore"].copy_(torch.where(better, pred, st["bestscore"]))
            o_better = ok & (dist_val < st["o_bestdist"])
            st["o_bestdist"].copy_(torch.where(o_better, dist_val, st["o_bestdist"]))
            st["o_bestscore"].copy_(torch.where(o_better, pred, st["o_bestscore"]))
            st["o_bestattack"].copy_(torch.where(o_better[:, None, None], adv, st["o_bestattack"]))
        B = adv.shape[0]
        denom = float(self.global_batch or B)
        adv_loss = adv_sum / denom
        dist_loss = self.dist_func(adv.transpose(1, 2), ori.transpose(1, 2), st["weight"], batch_avg=False).sum() / denom
        loss = adv_loss + dist_loss
        st["opt"].zero_grad(set_to_none=False)
        loss.backward()
        st["opt"].step()
        if self.clip_func is not None:
            self.clip_func(adv.data, ori)
        st["loss"].copy_(loss.detach())

    def attack(self, data, target, seed=0, first_sample=0, init_noise=None):
        """data [B, K, 3], target [B] -> (o_bestdist[B], o_bestattack[B,K,3], success mask[B]).
        init_noise [binary_step, B, 3, K] replaces the per-sample generator draws (parity tests
        replay the reference's own torch.randn draws, CW_attack.py:94)."""
        from .sharding import per_sample_noise
        dev = data.device
        if dev.type != "cuda":
            raise RuntimeError("CWAttack runs on CUDA only")
        B, K = data.shape[:2]
        ori = data.float().transpose(1, 2).contiguous().detach()
        target = target.long().to(dev)
        lower = torch.zeros(B, device=dev)
        upper = torch.full((B,), float(self.max_weight), device=dev)
        st = {
            "ori": ori, "target": target,
            "weight": torch.full((B,), float(self.init_weight), device=dev),
            "o_bestdist": torch.full((B,), 1e10, device=dev),
            "o_bestscore": torch.full((B,), -1, dtype=torch.long, device=dev),
            "o_bestattack": torch.zeros((B, 3, K), device=dev),
            "bestdist": torch.full((B,), 1e10, device=dev),
            "bestscore": torch.full((B,), -1, dtype=torch.long, device=dev),
            "loss": torch.zeros((), device=dev),
            "last_input": ori.clone(),
            "adv": ori.clone().requires_grad_(True),
        }
        graph = None
        spans = []
        for step in range(self.binary_step):
            if init_noise is not None:
                noise = init_noise[step].to(dev) * 1e-7
            else:
                noise = per_sample_noise((3, K), first_sample, B, 1e-7, seed=seed + step, device=dev)
            with torch.no_grad():
                st["adv"].copy_(ori + noise)
                st["bestdist"].fill_(1e10); st["bestscore"].fill_(-1)
            st["adv"].grad = None
            st["opt"] = torch.optim.Adam([st["adv"]], lr=self.attack_lr, weight_decay=0.,
                                         capturable=self.use_graph, foreach=True)
            if self.use_graph:
                graph = self._capture(st)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if self.use_graph:
                for _ in range(self.num_iter):
                    graph.replay()
            else:
                for _ in range(self.num_iter):
                    self._iteration(st)
            e1.record()
            spans.append((e0, e1))
            with torch.no_grad():                     # binary search of the distance weight (CW_attack.py:182-200)
                hit = (st["bestscore"] != target) if self.attack_method == "untarget" else (st["bestscore"] == target)
                succ = hit & (st["bestscore"] != -1) & (st["bestdist"] <= st["o_bestdist"])
                lower = torch.where(succ, torch.maximum(lower, st["weight"]), lower)
                upper = torch.where(succ, upper, torch.minimum(upper, st["weight"]))
                st["weight"].copy_((lower + upper) / 2.)
        with torch.no_grad():        # samples never attacked successfully get `input_val` of the last iteration, i.e. the
            fail = lower == 0.       # iterate BEFORE the final Adam step and clip (CW_attack.py:203-206)
            st["o_bestattack"].copy_(torch.where(fail[:, None, None], st["last_input"], st["o_bestattack"]))
        torch.cuda.synchronize(dev)
        self.loop_ms = sum(a.elapsed_time(b) for a, b in spans)
        return st["o_bestdist"], st["o_bestattack"].transpose(1, 2).contiguous(), ~fail

    def _capture(self, st, warmup=3):
        """Capture one iteration.  The warm-up iterations run on the real state tensors (the graph must
        record their addresses), so the state -- cloud, trackers, Adam moments and step count -- is
        saved before and restored after: replaying num_iter times is exactly num_iter iterations."""
        saved = {k: v.detach().clone() for k, v in st.items() if isinstance(v, torch.Tensor)}
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._iteration(st)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            self._iteration(st)
        with torch.no_grad():
            for k, v in saved.items():
                st[k].copy_(v)
            for state in st["opt"].state.values():
                for t in state.values():
                    if isinstance(t, torch.Tensor):
                        t.zero_()
            if st["adv"].grad is not None:
                st["adv"].grad.zero_()
        return g


class KNNAttack:
    """Device-resident, batch-safe restatement of the kNN attack loop (attack/KNN/KNN_attack.py:56-246):
    one long Adam loop, loss = adv_func(logits).mean() + dist_func(adv, ori).mean() * K, then
    clip_func(adv, ori, normal) after every step (normal = the cloud itself when the input has
    only xyz, KNN_attack.py:70-74).  `dist_func(adv[B,K,3], ori[B,K,3], weights=None,
    batch_avg=False) -> [B]` is this package's ChamferDist / ChamferkNNDist."""

    def __init__(self, model, adv_func, dist_func, clip_func, attack_lr=1e-3, num_iter=2500, global_batch=None,
                 use_graph=False):
        self.model = model.eval()
        for p in self.model.parameters():
            p.requires_grad_(False)
        self.adv_func, self.dist_func, self.clip_func = adv_func, dist_func, clip_func
        self.attack_lr, self.num_iter = attack_lr, num_iter
        self.global_batch, self.use_graph = global_batch, use_graph
        self.loop_ms = 0.0

    def _iteration(self, st):
        adv, ori = st["adv"], st["ori"]
        K = adv.shape[2]
        out = self.model(adv)
        logits = out[0] if isinstance(out, tuple) else out
        denom = float(self.global_batch or adv.shape[0])
        adv_loss = self.adv_func(logits, st["target"], reduce=False).sum() / denom
        dist_loss = self.dist_func(adv.transpose(1, 2), ori.transpose(1, 2), None, batch_avg=False).sum() / denom * K
        loss = adv_loss + dist_loss
        st["opt"].zero_grad(set_to_none=False)
        loss.backward()
        st["opt"].step()
        self.clip_func(adv.data, ori, st["normal"])
        st["loss"].copy_(loss.detach())

    def attack(self, data, target, seed=0, first_sample=0, init_noise=None):
        """data [B, K, 3] (or [B, K, 6] with normals), target [B] -> (adv[B,K,3], success mask[B])."""
        from .sharding import per_sample_noise
        dev = data.device
        if dev.type != "cuda":
            raise RuntimeError("KNNAttack runs on CUDA only")
        B, K = data.shape[:2]
        full = data.float().transpose(1, 2).contiguous().detach()
        ori = full[:, :3].contiguous()
        normal = ori if full.shape[1] == 3 else full[:, 3:].contiguous()
        target = target.long().to(dev)
        noise = init_noise.to(dev) * 1e-7 if init_noise is not None else \
            per_sample_noise((3, K), first_sample, B, 1e-7, seed=seed, device=dev)
        st = {"ori": ori, "normal": normal, "target": target, "loss": torch.zeros((), device=dev),
              "adv": (ori + noise).requires_grad_(True)}
        st["opt"] = torch.optim.Adam([st["adv"]], lr=self.attack_lr, weight_decay=0., capturable=self.use_graph, foreach=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if self.use_graph:
            graph = CWAttack._capture(self, st)
            e0.record()
            for _ in range(self.num_iter):
                graph.replay()
        else:
            e0.record()
            for _ in range(self.num_iter):
                self._iteration(st)
        e1.record()
        with torch.no_grad():
            out = self.model(st["adv"])
            pred = torch.argmax(out[0] if isinstance(out, tuple) else out, dim=-1)
        torch.cuda.synchronize(dev)
        self.loop_ms = e0.elapsed_time(e1)
        return st["adv"].detach().transpose(1, 2).contiguous(), pred != target
