"""Device-resident, batched SI-Adv shape-invariant attack <- attack/SIadv/SIadv_attack.py
(PointCloudAttack.shape_invariant_ifgm, the white-box / transfer attack of SI-Adv).

Every iteration of the reference runs at B = 1, copies the cloud to the host for open3d's normal estimation and builds
the spin-axis frames and the step from about 40 small torch ops.  Here an iteration is the victim's forward and
backward plus four library launches, with no host synchronisation:
  * the step: functional.shape_invariant_step_ (one fused kernel: spin-axis frames, tangent-plane gradient normalised
    per sample, the inverse transform and the reference's clip);
  * the normals of the moved cloud: functional.estimate_normals (the self k-NN, then local_frames), in place of open3d's
    KD-tree estimate.  Its signs and neighbour-tie order are this library's; the step does not depend on the signs.
One whole iteration can be captured into a CUDA graph and replayed (`use_graph=True`).

Defences come in through the model: DefendedVictim(victim, SRSDefense / SORDefense(..., sampler=PointSampler(...)))
is the reference's wb_classifier(pre_head(points)), and eval_model plays its black-box classifier in transfer runs.
There is no install() patch for this module: the class layout of PointCloudAttack is not recorded here, as for
defense.py.  The query-based attack (shape_invariant_query_attack) is not restated.
"""
import torch

from . import functional as F

__all__ = ["SIAdvAttack"]


def _samplers(model):
    """the PointSamplers of the defences inside the model (their draw counters are part of the attack's state)"""
    out = []
    for mod in model.modules():
        s = getattr(mod, "sampler", None)
        if isinstance(s, F.PointSampler) and all(s is not o for o in out):
            out.append(s)
    return out


class SIAdvAttack:
    """shape_invariant_ifgm for batches: max_steps iterations (no early stop) of
        logits = model(P.transpose(1, 2))[0]
        loss   = sum over the batch of the C&W margin with kappa = 0: clamp(real - other, min=0), or
                 clamp(other - real, min=0) when targeted (real: the logit of target, other: the largest other logit)
        grad   = dL/dP;  P = shape_invariant_step_(P, ori, normal, grad, step_size, eps, step_scale)
        normal = estimate_normals(P, knn)
    step_scale keeps the reference's hard-coded sqrt(3 * 1024) whatever N is.  The victim is in eval mode and the step
    is normalised per sample, so a sample's result does not depend on the rest of the batch (which is also what makes
    sharding work with no extra code)."""

    def __init__(self, model, eps=0.16, step_size=0.007, max_steps=50, step_scale=F.SI_STEP_SCALE, knn=20,
                 eval_model=None, targeted=False, use_graph=False):
        self.model = model.eval()
        for p in self.model.parameters():
            p.requires_grad_(False)
        self.eval_model = eval_model.eval() if eval_model is not None else None
        self.eps, self.step_size, self.max_steps, self.step_scale = float(eps), float(step_size), int(max_steps), float(step_scale)
        self.knn, self.targeted, self.use_graph = int(knn), bool(targeted), bool(use_graph)
        self.loop_ms = 0.0                       # device time of the iteration loop of the last attack()

    def _loss(self, logits, target):
        one_hot = torch.zeros_like(logits).scatter_(1, target.view(-1, 1), 1.)
        real = torch.sum(one_hot * logits, dim=1)
        other = torch.max((1. - one_hot) * logits - one_hot * 10000., dim=1)[0]
        margin = other - real if self.targeted else real - other
        return torch.clamp(margin, min=0.).sum()

    def _iteration(self, st):
        pc = st["pc"]
        with torch.enable_grad():
            x = pc.detach().requires_grad_(True)
            loss = self._loss(self.model(x.transpose(1, 2))[0], st["target"])
            grad, = torch.autograd.grad(loss, x)
        with torch.no_grad():
            F.shape_invariant_step_(pc, st["ori"], st["normal"], grad, self.step_size, self.eps, self.step_scale)
            st["normal"].copy_(F.estimate_normals(pc, self.knn))
            st["loss"].copy_(loss.detach())

    def attack(self, points, target):
        """points [B,N,3] (or [B,N,6] with normals in channels 3:6), target [B] ->
        (adv [B,N,3], pred [B] = argmax of eval_model (or model) on adv, success [B])"""
        dev = points.device
        if dev.type != "cuda":
            raise RuntimeError("SIAdvAttack runs on CUDA only")
        if points.dim() != 3 or points.shape[2] not in (3, 6):
            raise ValueError(f"points must be [B, N, 3] or [B, N, 6], got {tuple(points.shape)}")
        data = points.detach().float()
        ori = data[..., :3].contiguous()
        if data.shape[2] == 6:
            n = data[..., 3:]
            normal = (n / torch.sqrt(torch.sum(n * n, dim=-1, keepdim=True))).contiguous()
        else:
            normal = F.estimate_normals(ori, self.knn)
        st = {"ori": ori, "pc": ori.clone(), "normal": normal, "target": target.long().to(dev),
              "loss": torch.zeros((), device=dev)}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if self.use_graph:
            graph = self._capture(st)
            e0.record()
            for _ in range(self.max_steps):
                graph.replay()
        else:
            e0.record()
            for _ in range(self.max_steps):
                self._iteration(st)
        e1.record()
        with torch.no_grad():
            judge = self.model if self.eval_model is None else self.eval_model
            pred = torch.argmax(judge(st["pc"].transpose(1, 2))[0], dim=1)
        success = pred == st["target"] if self.targeted else pred != st["target"]
        torch.cuda.synchronize(dev)
        self.loop_ms = e0.elapsed_time(e1)
        return st["pc"], pred, success

    def _capture(self, st, warmup=3):
        """Capture one iteration.  The warm-up iterations run on the real state tensors (the graph records their
        addresses), so the cloud, the normals and the draw counters of any device-sampled defence are saved before
        and restored after: replaying max_steps times is exactly max_steps iterations."""
        saved = {k: v.clone() for k, v in st.items()}
        samplers = _samplers(self.model)
        counters = [s.state.clone() for s in samplers]
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
        for k, v in saved.items():
            st[k].copy_(v)
        for s, c in zip(samplers, counters):
            s.state.copy_(c)
        return g
