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
SI-Adv's query-based black-box attack (shape_invariant_query_attack) is SIAdvQueryAttack: B clouds are queried
together, and one query round is a no-grad forward of the black box on the B trial clouds plus ONE library launch
(functional.si_query_round_), which scores the logits, makes every sample's accept / reject decision and builds every
sample's next trial.  Only a periodic stop check reads back to the host.

There is no install() patch for this module: the class layout of PointCloudAttack is not recorded here, as for
defense.py.
"""
import torch

from . import functional as F

__all__ = ["SIAdvAttack", "SIAdvQueryAttack"]


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
        normal = _unit_normals(data, self.knn)
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


def _unit_normals(data, knn):
    """the normals of [B,N,6] input (channels 3:6, normalised), else estimate_normals of the cloud"""
    if data.shape[2] == 6:
        n = data[..., 3:]
        return (n / torch.sqrt(torch.sum(n * n, dim=-1, keepdim=True))).contiguous()
    return F.estimate_normals(data[..., :3].contiguous(), knn)


class SIAdvQueryAttack:
    """SI-Adv's query-based black-box attack (shape_invariant_query_attack) for batches.  This restates the published
    algorithm and is not pinned against the reference's code, which is not recorded here (as defense.SRSDefense):
      1. normals as SIAdvAttack takes them, once, on the clean cloud; U_i = the spin-axis frame of pcd_si_step;
      2. the sensitivity map, once: G = d sum_b margin(surrogate(ori)) / d ori (margin: the C&W margin of
         SIAdvAttack._loss without the clamp); per point the tangent length s_i = |(U_i G_i)_xy| and its direction; the
         points ranked by descending s (functional.si_sensitivity);
      3. query rounds: round 0 scores the clean cloud; afterwards the trial moves the point at the cursor by -step_size,
         then +step_size, along its direction in its tangent plane, and clips the cloud to eps as the step does.  A trial
         that fools the black box ends the sample; one that lowers the margin is kept and the cursor moves on; after
         both signs fail the cursor moves on (functional.si_query_round_, include/pcdist.h for the exact rules).
    A sample ends on success or after max_query queries.  step_size = 0.05 is this library's default: the reference's
    value is not recorded here.  model is the black box and runs only under no_grad; surrogate (default: model) gives
    the gradient in one forward and one backward; neither gets a .grad.  Defences come in through the model, e.g.
    DefendedVictim with a device-sampled SRS or SOR.  The host reads the active count every check_every rounds and
    stops when it is 0; with use_graph=True one round is captured and replayed.  A sample's result depends only on its
    own inputs (given a black box whose logits for a cloud do not depend on the batch), so sharding needs no extra code."""

    def __init__(self, model, surrogate=None, eps=0.16, step_size=0.05, max_query=2000, knn=20, targeted=False,
                 check_every=50, use_graph=False):
        self.model = model.eval()
        self.surrogate = surrogate.eval() if surrogate is not None else None
        self.eps, self.step_size, self.max_query = float(eps), float(step_size), int(max_query)
        self.knn, self.targeted, self.check_every, self.use_graph = int(knn), bool(targeted), int(check_every), bool(use_graph)
        if self.max_query < 1 or self.check_every < 1:
            raise ValueError(f"max_query and check_every must be >= 1, got {max_query}, {check_every}")
        self.rounds = 0                          # query rounds run by the last attack()
        self.loop_ms = 0.0                       # device time of those rounds

    def _margin(self, logits, target):
        one_hot = torch.zeros_like(logits).scatter_(1, target.view(-1, 1), 1.)
        real = torch.sum(one_hot * logits, dim=1)
        other = torch.max((1. - one_hot) * logits - one_hot * 10000., dim=1)[0]
        return other - real if self.targeted else real - other

    def _round(self, st):
        with torch.no_grad():
            logits = self.model(st["trial"].transpose(1, 2))[0]
            if logits.dtype != torch.float32:
                logits = logits.float()
            F.si_query_round_(logits, st["target"], st["ori"], st["normal"], st["order"], st["dir"], st["cloud"],
                              st["trial"], st["state"], st["best"], self.step_size, self.eps, self.max_query,
                              self.targeted, st["active"])

    def attack(self, points, target):
        """points [B,N,3] (or [B,N,6] with normals in channels 3:6), target [B] ->
        (adv [B,N,3], pred [B] = argmax of the black box on adv (one more forward, not counted), success [B] (the
        query that ended the sample fooled the black box), queries [B] int64)"""
        dev = points.device
        if dev.type != "cuda":
            raise RuntimeError("SIAdvQueryAttack runs on CUDA only")
        if points.dim() != 3 or points.shape[2] not in (3, 6):
            raise ValueError(f"points must be [B, N, 3] or [B, N, 6], got {tuple(points.shape)}")
        data = points.detach().float()
        ori = data[..., :3].contiguous()
        normal = _unit_normals(data, self.knn)
        target = target.long().to(dev).contiguous()
        B = ori.shape[0]
        surrogate = self.model if self.surrogate is None else self.surrogate
        with torch.enable_grad():
            x = ori.clone().requires_grad_(True)
            grad, = torch.autograd.grad(self._margin(surrogate(x.transpose(1, 2))[0], target).sum(), x)
        order, dir = F.si_sensitivity(grad, normal)
        st = {"ori": ori, "normal": normal, "target": target, "order": order, "dir": dir, "cloud": ori.clone(),
              "trial": ori.clone(), "state": torch.tensor([[-1, 0, 0, 0]], dtype=torch.int32, device=dev).repeat(B, 1),
              "best": torch.zeros(B, device=dev), "active": torch.full((1,), B, dtype=torch.int32, device=dev)}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        graph = self._capture(st) if self.use_graph else None
        e0.record()
        self.rounds = 0
        while self.rounds < self.max_query:
            if graph is not None:
                graph.replay()
            else:
                self._round(st)
            self.rounds += 1
            if self.rounds % self.check_every == 0 and self.rounds < self.max_query and int(st["active"].item()) == 0:
                break
        e1.record()
        with torch.no_grad():
            pred = torch.argmax(self.model(st["cloud"].transpose(1, 2))[0], dim=1)
        torch.cuda.synchronize(dev)
        self.loop_ms = e0.elapsed_time(e1)
        return st["cloud"], pred, st["state"][:, 3] == 1, st["state"][:, 2].long()

    def _capture(self, st, warmup=3):
        """Capture one round.  The warm-up rounds run on the real state (the graph records its addresses), so the
        clouds, the decision state and the draw counters of any device-sampled defence are saved before and restored
        after: replaying k times is exactly k rounds."""
        saved = {k: st[k].clone() for k in ("cloud", "trial", "state", "best", "active")}
        samplers = _samplers(self.model)
        counters = [s.state.clone() for s in samplers]
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._round(st)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            self._round(st)
        for k, v in saved.items():
            st[k].copy_(v)
        for s, c in zip(samplers, counters):
            s.state.copy_(c)
        return g
