"""Drop-in for the graph helpers of attack/AOF/TAOF_attack.py:13-52 (same in attack/AOF/Eval_AOF.py), and the AOF attack
itself as a batched, device-resident loop.

`knn` is model/dgcnn.py's formulation (see dgcnn.knn).  `get_Laplace_from_pc` assembles the dense
graph Laplacian of the symmetrised 30-NN graph with Gaussian weights in one kernel pass over the index
tensor instead of materialising [B,N,N,3] differences, a scatter mask and its transpose; the dense
eigendecomposition stays with torch (`torch.linalg.eigh` replaces the removed `torch.symeig`; it is a
LAPACK/cuSOLVER call, not part of the point-set distance path).

AOFAttack ("attacking on frequency", Liu et al. 2022) is restated from the published method; the reference's loop is
not recorded here, so it is not pinned against it.  The choices the method leaves open are this library's:
  * the basis is computed once per attack, on the clean cloud: L = laplacian_from_pc(ori, 30), torch.linalg.eigh of L
    in float64 (fp32 eigh at N = 1024 gives vectors orthonormal only to about 1e-6, float64 to 2e-8 after rounding to
    fp32, and the projection has to be idempotent), and the eigenvectors of the low_pass smallest eigenvalues as the
    rows of V [B, low_pass, N] float32 (low_frequency_basis);
  * low(x) = V^T (V x) per sample and channel (functional.low_pass, one launch forward and one backward);
  * the optimisation is cw_loop.CWAttack's (binary search of the distance weight, Adam on the cloud, best-result tracking,
    the optional clip) with the adversarial term
        ((1 - gamma) * adv_func(model(adv)) + gamma * adv_func(model(low(adv)))).sum() / (global_batch or B)
    where the victim runs once on torch.cat([adv, low(adv)]) (it is in eval mode, so rows are independent); tracking and
    success use the adv half only;
  * gamma = 0.25 and low_pass = 100 are this library's defaults; gamma = 0 skips the
    basis and the low-frequency forward, and is then CWAttack bit for bit.
There is no install() patch for AOFAttack: the reference's class layout is not recorded here.
"""
import torch

from . import functional as F
from .cw_loop import CWAttack
from .dgcnn import knn  # noqa: F401


def laplacian_from_pc(ori_pc, k=30):
    """ori_pc [B,3,N] -> L [B,N,N] = D - A (TAOF_attack.py:36-50)."""
    pc = ori_pc.detach()
    pts = pc.transpose(2, 1)
    _, idx = F.knn(pts, pts, k, form=F.FORM_COL_ROW, norm=F.NORM_MULSUM)
    return F.graph_laplacian(pts, idx)


def get_Laplace_from_pc(ori_pc):
    """TAOF_attack.py:31-52 -> (eigenvalues [B,N] ascending, eigenvectors [B,N,N])."""
    with torch.no_grad():
        L = laplacian_from_pc(ori_pc, 30)
        e, v = torch.linalg.eigh(L)
    return e.to(ori_pc), v.to(ori_pc)


def low_frequency_basis(ori_pc, low_pass=100, k=30):
    """ori_pc [B,3,N] -> V [B, low_pass, N] float32, contiguous: the eigenvectors of the low_pass smallest eigenvalues of
    the k-NN graph Laplacian, one per row (float64 eigh, so the rows are orthonormal to float32 rounding)."""
    N = ori_pc.shape[2]
    low_pass = int(low_pass)
    if not 1 <= low_pass <= N:
        raise ValueError(f"low_pass must be in [1, N = {N}], got {low_pass}")
    with torch.no_grad():
        L = laplacian_from_pc(ori_pc, k)
        _, v = torch.linalg.eigh(L.double())
    return v[..., :low_pass].transpose(1, 2).float().contiguous()


class AOFAttack(CWAttack):
    """AOF for batches: CWAttack with the adversarial term split between the cloud and its low-frequency component (see
    the module docstring).  Takes CWAttack's arguments; dist_func is normally dist_utils.L2Dist.  attack() returns what
    CWAttack.attack returns."""

    def __init__(self, model, adv_func, dist_func, gamma=0.25, low_pass=100, attack_lr=1e-2, init_weight=10.,
                 max_weight=80., binary_step=10, num_iter=500, clip_func=None, global_batch=None, use_graph=False,
                 attack_method="untarget"):
        gamma, low_pass = float(gamma), int(low_pass)
        if not 0. <= gamma <= 1.:
            raise ValueError(f"gamma must be in [0, 1], got {gamma}")
        if low_pass < 1:
            raise ValueError(f"low_pass must be >= 1, got {low_pass}")
        super().__init__(model, adv_func, dist_func, attack_lr=attack_lr, init_weight=init_weight, max_weight=max_weight,
                         binary_step=binary_step, num_iter=num_iter, clip_func=clip_func, global_batch=global_batch,
                         use_graph=use_graph, attack_method=attack_method)
        self.gamma, self.low_pass = gamma, low_pass
        self._basis = None

    def _victim(self, adv, target):
        if self.gamma == 0.:
            return super()._victim(adv, target)
        B = adv.shape[0]
        low = F.low_pass(adv.transpose(1, 2), self._basis).transpose(1, 2)      # [B,3,N], adv's layout
        logits = self.model(torch.cat([adv, low]))[0]
        adv_logits = logits[:B]
        term = (1. - self.gamma) * self.adv_func(adv_logits, target, reduce=False) \
            + self.gamma * self.adv_func(logits[B:], target, reduce=False)
        return adv_logits, term.sum()

    def attack(self, data, target, basis=None, seed=0, first_sample=0, init_noise=None):
        """data [B, N, 3], target [B]; basis: None (computed here with low_frequency_basis) or V [B, low_pass, N] float32
        -> (o_bestdist[B], o_bestattack[B,N,3], success mask[B])."""
        if data.device.type != "cuda":
            raise RuntimeError("AOFAttack runs on CUDA only")
        B, N = data.shape[:2]
        if self.low_pass > N:
            raise ValueError(f"low_pass = {self.low_pass} exceeds the {N} points of a cloud")
        if self.gamma == 0.:
            basis = None
        elif basis is None:
            basis = low_frequency_basis(data.float().transpose(1, 2), self.low_pass)
        elif tuple(basis.shape) != (B, self.low_pass, N):
            raise ValueError(f"basis must be [{B}, {self.low_pass}, {N}], got {tuple(basis.shape)}")
        self._basis = basis
        try:
            return super().attack(data, target, seed=seed, first_sample=first_sample, init_noise=init_noise)
        finally:
            self._basis = None
