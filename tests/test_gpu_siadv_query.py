"""GPU: SI-Adv's query-based attack.  The round kernel (functional.si_query_round_, pcd_si_query_round) equals the float32
oracle bit for bit on cloud, trial, state, best and the active count, from random states in every phase, whatever the
batch, the class count, the layout or the goal; the sensitivity kernel equals the oracle and its order the stable sort.
SIAdvQueryAttack gives the host loop's bits at B = 1, each sample's result alone and inside a batch, the same bits as a
graph and eager (through an SRS defence too), keeps its invariants, never touches the black box's .grad and makes one
library launch per round."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from oracle import siadv_query_oracle as Q

pytestmark = pytest.mark.gpu

pcd = importlib.import_module("3dpointcloudattack_b200")
synth = importlib.import_module("3dpointcloudattack_b200.synth")
F, D = pcd.functional, pcd.defense
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tiny_victim  # noqa: E402

STEP, EPS = 0.05, 0.16


def unit(v):
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)


def same_bits(a, b):
    """bit-equal, except that any NaN equals any NaN (payloads differ between the GPU and numpy)"""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype != np.float32:
        return a.shape == b.shape and np.array_equal(a, b)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and (na == nb).all() and (a[~na].view(np.uint32) == b[~nb].view(np.uint32)).all()


def layout(x, channel_first):
    t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    return t.transpose(1, 2).contiguous().transpose(1, 2) if channel_first else t.contiguous()


def random_round(B, N, C, targeted, seed, max_query=50):
    """inputs of one round with every sample in a phase of its own: round 0, after a rejected -step, a cursor past N,
    the last query, NaN logits, already ended (success / failure)"""
    rng = np.random.default_rng(seed)
    ori = rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    normal = unit(rng.standard_normal((B, N, 3)))
    normal[:, ::5] = [0, 0, 1]                                                 # the boundary frame
    grad = rng.standard_normal((B, N, 3)).astype(np.float32)
    grad[:, ::3] = 0                                                           # ties in the ranking
    _, dir, order = Q.sensitivity(grad, normal)
    cloud = (ori + 0.02 * rng.standard_normal((B, N, 3))).astype(np.float32)
    trial = (cloud + 0.02 * rng.standard_normal((B, N, 3))).astype(np.float32)
    state = np.zeros((B, 4), np.int32)
    state[:, 0] = rng.choice([-1, 1], B)
    state[:, 1] = rng.integers(0, 3 * N + 2, B)
    state[:, 2] = rng.integers(1, max_query - 1, B)
    logits = (3 * rng.standard_normal((B, C))).astype(np.float32)
    target = rng.integers(0, C, B).astype(np.int64)
    phase = rng.integers(0, 7, B)
    phase[:min(B, 7)] = np.arange(min(B, 7))
    for b in range(B):
        keep = rng.random() < 0.6                                              # the label stays on top: no success
        if keep != targeted:
            logits[b, target[b]] = logits[b].max() + rng.uniform(0.1, 2)
        if phase[b] == 0:
            state[b] = [-1, 0, 0, 0]
            cloud[b] = trial[b] = ori[b]
        elif phase[b] == 2:
            state[b, 1] = rng.integers(N, 2 * N + 1)
        elif phase[b] == 3:
            state[b, 2] = max_query - 1
        elif phase[b] == 4:
            logits[b, rng.integers(0, C)] = np.nan
        elif phase[b] in (5, 6):
            state[b, 3] = phase[b] - 4
            trial[b] = cloud[b]
    margin = np.array([Q.score(logits[b], int(target[b]), targeted)[1] for b in range(B)], np.float32)
    best = np.where(rng.random(B) < 0.5, margin + np.float32(0.25), margin - np.float32(0.25)).astype(np.float32)
    tie = rng.random(B) < 0.1                                                 # margin == best: no improvement
    best[tie] = margin[tie]
    return dict(logits=logits, target=target, ori=ori, normal=normal, order=order, dir=dir, cloud=cloud, trial=trial,
                state=state, best=best, grad=grad)


@pytest.mark.parametrize("C", [2, 40, 106])
@pytest.mark.parametrize("N", [1, 7, 1024, 4097, 16384])
@pytest.mark.parametrize("B", [1, 3, 64])
def test_round_equals_the_float32_oracle_bit_for_bit(B, N, C):
    for targeted in (False, True):
        r = random_round(B, N, C, targeted, seed=B * 1000 + N + C + targeted)
        n_active = int((r["state"][:, 3] == 0).sum())
        want = Q.query_round(r["logits"], r["target"], r["ori"], r["normal"], r["order"], r["dir"], r["cloud"],
                             r["trial"], r["state"], r["best"], STEP, EPS, 50, targeted, active=n_active)
        for channel_first in (False, True):
            cloud, trial = layout(r["cloud"], channel_first), layout(r["trial"], channel_first)
            state, best = torch.from_numpy(r["state"]).cuda(), torch.from_numpy(r["best"]).cuda()
            active = torch.tensor([n_active], dtype=torch.int32, device="cuda")
            logits = torch.from_numpy(r["logits"]).cuda()
            if channel_first:
                logits = logits.t().contiguous().t()                           # column-major logits
            F.si_query_round_(logits, torch.from_numpy(r["target"]).cuda(), layout(r["ori"], channel_first),
                              layout(r["normal"], channel_first), torch.from_numpy(r["order"]).cuda(),
                              torch.from_numpy(np.ascontiguousarray(r["dir"])).cuda(), cloud, trial, state, best,
                              STEP, EPS, 50, targeted, active)
            got = (cloud.cpu().numpy(), trial.cpu().numpy(), state.cpu().numpy(), best.cpu().numpy())
            for name, g, w in zip(("cloud", "trial", "state", "best"), got, want[:4]):
                assert same_bits(g, w), (name, targeted, channel_first)
            assert int(active.item()) == want[4]


@pytest.mark.parametrize("N", [1, 7, 1024, 16384])
@pytest.mark.parametrize("channel_first", [False, True])
def test_sensitivity_equals_the_oracle_and_the_stable_sort(N, channel_first):
    r = random_round(3, N, 2, False, seed=N)
    grad = r["grad"].copy()
    grad[1, ::7, 1] = np.nan
    s_want, d_want, o_want = Q.sensitivity(grad, r["normal"])
    g, n = layout(grad, channel_first), layout(r["normal"], channel_first)
    order, dir = F.si_sensitivity(g, n)
    assert same_bits(dir.cpu().numpy(), d_want) and np.array_equal(order.cpu().numpy(), o_want)
    assert order.dtype == torch.int32
    s = torch.empty(3, N, device="cuda")
    d2 = torch.empty(3, N, 2, device="cuda")
    lib = pcd._lib.load()
    pcd._lib.check(lib.pcd_si_sensitivity(*F._cloud_args(g), *F._cloud_args(n), 3, N, s.data_ptr(), d2.data_ptr(),
                                          F._stream()), "pcd_si_sensitivity")
    assert same_bits(s.cpu().numpy(), s_want)
    assert torch.equal(torch.sort(s, dim=1, descending=True, stable=True)[1].int(), order)


# ---------------------------------------------------------------------------------------------------------- the loop
class PerSample(torch.nn.Module):
    """the black box run one cloud at a time: its logits for a cloud then cannot depend on the batch around it"""

    def __init__(self, model):
        super().__init__()
        self.model = model

    def forward(self, x):
        return torch.cat([self.model(x[b:b + 1])[0] for b in range(x.shape[0])]), None, None


def victim_and_data(B, N=1024, seed=0):
    model = tiny_victim.make(seed).cuda()
    x = synth.face_clouds(B, N, seed=seed + 100).cuda()
    with torch.no_grad():
        label = model(x.transpose(1, 2))[0].argmax(1)
    return model, x, label


def with_normals(x, seed=1):
    n = np.random.default_rng(seed).standard_normal(tuple(x.shape)).astype(np.float32)
    return torch.cat([x, torch.from_numpy(n).cuda()], -1)


def test_equals_the_host_loop_at_b1():
    model, x, label = victim_and_data(3, N=512)
    data = with_normals(x)
    normal = pcd.siadv._unit_normals(data, 20)
    moved = 0
    for b in range(3):
        atk = pcd.siadv.SIAdvQueryAttack(model, eps=0.5, step_size=0.1, max_query=150, check_every=7)
        adv, pred, success, queries = atk.attack(data[b:b + 1], label[b:b + 1])
        h_adv, h_pred, h_success, h_queries = Q.host_loop(model, x[b], normal[b], int(label[b]), eps=0.5, step_size=0.1,
                                                          max_query=150)
        assert torch.equal(adv[0], h_adv) and int(queries[0]) == h_queries and bool(success[0]) == h_success, b
        assert int(pred[0]) == h_pred
        moved += int(not torch.equal(adv[0], x[b]))
    assert moved >= 2


def test_sample_alone_equals_sample_in_a_batch_of_32():
    model, x, label = victim_and_data(32, N=256)
    box = PerSample(model)
    kw = dict(eps=0.5, step_size=0.1, max_query=60, check_every=10)
    adv, pred, success, queries = pcd.siadv.SIAdvQueryAttack(box, **kw).attack(x, label)
    for b in (0, 5, 31):
        a1, p1, s1, q1 = pcd.siadv.SIAdvQueryAttack(box, **kw).attack(x[b:b + 1], label[b:b + 1])
        assert torch.equal(a1[0], adv[b]) and p1[0] == pred[b] and s1[0] == success[b] and q1[0] == queries[b], b


def test_invariants_no_grad_and_one_launch_per_round():
    model, x, label = victim_and_data(8)
    for eps, targeted in ((0.16, False), (2.0, False), (2.0, True)):
        tgt = (label + 1) % 7 if targeted else label
        n0 = F.launches()
        atk = pcd.siadv.SIAdvQueryAttack(model, eps=eps, step_size=0.2, max_query=300, targeted=targeted, check_every=25)
        adv, pred, success, queries = atk.attack(x, tgt)
        assert F.launches() - n0 == 3 + 1 + atk.rounds                       # normals, sensitivity, one per round
        assert atk.rounds == 300 or atk.rounds % 25 == 0
        assert adv.shape == x.shape and torch.isfinite(adv).all()
        assert ((adv - x).norm(dim=1) <= eps * (1 + 1e-6)).all()
        assert (queries >= 1).all() and (queries <= 300).all() and queries.dtype == torch.int64
        assert torch.equal(success, pred == tgt if targeted else pred != tgt)
        assert (queries[~success] == 300).all()
    assert all(p.grad is None for p in model.parameters())
    n0 = F.launches()
    atk = pcd.siadv.SIAdvQueryAttack(model, max_query=20)
    atk.attack(with_normals(x), label)
    assert F.launches() - n0 == 1 + atk.rounds == 21                           # given normals: no estimate


@pytest.mark.parametrize("defence", [None, "srs"])
def test_graph_equals_eager(defence):
    model, x, label = victim_and_data(4)
    runs = []
    for use_graph in (False, True):
        box, sampler = model, None
        if defence:
            sampler = F.PointSampler(1234, device="cuda")
            box = D.DefendedVictim(model, D.SRSDefense(200, sampler=sampler))
        atk = pcd.siadv.SIAdvQueryAttack(box, surrogate=model, eps=1.0, step_size=0.2, max_query=80, check_every=20,
                                         use_graph=use_graph)
        out = atk.attack(x, label)
        if sampler is not None:
            assert int(sampler.counter.item()) == atk.rounds + 1              # one draw per round and one for pred
        runs.append((out, atk.rounds))
    (a, ra), (b, rb) = runs
    assert ra == rb and all(torch.equal(u, v) for u, v in zip(a, b))
