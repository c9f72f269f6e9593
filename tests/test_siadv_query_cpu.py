"""SI-Adv's query-based attack without a GPU: the decision state machine of the float32 oracle on hand-built logits, the
trial's geometry, the torch host loop (the reference's shape) against the oracle loop, the argument errors of
pcd_si_sensitivity and pcd_si_query_round that come before any CUDA call, and the attack's refusal to run on the CPU."""
import ctypes
import importlib
import os
import sys

import numpy as np
import pytest
import torch

from oracle import siadv_query_oracle as Q

pcd = importlib.import_module("3dpointcloudattack_b200")
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import tiny_victim  # noqa: E402

STEP, EPS = 0.05, 0.16


def unit(v):
    return (v / np.linalg.norm(v, axis=-1, keepdims=True)).astype(np.float32)


class Loop:
    """one sample, untargeted, driven round by round with hand-built logits rows: with y = 0 the row [m, 0] has margin m
    and no success while m > 0"""

    def __init__(self, N=3, max_query=100, seed=0):
        rng = np.random.default_rng(seed)
        self.ori = rng.uniform(-1, 1, (1, N, 3)).astype(np.float32)
        self.normal = unit(rng.standard_normal((1, N, 3)))
        _, self.dir, self.order = Q.sensitivity(rng.standard_normal((1, N, 3)).astype(np.float32), self.normal)
        self.cloud, self.trial = self.ori.copy(), self.ori.copy()
        self.state, self.best = Q.initial_state(1), np.zeros(1, np.float32)
        self.active, self.max_query = 1, max_query

    def round(self, row, y=0):
        self.scored = self.trial.copy()
        self.cloud, self.trial, self.state, self.best, self.active = Q.query_round(
            np.array([row], np.float32), [y], self.ori, self.normal, self.order, self.dir, self.cloud, self.trial,
            self.state, self.best, STEP, EPS, self.max_query, active=self.active)
        return tuple(int(v) for v in self.state[0])

    def expected_trial(self, cursor, sigma):
        i = int(self.order[0][cursor % self.ori.shape[1]])
        return Q.trial(self.cloud[0], self.ori[0], self.normal[0], self.dir[0], i, sigma, STEP, EPS)


def test_accept_on_minus_and_reject_minus_then_accept_plus():
    lp = Loop()
    assert lp.round([5, 0]) == (-1, 0, 1, Q.ACTIVE) and lp.best[0] == 5      # round 0 scores the clean cloud
    assert np.array_equal(lp.cloud, lp.ori) and np.array_equal(lp.trial[0], lp.expected_trial(0, -1))
    assert lp.round([4, 0]) == (-1, 1, 2, Q.ACTIVE) and lp.best[0] == 4      # -step lowers the margin: taken
    assert np.array_equal(lp.cloud, lp.scored) and np.array_equal(lp.trial[0], lp.expected_trial(1, -1))
    kept = lp.cloud.copy()
    assert lp.round([4, 0]) == (1, 1, 3, Q.ACTIVE)                            # not strictly lower: same point, +step
    assert np.array_equal(lp.cloud, kept) and np.array_equal(lp.trial[0], lp.expected_trial(1, 1))
    assert lp.round([3.5, 0]) == (-1, 2, 4, Q.ACTIVE) and lp.best[0] == 3.5  # +step taken
    assert np.array_equal(lp.cloud, lp.scored)


def test_reject_both_moves_on_and_wraps_past_n():
    lp = Loop(N=3)
    lp.round([5, 0])
    seen = []
    for _ in range(8):                                                         # 4 points' worth of (-, +) on N = 3
        seen.append(lp.round([6, 0])[:2])
    assert seen == [(1, 0), (-1, 1), (1, 1), (-1, 2), (1, 2), (-1, 3), (1, 3), (-1, 4)]
    assert np.array_equal(lp.cloud, lp.ori) and lp.best[0] == 5
    assert np.array_equal(lp.trial[0], lp.expected_trial(4, -1))             # cursor 4 is point order[1]


def test_success_is_taken_even_without_a_lower_margin_and_then_frozen():
    lp = Loop()
    lp.round([1, 0])
    lp.round([2, 0])
    assert lp.round([0, 1]) == (1, 0, 3, Q.SUCCESS) and lp.active == 0       # margin -1 is lower here, ...
    assert np.array_equal(lp.cloud, lp.scored) and np.array_equal(lp.trial, lp.cloud)
    frozen = (lp.cloud.copy(), lp.trial.copy(), lp.state.copy(), lp.best.copy())
    for row in ([-5, 0], [0, 9], [np.nan, 0]):                               # ... and nothing moves afterwards
        lp.round(row)
        assert all(np.array_equal(a, b) for a, b in zip(frozen, (lp.cloud, lp.trial, lp.state, lp.best)))
    assert lp.active == 0
    # a success whose margin is not below best: only a tie allows it (argmax takes the first maximal index)
    lp = Loop()
    assert lp.round([1, 2, 2], y=1)[3] == Q.ACTIVE and lp.best[0] == 0       # argmax 1 == y, margin 0
    lp.round([1, 3, 2], y=1)
    assert Q.score([2, 2, 0], 1, False) == (True, np.float32(0), True)
    assert lp.round([2, 2, 0], y=1)[3] == Q.SUCCESS and np.array_equal(lp.cloud, lp.scored)
    assert not np.array_equal(lp.cloud, lp.ori)


def test_targeted_success_and_margin():
    assert Q.score([1, 3, 2], 1, True) == (True, np.float32(-1), True)
    assert Q.score([1, 3, 2], 2, True) == (True, np.float32(1), False)
    assert Q.score([1, 3, 2], 1, False) == (True, np.float32(1), False)
    assert Q.score([-20000, -30000], 0, False)[1] == np.float32(-10000)      # the one-hot row caps other at -10000
    assert Q.score([2, 2], 1, False)[2]                                        # the first arg-max: 0 != 1


@pytest.mark.parametrize("row", [[np.nan, 0], [0, np.nan], [np.inf, 0], [-np.inf, 0, 1]])
def test_nan_rows_and_non_finite_margins_are_rejected(row):
    valid, _, success = Q.score(row, 0, False)
    assert not valid and not success
    lp = Loop()
    lp.round([5, 0])
    assert lp.round(row)[:2] == (1, 0) and np.array_equal(lp.cloud, lp.ori) and lp.best[0] == 5


def test_already_misclassified_sample_takes_one_query_and_comes_back_unchanged():
    lp = Loop()
    assert lp.round([0, 1]) == (-1, 0, 1, Q.SUCCESS)
    assert np.array_equal(lp.cloud, lp.ori) and np.array_equal(lp.trial, lp.ori) and lp.active == 0


@pytest.mark.parametrize("max_query", [1, 2, 7])
def test_failure_ends_at_exactly_max_query(max_query):
    lp = Loop(max_query=max_query)
    for q in range(1, max_query + 1):
        st = lp.round([5 - 0.5 * q, 0])                                        # improves every round, never succeeds
        assert st[2] == q and st[3] == (Q.FAILED if q == max_query else Q.ACTIVE)
    assert lp.active == 0 and np.array_equal(lp.trial, lp.cloud)
    assert lp.round([-9, 0])[2:] == (max_query, Q.FAILED)


def test_trial_moves_one_point_in_its_tangent_plane_then_clips():
    rng = np.random.default_rng(4)
    N = 50
    ori = rng.uniform(-1, 1, (N, 3)).astype(np.float32)
    n = unit(rng.standard_normal((N, 3)) * [1, 1, 0.3])
    s, d, order = Q.sensitivity(rng.standard_normal((1, N, 3)).astype(np.float32), n[None])
    assert np.allclose(np.linalg.norm(d[0], axis=-1), 1, atol=1e-6) and (np.diff(s[0][order[0]]) <= 0).all()
    i = int(order[0][0])
    t = Q.trial(ori, ori, n, d[0], i, -1, STEP, 10.0).astype(np.float64)      # eps large: the clip leaves it alone
    move = t - ori
    assert np.abs(np.delete(move, i, 0)).max() < 1e-6                          # the others only by ori + (p - ori) * 1
    assert abs(np.linalg.norm(move[i]) - STEP) < 1e-6 and abs(move[i] @ n[i]) < 1e-6
    u = Q.spin_axis(n[i].astype(np.float64), np.float64)
    assert np.allclose((u @ move[i])[:2], -STEP * d[0][i], atol=1e-6)        # along -dir in the frame
    clipped = Q.trial(ori, ori, n, d[0], i, 1, 0.5, 0.01).astype(np.float64)
    assert np.sqrt(((clipped - ori) ** 2).sum(0)).max() <= 0.01 * (1 + 1e-6)


def test_sensitivity_nan_ranks_last_and_moves_nothing():
    g = np.ones((1, 4, 3), np.float32)
    g[0, 1, 0] = np.nan
    s, d, order = Q.sensitivity(g, unit(np.random.default_rng(0).standard_normal((1, 4, 3))))
    assert s[0, 1] == -1 and (d[0, 1] == 0).all() and order[0, -1] == 1


def test_torch_host_loop_equals_the_oracle_loop():
    """the reference's shape (torch ops, one Python decision per query) is the contract's arithmetic: on the CPU, with
    the tiny victim as black box, it gives the oracle loop's bits"""
    model = tiny_victim.make(2)
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    x = synth.face_clouds(2, 128, seed=5)
    normal = unit(np.random.default_rng(6).standard_normal((2, 128, 3)))
    with torch.no_grad():
        label = model(x.transpose(1, 2))[0].argmax(1)

    def black_box(c):
        with torch.no_grad():
            return model(torch.from_numpy(c).transpose(1, 2))[0].numpy()

    for b in range(2):
        adv, pred, success, queries = Q.host_loop(model, x[b], torch.from_numpy(normal[b]), int(label[b]), eps=0.5,
                                                  step_size=0.2, max_query=60)
        xb = x[b:b + 1].clone().requires_grad_(True)
        grad, = torch.autograd.grad(Q.margin_loss(model(xb.transpose(1, 2))[0], label[b:b + 1], False).sum(), xb)
        want, wq, ws, _ = Q.run(black_box, x[b:b + 1].numpy(), normal[b:b + 1], grad.numpy(), [int(label[b])], 0.2, 0.5, 60)
        assert np.array_equal(adv.numpy(), want[0]) and queries == wq[0] and success == ws[0], b
        assert not np.array_equal(want[0], x[b].numpy())                      # the attack moved something
        assert success == (pred != int(label[b]))


def test_query_abi_argument_errors():
    lib = pcd._lib.load()
    fake = ctypes.c_void_p(256)             # never dereferenced: every call below fails its argument check
    cloud = [48, 3, 1]

    def sens(grad=fake, normal=fake, s=fake, d=fake, B=2, N=16):
        return lib.pcd_si_sensitivity(grad, *cloud, normal, *cloud, B, N, s, d, None)

    assert sens(grad=None) == 1 and sens(normal=None) == 1 and sens(s=None) == 1 and sens(d=None) == 1
    assert sens(N=0) == 1 and sens(B=-1) == 1
    assert b"pcd_si_sensitivity" in lib.pcd_last_error()
    assert sens(B=0) == 0 and sens(B=0, grad=None) == 0

    def rnd(logits=fake, target=fake, ori=fake, normal=fake, order=fake, dir=fake, cl=fake, tr=ctypes.c_void_p(512),
            state=fake, best=fake, B=2, N=16, C=10, step=0.05, eps=0.16, max_query=100, targeted=0, active=None):
        return lib.pcd_si_query_round(logits, 10, 1, C, target, ori, *cloud, normal, *cloud, order, dir, cl, *cloud, tr,
                                      *cloud, state, best, B, N, step, eps, max_query, targeted, active, None)

    for name in ("logits", "target", "ori", "normal", "order", "dir", "cl", "tr", "state", "best"):
        assert rnd(**{name: None}) == 1, name
    assert rnd(tr=fake) == 1                                                   # cloud and trial are the same memory
    assert rnd(N=0) == 1 and rnd(B=-1) == 1 and rnd(C=1) == 1
    assert rnd(step=float("nan")) == 1 and rnd(step=float("inf")) == 1
    assert rnd(eps=-1e-3) == 1 and rnd(eps=float("nan")) == 1
    assert rnd(max_query=0) == 1 and rnd(targeted=2) == 1 and rnd(targeted=-1) == 1
    assert b"pcd_si_query_round" in lib.pcd_last_error()
    assert rnd(N=16385) == 4                                                   # PCD_ERR_UNSUPPORTED
    assert b"16384" in lib.pcd_last_error()
    assert rnd(B=0) == 0 and rnd(B=0, logits=None, cl=None) == 0              # an empty batch is a no-op


def test_attack_runs_on_cuda_only():
    atk = pcd.siadv.SIAdvQueryAttack(tiny_victim.make(0))
    with pytest.raises(RuntimeError, match="CUDA only"):
        atk.attack(torch.zeros(1, 16, 3), torch.zeros(1, dtype=torch.long))
    with pytest.raises(ValueError):
        pcd.siadv.SIAdvQueryAttack(tiny_victim.make(0), max_query=0)
