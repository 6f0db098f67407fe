"""CPU: the shard contract of the data-parallel learner (fl_policy_ppo_counts, fl_policy_ppo_grad_shard_f32 / _bf16,
include/flatland_policy_b200.h) restated in float64 over tests/policy_grad_oracle.py, and the argument checks of the three
entry points, which return codes before any CUDA call.

A minibatch split into shards, each shard's loss divided by the counts of the whole minibatch, gives shard gradients whose
sum is the gradient of the whole minibatch; the mean of gradients normalised by each shard's own counts does not."""
import ctypes as C

import numpy as np
import pytest
import torch

import policy_grad_oracle as pgo
from test_cabi import lib  # noqa: F401  (fixture: builds and loads the libraries)
from test_policy_grad import golden_obs
import flatland_marl_b200.policy_weights as pw

CLIP, VF, ENT = 0.2, 0.5, 0.01
OBS = ("agent_attr", "forest", "adjacency", "node_order", "edge_order", "valid_actions")


def minibatch():
    """Six Test_00 rows of 7 agents.  Row 0 is a reset row (acted = 0); row 1 has agents with no valid action; row 2 has no
    agent with a valid action.  Shards [0:1] (reset rows only), [1:3] (the agents with no valid action), [3:6]."""
    steps = (3, 35, 67, 99, 131, 164)
    o = {k: np.stack([golden_obs("t00_l0_random", s)[k] for s in steps]) for k in OBS}
    o["valid_actions"] = o["valid_actions"].copy()
    o["valid_actions"][1, :3] = 0
    o["valid_actions"][2] = 0
    o["valid_actions"][4, :, 2] = 1
    E, N = o["agent_attr"].shape[:2]
    rng = np.random.RandomState(5)
    actions = np.argmax(o["valid_actions"] * rng.rand(E, N, 5), -1).astype(np.uint8)
    w = pw.init_weights(7)
    with torch.no_grad():
        logits, _ = pgo.forward(pgo.params(w, False), o["agent_attr"], o["forest"], o["adjacency"], o["node_order"],
                                o["edge_order"])
        lp, _, _ = pgo.log_probs(logits, o["valid_actions"], actions)
    old = lp.numpy() - np.log(np.array([1.0, 1.5, 0.6, 1.1]))[rng.randint(0, 4, (E, N))]
    mb = dict(actions=actions, log_probs=old, advantages=rng.randn(E) * 2, returns=rng.randn(E) * 3,
              acted=np.array([0, 1, 1, 1, 0, 1], np.uint8))
    return w, o, mb, [(0, 1), (1, 3), (3, 6)]


def rows(d, lo, hi):
    return {k: v[lo:hi] for k, v in d.items()}


def counts(o, mb):
    """[|S|, acted rows]: fl_policy_ppo_counts."""
    acted = np.asarray(mb["acted"]) != 0
    return int(((np.asarray(o["valid_actions"]) != 0).any(-1) & acted[:, None]).sum()), int(acted.sum())


def shard_loss(logits, value, o, mb, nS_g, nR_g):
    """The header's L_shard and the 8 shard statistics: sums over this shard's S and acted rows divided by the minibatch's
    counts nS_g, nR_g; stats 5 and 6 are this shard's counts."""
    lp, logp, valid = pgo.log_probs(logits, o["valid_actions"], mb["actions"])
    acted = torch.as_tensor(np.asarray(mb["acted"]) != 0)
    S = valid.any(-1) & acted[:, None]
    old = torch.as_tensor(np.asarray(mb["log_probs"], np.float64))
    A = torch.as_tensor(np.asarray(mb["advantages"], np.float64))[:, None]
    R = torch.as_tensor(np.asarray(mb["returns"], np.float64))
    r = torch.exp(lp - old)
    s1, s2 = r * A, torch.clamp(r, 1 - CLIP, 1 + CLIP) * A
    pol = -torch.where(s1 <= s2, s1, s2)
    p = torch.where(valid, logp.exp(), torch.zeros_like(logp))
    H = -torch.where(valid, p * logp, torch.zeros_like(logp)).sum(-1)
    zero = torch.zeros((), dtype=torch.float64)

    def sum_S(t, den):
        return torch.where(S, t, torch.zeros_like(t)).sum() / den if den else zero
    L_pol, L_ent = sum_S(pol, nS_g), sum_S(H, nS_g)
    L_val = torch.where(acted, (value - R) ** 2, torch.zeros_like(value)).sum() / nR_g if nR_g else zero
    L = L_pol - ENT * L_ent + VF * L_val
    stats = [L_pol, L_val, L_ent, sum_S(old - lp, nS_g), sum_S(((r - 1).abs() > CLIP).double(), nS_g), int(S.sum()),
             int(acted.sum()), L]
    return L, np.array([float(s.detach()) if torch.is_tensor(s) else float(s) for s in stats])


def shard_grads(w, o, mb, nS_g, nR_g):
    p = pgo.params(w)
    logits, value = pgo.forward(p, o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"])
    L, stats = shard_loss(logits, value, o, mb, nS_g, nR_g)
    if L.requires_grad:                                             # both denominators 0: the loss is the constant 0
        L.backward()
    return stats, {k: (v.grad.numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in p.items()}


@pytest.fixture(scope="module")
def case():
    w, o, mb, split = minibatch()
    _, full_stats, _, _, full = pgo.loss_and_grads(w, o, mb, CLIP, VF, ENT)
    return w, o, mb, split, full_stats, full


def test_split_covers_the_degenerate_shards(case):
    w, o, mb, split, _, _ = case
    c = [counts(rows(o, lo, hi), rows(mb, lo, hi)) for lo, hi in split]
    assert c[0] == (0, 0)                                           # a shard of reset rows only
    va = o["valid_actions"][1:3].any(-1)
    assert (~va).any() and va.any()                                  # a shard with agents that have no valid action
    assert tuple(np.sum(c, 0)) == counts(o, mb)
    nS, nR = counts(o, mb)
    assert nS > 0 and nR == 4


def test_shard_gradients_with_global_counts_sum_to_the_minibatch_gradient(case):
    w, o, mb, split, full_stats, full = case
    nS, nR = counts(o, mb)
    total = {k: np.zeros_like(v) for k, v in full.items()}
    stats = np.zeros(8)
    for lo, hi in split:
        st, g = shard_grads(w, rows(o, lo, hi), rows(mb, lo, hi), nS, nR)
        stats += st
        for k in total:
            total[k] += g[k]
    worst = 0.0
    for k, ref in full.items():
        scale = np.abs(ref).max()
        assert scale > 0, k
        err = np.abs(total[k] - ref).max() / scale
        assert err <= 1e-12, "%s: %.3e" % (k, err)
        worst = max(worst, err)
    np.testing.assert_allclose(stats, full_stats, rtol=1e-12, atol=1e-14)
    assert stats[5] == nS and stats[6] == nR
    print("worst relative difference of the summed shard gradients: %.2e" % worst)


def test_the_mean_of_locally_normalised_gradients_is_not_the_minibatch_gradient(case):
    """What a caller could do without the global counts: each shard normalised by its own |S| and acted rows, the gradients
    averaged over shards (or summed: no single factor repairs it, the two terms have different denominators)."""
    w, o, mb, split, _, full = case
    local = []
    for lo, hi in split:
        so, sm = rows(o, lo, hi), rows(mb, lo, hi)
        local.append(shard_grads(w, so, sm, *counts(so, sm))[1])
    worst_mean = worst_sum = 0.0
    for k, ref in full.items():
        mean = sum(g[k] for g in local) / len(local)
        sm = sum(g[k] for g in local)
        scale = np.abs(ref).max()
        worst_mean = max(worst_mean, np.abs(mean - ref).max() / scale)
        worst_sum = max(worst_sum, np.abs(sm - ref).max() / scale)
    assert worst_mean > 1e-2 and worst_sum > 1e-2, (worst_mean, worst_sum)


def test_shard_entry_points_bad_arguments(lib):  # noqa: F811
    from flatland_marl_b200 import policy
    L = policy.lib()
    buf = C.create_string_buffer(64)
    p = C.cast(buf, C.c_void_p)
    n_t = 46
    good = (C.c_void_p * n_t)(*([p.value] * n_t))
    ws_need = int(L.fl_policy_workspace_bytes_grad_f32(6))

    for fn in (L.fl_policy_ppo_grad_shard_f32, L.fl_policy_ppo_grad_shard_bf16):
        def call(E=2, N=3, ptrs=None, wts=good, grads=good, ws_bytes=ws_need, clip=0.2, params=True):
            ptrs = ptrs or [p] * 15
            prm = policy.FlPpoParams(clip, 0.5, 0.01)
            return fn(wts, ptrs[0], ws_bytes, E, N, *ptrs[1:12], C.byref(prm) if params else None, grads,
                      ptrs[12], ptrs[13], ptrs[14], None)
        for k in range(15):                                # workspace, 10 inputs, global counts, logits, value, stats
            ptrs = [p] * 15
            ptrs[k] = None
            assert call(ptrs=ptrs) == -1, k
        assert call(wts=None) == -1 and call(grads=None) == -1 and call(params=False) == -1
        for k in (0, 17, 45):
            bad = (C.c_void_p * n_t)(*([p.value] * n_t))
            bad[k] = None
            assert call(wts=bad) == -1 and call(grads=bad) == -1
        assert call(E=0) == -1 and call(N=0) == -1 and call(E=-1) == -1 and call(N=-4) == -1
        assert call(ws_bytes=ws_need - 1) == -1 and call(E=4, ws_bytes=ws_need) == -1
        assert call(clip=0.0) == -1 and call(clip=-0.1) == -1 and call(clip=float("nan")) == -1
        assert call(E=2 ** 40, N=2 ** 30) == -1

    def counts_call(E=2, N=3, valid=p, acted=p, out=p):
        return L.fl_policy_ppo_counts(E, N, valid, acted, out, None)
    assert counts_call(valid=None) == -1 and counts_call(acted=None) == -1 and counts_call(out=None) == -1
    assert counts_call(E=0) == -1 and counts_call(N=0) == -1 and counts_call(E=-1) == -1 and counts_call(N=-4) == -1
    assert counts_call(E=2 ** 40, N=2 ** 30) == -1 and counts_call(E=1, N=2 ** 31) == -1
