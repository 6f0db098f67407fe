"""CPU: the float64 yardstick of the PPO gradients (tests/policy_grad_oracle.py) against the numpy oracle of the reference
network and against finite differences, and the argument checks of fl_policy_ppo_grad_f32 (include/flatland_policy_b200.h),
which return codes before any CUDA call."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import policy_grad_oracle as pgo
from oracle import policy_oracle as po
from test_cabi import lib  # noqa: F401  (fixture: builds and loads the libraries)
import flatland_marl_b200.policy_weights as pw

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def golden_obs(fixture, step):
    with np.load(os.path.join(GOLD, fixture + ".npz")) as z:
        p = "obs%d_" % step
        return dict(agent_attr=z[p + "attr"], forest=z[p + "forest"], adjacency=z[p + "adjacency"], node_order=z[p + "node_order"],
                    edge_order=z[p + "edge_order"], valid_actions=z[p + "valid_actions"])


def test_torch_forward_equals_numpy_oracle_on_golden_cases():
    with np.load(os.path.join(GOLD, "policy_golden.npz")) as z:
        gold = {k: z[k] for k in z.files}
    w = pw.init_weights(int(gold["weight_seed"]))
    p = pgo.params(w, requires_grad=False)
    worst = 0.0
    for fixture, step in sorted(set(zip(gold["case_fixture"].tolist(), gold["case_step"].tolist()))):
        o = golden_obs(str(fixture), int(step))
        want, wval = po.forward(w, o["agent_attr"][None], po.clean_forest(o["forest"])[None], o["adjacency"][None],
                                o["node_order"][None], o["edge_order"][None])
        with torch.no_grad():
            got, val = pgo.forward(p, o["agent_attr"][None], o["forest"][None], o["adjacency"][None], o["node_order"][None],
                                   o["edge_order"][None])
        np.testing.assert_allclose(got.numpy(), want, rtol=0, atol=1e-5, err_msg="%s step %d" % (fixture, step))
        np.testing.assert_allclose(val.numpy(), wval, rtol=0, atol=1e-5)
        worst = max(worst, float(np.abs(got.numpy() - want).max()))
    assert worst < 1e-5


def tiny_case():
    """One environment of 4 agents (Test_00 observation): agent 0 has r = 1.5 (clipped side: no gradient for A > 0),
    agent 1 r = 0.5 (unclipped side), agent 2 r = 1 (tie: r A = clip(r) A), agent 3 no valid action."""
    o = {k: v[:4][None] for k, v in golden_obs("t00_l0_random", 3).items()}
    o["valid_actions"] = o["valid_actions"].copy()
    o["valid_actions"][0, :3] |= np.array([[1, 1, 0, 0, 1], [0, 1, 1, 1, 0], [1, 0, 1, 0, 1]], np.uint8)
    o["valid_actions"][0, 3] = 0
    actions = np.array([[1, 2, 4, 0]], np.uint8)
    w = pw.init_weights(3)
    with torch.no_grad():
        logits, _ = pgo.forward(pgo.params(w, False), o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"])
        lp, _, _ = pgo.log_probs(logits, o["valid_actions"], actions)
    old = lp.numpy() - np.log(np.array([[1.5, 0.5, 1.0, 1.0]]))
    mb = dict(actions=actions, log_probs=old, advantages=np.array([0.7]), returns=np.array([0.3]), acted=np.array([1], np.uint8))
    return w, o, mb


def test_gradcheck_tiny_case():
    w, o, mb = tiny_case()
    names = ["actor_net.4.bias", "critic_net.4.bias", "actor_net.2.bias", "tree_lstm.W_f.bias", "tree_lstm.W_c.bias",
             "transformer.0.attention.in_proj_bias"]
    base = pgo.params(w, requires_grad=False)

    def loss(*ts):
        p = dict(base)
        p.update(zip(names, ts))
        logits, value = pgo.forward(p, o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"])
        L, stats = pgo.ppo_loss(logits, value, o["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"],
                                mb["returns"], mb["acted"], 0.2, 0.5, 0.01)
        return L
    inputs = tuple(base[n].clone().requires_grad_(True) for n in names)
    assert torch.autograd.gradcheck(loss, inputs, eps=1e-6, atol=1e-6, rtol=1e-4)
    L, stats = pgo.ppo_loss(*pgo.forward(base, o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"]),
                            o["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"], mb["returns"], mb["acted"],
                            0.2, 0.5, 0.01)
    assert stats[5] == 3 and stats[6] == 1                      # agent 3 (no valid action) is not in S
    np.testing.assert_allclose(stats[4], 2 / 3)                  # agents 0 and 1 outside the clip range
    np.testing.assert_allclose(stats[3], -np.log([1.5, 0.5, 1.0]).mean(), rtol=1e-9)   # mean_S(log pi_old - log pi_new)


def test_clipped_agent_has_no_policy_gradient():
    """The clip rule itself: with ent_coef = vf_coef = 0, only agents 1 (unclipped) and 2 (tie) move the logits."""
    w, o, mb = tiny_case()
    p = pgo.params(w, requires_grad=False)
    logits, value = pgo.forward(p, o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"])
    logits = logits.detach().requires_grad_(True)
    L, _ = pgo.ppo_loss(logits, value.detach(), o["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"],
                        mb["returns"], mb["acted"], 0.2, 0.0, 0.0)
    L.backward()
    g = logits.grad.numpy()[0]
    assert (g[0] == 0).all() and (g[3] == 0).all()
    assert (np.abs(g[1]) > 0).any() and (np.abs(g[2]) > 0).any()
    assert (g[1][o["valid_actions"][0, 1] == 0] == 0).all()


def test_ppo_grad_bad_arguments(lib):  # noqa: F811
    from flatland_marl_b200 import policy
    L = policy.lib()
    assert L.fl_policy_workspace_bytes_grad_f32(0) == 0 and L.fl_policy_workspace_bytes_grad_f32(-5) == 0
    assert L.fl_policy_workspace_bytes_grad_f32(2) > 0
    assert L.fl_policy_workspace_bytes_grad_f32(2000) > L.fl_policy_workspace_bytes_grad_f32(1000)
    buf = C.create_string_buffer(64)
    p = C.cast(buf, C.c_void_p)
    n_t = 46
    good = (C.c_void_p * n_t)(*([p.value] * n_t))
    ws_need = int(L.fl_policy_workspace_bytes_grad_f32(6))

    def call(E=2, N=3, ptrs=None, wts=good, grads=good, ws_bytes=ws_need, clip=0.2, params=True):
        ptrs = ptrs or [p] * 14
        prm = policy.FlPpoParams(clip, 0.5, 0.01)
        return L.fl_policy_ppo_grad_f32(wts, ptrs[0], ws_bytes, E, N, *ptrs[1:11], C.byref(prm) if params else None, grads,
                                        ptrs[11], ptrs[12], ptrs[13], None)
    for k in range(14):                                    # workspace, 10 inputs, logits, value, stats
        ptrs = [p] * 14
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
