"""CPU: the options of the PPO loss (FlPpoOptions, include/flatland_policy_b200.h: clipped value loss and advantage
normalisation) restated in float64 (tests/policy_grad_oracle_ex.py) — its reduction to the plain loss, its normalisation
against numpy, its gradients against finite differences — and the argument checks of fl_policy_ppo_grad_ex_f32 / _bf16 and
fl_policy_ppo_moments, which return codes before any CUDA call."""
import ctypes as C

import numpy as np
import pytest
import torch

import policy_grad_oracle as pgo
import policy_grad_oracle_ex as pge
from test_cabi import lib  # noqa: F401  (fixture: builds and loads the libraries)
from test_policy_grad import golden_obs, tiny_case
import flatland_marl_b200.policy_weights as pw

OBS = ("agent_attr", "forest", "adjacency", "node_order", "edge_order", "valid_actions")
CLIP, VF, ENT, VCLIP = 0.2, 0.5, 0.01, 0.2
GRAD_NAMES = ["actor_net.4.bias", "critic_net.4.bias", "critic_net.2.bias", "actor_net.2.bias", "tree_lstm.W_c.bias"]


def four_rows():
    """Four Test_00 rows of 4 agents, advantages of both signs, and behaviour values V_old and returns R placed around each
    row's V (float64 forward) so that every value-clip case occurs with a wide margin (no branch changes under finite
    differences): row 0 V above the band and the clipped square larger, row 1 V below the band and the unclipped square
    larger, row 2 V inside the band, row 3 V below the band and the clipped square larger."""
    steps = (3, 35, 67, 99)
    o = {k: np.stack([golden_obs("t00_l0_random", s)[k][:4] for s in steps]) for k in OBS}
    o["valid_actions"] = o["valid_actions"].copy()
    o["valid_actions"][:, :, 4] = 1                       # every agent in S, some with one valid action
    rng = np.random.RandomState(2)
    actions = np.argmax(o["valid_actions"] * rng.rand(4, 4, 5), -1).astype(np.uint8)
    w = pw.init_weights(5)
    with torch.no_grad():
        logits, value = pgo.forward(pgo.params(w, False), o["agent_attr"], o["forest"], o["adjacency"], o["node_order"],
                                    o["edge_order"])
        lp, _, _ = pgo.log_probs(logits, o["valid_actions"], actions)
    V = value.numpy()
    old = lp.numpy() - np.log(np.array([1.0, 1.5, 0.6, 1.1]))[rng.randint(0, 4, (4, 4))]
    vo = V + np.array([-0.5, 0.5, 0.05, 0.5])            # V - V_old: 0.5 (above), -0.5 (below), -0.05 (inside), -0.5
    ret = V + np.array([1.0, 1.0, -1.0, -1.0])
    mb = dict(actions=actions, log_probs=old, advantages=np.array([0.7, -1.3, 2.1, 0.2]), returns=ret,
              acted=np.ones(4, np.uint8), values=vo)
    return w, o, mb


def value_cases(V, mb, c):
    """Per row: (V above the band, below it, the clipped square strictly larger)."""
    Vo, R = np.asarray(mb["values"]), np.asarray(mb["returns"])
    Vc = Vo + np.clip(V - Vo, -c, c)
    return V - Vo > c, V - Vo < -c, (Vc - R) ** 2 > (V - R) ** 2


def loss_fn(w, o, mb, **opts):
    base = pgo.params(w, requires_grad=False)

    def loss(*ts):
        p = dict(base)
        p.update(zip(GRAD_NAMES, ts))
        logits, value = pgo.forward(p, o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"])
        L, _ = pge.ppo_loss_ex(logits, value, o["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"],
                               mb["returns"], mb["acted"], CLIP, VF, ENT, old_values=mb.get("values"), **opts)
        return L
    return loss, tuple(base[n].clone().requires_grad_(True) for n in GRAD_NAMES)


def test_options_off_is_the_plain_loss_bit_for_bit():
    w, o, mb = four_rows()
    p = pgo.params(w)
    logits, value = pgo.forward(p, o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"])
    args = (logits, value, o["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"], mb["returns"], mb["acted"],
            CLIP, VF, ENT)
    L0, s0 = pgo.ppo_loss(*args)
    g0 = torch.autograd.grad(L0, [p[n] for n in GRAD_NAMES], retain_graph=True)
    L1, s1 = pge.ppo_loss_ex(*args, vf_clip=0.0, norm_adv=False, adv_eps=1e-8, old_values=mb["values"])
    g1 = torch.autograd.grad(L1, [p[n] for n in GRAD_NAMES])
    assert L0.item() == L1.item() and np.array_equal(s0, s1)
    assert all(torch.equal(a, b) for a, b in zip(g0, g1))
    # a band wider than any |V - V_old| and the unclipped square: the value term and the whole loss stay the same
    L2, s2 = pge.ppo_loss_ex(*args, vf_clip=100.0, old_values=mb["values"])
    np.testing.assert_allclose(s2, s0, rtol=1e-12, atol=0)


def test_normalised_advantages_are_numpys_over_the_agent_list():
    rng = np.random.RandomState(0)
    va = (rng.rand(9, 6, 5) < 0.12).astype(np.uint8)
    acted = np.array([1, 1, 0, 1, 1, 1, 0, 1, 1], np.uint8)
    adv = (rng.randn(9) * 3 + 1).astype(np.float32)
    S = pge.agent_set(va, acted)
    a = np.repeat(adv.astype(np.float64), S.sum(-1))     # the row advantage once per agent of S
    assert a.size == S.sum() and len(np.unique(S.sum(-1))) > 2
    mom = pge.moments(va, acted, adv)
    np.testing.assert_allclose(mom, [a.sum(), (a * a).sum()], rtol=1e-14)
    for eps in (1e-8, 0.0, 0.5):
        want = (adv.astype(np.float64) - a.mean()) / (a.std(ddof=1) + float(np.float32(eps)))
        got = pge.normalised_advantages(adv, int(S.sum()), mom, eps)
        np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-7)
        assert np.array_equal(got, got.astype(np.float32).astype(np.float64))     # rounded once to fp32
        assert torch.allclose(torch.as_tensor(a).std(), torch.as_tensor(np.std(a, ddof=1)), rtol=1e-12)
    # |S| = 1 and equal advantages: sigma = 0, so A_hat = 0 with and without adv_eps
    assert (pge.normalised_advantages(adv[:1], 1, [adv[0], adv[0] ** 2], 1e-8) == 0).all()
    eq = np.full(9, 0.5, np.float32)
    for eps in (1e-8, 0.0):
        assert (pge.normalised_advantages(eq, int(S.sum()), pge.moments(va, acted, eq), eps) == 0).all()


def test_gradcheck_both_options_value_clip_cases():
    w, o, mb = four_rows()
    with torch.no_grad():
        _, V = pgo.forward(pgo.params(w, False), o["agent_attr"], o["forest"], o["adjacency"], o["node_order"], o["edge_order"])
    above, below, clipped = value_cases(V.numpy(), mb, VCLIP)
    assert above.tolist() == [True, False, False, False] and below.tolist() == [False, True, False, True]
    assert clipped.tolist() == [True, False, False, True]
    loss, inputs = loss_fn(w, o, mb, vf_clip=VCLIP, norm_adv=True, adv_eps=1e-8)
    assert torch.autograd.gradcheck(loss, inputs, eps=1e-6, atol=1e-6, rtol=1e-4)
    # the clipped rows give the critic no gradient: with only them acted, the critic's last bias has none
    only = dict(mb, acted=np.array([1, 0, 0, 1], np.uint8))
    loss, inputs = loss_fn(w, o, only, vf_clip=VCLIP, norm_adv=True, adv_eps=1e-8)
    g = torch.autograd.grad(loss(*inputs), inputs)
    assert float(g[1].abs().max()) == 0.0 and float(g[0].abs().max()) > 0


def test_gradcheck_single_agent_set():
    """|S| = 1: sigma = 0, so A_hat = 0 and only the entropy and the value term move the parameters."""
    w, o, mb = tiny_case()
    o = dict(o, valid_actions=o["valid_actions"].copy())
    o["valid_actions"][0, 1:] = 0
    mb = dict(mb, values=np.array([0.0]))
    loss, inputs = loss_fn(w, o, mb, vf_clip=VCLIP, norm_adv=True, adv_eps=1e-8)
    assert torch.autograd.gradcheck(loss, inputs, eps=1e-6, atol=1e-6, rtol=1e-4)
    with torch.no_grad():
        logits, value = pgo.forward(pgo.params(w, False), o["agent_attr"], o["forest"], o["adjacency"], o["node_order"],
                                    o["edge_order"])
    _, stats = pge.ppo_loss_ex(logits, value, o["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"],
                               mb["returns"], mb["acted"], CLIP, VF, ENT, vf_clip=VCLIP, norm_adv=True, old_values=mb["values"])
    assert stats[5] == 1 and stats[0] == 0.0                # A_hat = 0: the policy term is 0


@pytest.mark.parametrize("adv_eps", [1e-8, 0.0])
def test_gradcheck_equal_advantages(adv_eps):
    w, o, mb = four_rows()
    mb = dict(mb, advantages=np.full(4, 0.5))
    loss, inputs = loss_fn(w, o, mb, vf_clip=VCLIP, norm_adv=True, adv_eps=adv_eps)
    assert torch.autograd.gradcheck(loss, inputs, eps=1e-6, atol=1e-6, rtol=1e-4)
    with torch.no_grad():
        logits, value = pgo.forward(pgo.params(w, False), o["agent_attr"], o["forest"], o["adjacency"], o["node_order"],
                                    o["edge_order"])
    _, stats = pge.ppo_loss_ex(logits, value, o["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"],
                               mb["returns"], mb["acted"], CLIP, VF, ENT, vf_clip=VCLIP, norm_adv=True, adv_eps=adv_eps,
                               old_values=mb["values"])
    assert stats[0] == 0.0 and np.isfinite(stats).all()


def test_ppo_grad_ex_and_moments_bad_arguments(lib):  # noqa: F811
    from flatland_marl_b200 import policy
    L = policy.lib()
    buf = C.create_string_buffer(64)
    p = C.cast(buf, C.c_void_p)
    n_t = 46
    good = (C.c_void_p * n_t)(*([p.value] * n_t))
    ws_need = int(L.fl_policy_workspace_bytes_grad_f32(6))
    assert ws_need == int(L.fl_policy_workspace_bytes_grad_bf16(6))

    for fn in (L.fl_policy_ppo_grad_ex_f32, L.fl_policy_ppo_grad_ex_bf16):
        def call(ptrs=None, clip=0.2, gcnt=p, old=p, gmom=p, opts=(0.2, 1, 1e-8), ws_bytes=ws_need, E=2, N=3):
            ptrs = ptrs or [p] * 14
            prm = policy.FlPpoParams(clip, 0.5, 0.01)
            o = policy.FlPpoOptions(*opts) if opts is not None else None
            return fn(good, ptrs[0], ws_bytes, E, N, *ptrs[1:11], gcnt, C.byref(prm), good, ptrs[11], ptrs[12], ptrs[13], None,
                      old, gmom, C.byref(o) if o is not None else None)
        for k in range(14):                                # workspace, 10 inputs, logits, value, stats: the plain checks
            ptrs = [p] * 14
            ptrs[k] = None
            assert call(ptrs=ptrs) == -1, k
        assert call(clip=0.0) == -1 and call(E=0) == -1 and call(ws_bytes=ws_need - 1) == -1
        assert call(opts=None) == -1
        for vf_clip in (-0.1, -1e-30, float("nan"), float("-inf")):
            assert call(opts=(vf_clip, 0, 1e-8)) == -1, vf_clip
        for norm in (2, -1, 7):
            assert call(opts=(0.2, norm, 1e-8)) == -1, norm
        for eps in (-1e-8, float("inf"), float("nan")):
            assert call(opts=(0.0, 1, eps)) == -1, eps
        assert call(old=None, opts=(0.2, 0, 1e-8)) == -1           # clipped value loss without V_old
        assert call(gcnt=None, gmom=p) == -1                       # the minibatch's moments without its counts
        assert call(gcnt=None, gmom=p, opts=(0.0, 0, 1e-8)) == -1

    def moments(E=2, N=3, ptrs=None):
        ptrs = ptrs or [p] * 4
        return L.fl_policy_ppo_moments(E, N, *ptrs, None)
    for k in range(4):
        ptrs = [p] * 4
        ptrs[k] = None
        assert moments(ptrs=ptrs) == -1, k
    assert moments(E=0) == -1 and moments(N=0) == -1 and moments(E=-1) == -1 and moments(E=2 ** 40, N=2 ** 30) == -1


def test_learner_option_checks_need_no_device():
    """PolicyLearner validates the options in Python before any call; the checks are those of the library."""
    from flatland_marl_b200.learner import PolicyLearner
    import inspect
    sig = inspect.signature(PolicyLearner.ppo_grad)
    assert [(k, sig.parameters[k].default) for k in ("vf_clip", "norm_adv", "adv_eps")] == \
        [("vf_clip", 0.0), ("norm_adv", False), ("adv_eps", 1e-8)]
    lrn = PolicyLearner.__new__(PolicyLearner)
    lrn.device = torch.device("cpu")
    mb = {"values": torch.zeros(3)}
    o, old = lrn._options(mb, 3, 0.0, False, 1e-8)
    assert (o.vf_clip, o.norm_adv, old) == (0.0, 0, None)
    o, old = lrn._options(mb, 3, 0.2, True, 0.0)
    assert o.norm_adv == 1 and old == mb["values"].data_ptr()
    for bad in (dict(vf_clip=-0.1), dict(vf_clip=float("nan")), dict(adv_eps=-1.0), dict(adv_eps=float("inf")),
                dict(norm_adv=2)):
        kw = dict(vf_clip=0.0, norm_adv=False, adv_eps=1e-8)
        kw.update(bad)
        with pytest.raises(ValueError):
            lrn._options(mb, 3, **kw)
    with pytest.raises(KeyError):
        lrn._options({}, 3, 0.2, False, 1e-8)
    with pytest.raises(ValueError):
        lrn._options({"values": torch.zeros(4)}, 3, 0.2, False, 1e-8)
