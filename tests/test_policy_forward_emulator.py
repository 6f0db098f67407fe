"""CPU: the float64 restatement of the bf16 policy forward (tests/policy_forward_emulator.py) against the numpy oracle of
the reference network, and the observation trees it generates against the observation's invariants.

With exact=True and fp32 packed weights the emulator is the reference network in float64: it must equal
oracle/policy_oracle.forward (fp32) to 2e-5 on every recorded observation, so that the stage checks of
tests/test_gpu_policy_stages.py compare the kernels with the reference's semantics and not with a copy of them.  With the
kernels' arithmetic (bf16 operands and stores, the fitted GELU) its logits stay within the 3e-2 that
tests/test_gpu_policy.py allows the bf16 forward."""
import os

import numpy as np
import pytest
import torch

import policy_forward_emulator as pfe
from oracle import policy_oracle as po

GOLD = os.path.join(os.path.dirname(__file__), "golden")
EXACT_ATOL = 2e-5
LOGIT_ATOL = 3e-2


@pytest.fixture(scope="module")
def weights():
    from flatland_marl_b200 import policy_weights as pw
    return pw.init_weights(0)


def golden_cases(golden):
    with np.load(os.path.join(GOLD, "policy_golden.npz")) as z:
        cases = list(zip(z["case_fixture"], z["case_step"]))
    for fixture, step in cases:
        g = golden(str(fixture))
        p = "obs%d_" % int(step)
        yield "%s/%d" % (fixture, step), {k: g[p + ("attr" if k == "agent_attr" else k)][None]
                                           for k in ("agent_attr", "forest", "adjacency", "node_order", "edge_order")}


def oracle(w, obs):
    return po.forward(w, obs["agent_attr"], po.clean_forest(obs["forest"]), obs["adjacency"], obs["node_order"], obs["edge_order"])


def test_exact_emulator_is_the_reference_network(weights, golden):
    t = pfe.packed(weights, rounding=False)
    worst = 0.0
    for name, obs in golden_cases(golden):
        want, wval = oracle(weights, obs)
        lg, v = pfe.forward(t, obs, exact=True)
        np.testing.assert_allclose(lg.numpy(), want, rtol=0, atol=EXACT_ATOL, err_msg=name)
        np.testing.assert_allclose(v.numpy(), wval, rtol=0, atol=EXACT_ATOL, err_msg=name)
        worst = max(worst, float(np.abs(lg.numpy() - want).max()), float(np.abs(v.numpy() - wval).max()))
    print("exact emulator vs policy_oracle: worst %.2e" % worst)


def test_kernel_arithmetic_stays_within_the_bf16_tolerance(weights, golden):
    t = pfe.packed(weights)
    worst = 0.0
    for name, obs in golden_cases(golden):
        want, wval = oracle(weights, obs)
        lg, v = pfe.forward(t, obs)
        np.testing.assert_allclose(lg.numpy(), want, rtol=0, atol=LOGIT_ATOL, err_msg=name)
        np.testing.assert_allclose(v.numpy(), wval, rtol=0, atol=LOGIT_ATOL, err_msg=name)
        worst = max(worst, float(np.abs(lg.numpy() - want).max()))
    print("bf16 emulator vs policy_oracle: worst |logit| error %.2e" % worst)


def test_kernel_functions_reduce_to_the_exact_ones_without_rounding():
    """The two arithmetics differ only where they should: the GELU fit stays within 4e-5 of the erf form, and the
    attention with exact=False on bf16-representable P equals the exact attention up to the rounding of P."""
    x = torch.linspace(-12, 12, 20001, dtype=torch.float64)
    assert float((pfe.gelu(x) - pfe.gelu(x, exact=True)).abs().max()) < 4e-5
    rng = np.random.RandomState(3)
    qkv = pfe.bf16(torch.from_numpy(rng.normal(0, 1, (6, 768))))
    a, b = pfe.attention(qkv, 2, 3), pfe.attention(qkv, 2, 3, exact=True)
    assert float((a - b).abs().max()) < 2e-2
    # the keys of another environment never enter: changing environment 1 leaves environment 0's rows as they were
    q2 = qkv.clone()
    q2[3:] += 1.0
    assert torch.equal(pfe.attention(q2, 2, 3)[:3], a[:3])


def check_tree(no, adj, eo, forest, null_inner):
    exists = no >= 0
    n = int(exists.sum())
    if n == 0:
        assert (adj == -2).all() and (eo == -2).all()
        return
    assert exists[:n].all() and not exists[n:].any() and n % 3 == 1       # slots 0..n-1, root plus whole groups
    assert (no <= 10).all()
    assert int((no == 0).sum()) <= 21
    assert int((no >= 1).sum()) <= 10
    children = {}
    for k in range(n - 1):
        p_, c_, ad = adj[k]
        assert c_ == k + 1 and ad == (k % 3) - 1 and 0 <= p_ < c_
        assert eo[k] == no[p_]
        children.setdefault(int(p_), []).append(int(c_))
    assert (adj[n - 1:] == -2).all() and (eo[n - 1:] == -2).all()
    for v in range(n):
        ch = children.get(v, [])
        assert len(ch) in (0, 3) and ch == sorted(ch) and (not ch or ch[2] - ch[0] == 2)
        assert no[v] == (0 if not ch else 1 + max(no[c] for c in ch))
    parents = sorted(children)
    assert [children[p][0] for p in parents] == sorted(children[p][0] for p in parents)   # breadth-first numbering
    f = np.where(np.isposinf(forest), -1.0, forest)
    null = (f == -1.0).all(-1)
    assert not null[0]
    if not null_inner:
        assert all(no[v] == 0 for v in range(1, n) if null[v])            # null nodes are leaves


@pytest.mark.parametrize("null_inner", [False, True])
def test_generated_trees_are_valid_observations(weights, null_inner):
    rng = np.random.RandomState(11 + null_inner)
    kinds = ["random"] * 40 + ["deep"] * 8 + ["full"] * 4 + ["root"] * 4 + ["empty"] * 4
    tr = pfe.random_trees(rng, len(kinds), null_inner=null_inner, kinds=kinds)
    for i in range(len(kinds)):
        check_tree(tr["node_order"][i], tr["adjacency"][i], tr["edge_order"][i], tr["forest"][i], null_inner)
    assert tr["node_order"].max() == 10                                      # the deepest tree occurs
    nl = pfe.random_trees(rng, 64)
    f = np.where(np.isposinf(nl["forest"]), -1.0, nl["forest"])
    assert ((f[:, 1:] == -1).all(-1) & (nl["node_order"][:, 1:] == 0)).any()  # null leaves occur
    if null_inner:
        f = np.where(np.isposinf(tr["forest"]), -1.0, tr["forest"])
        assert ((f[:, 1:] == -1).all(-1) & (tr["node_order"][:, 1:] > 0)).any()
    # policy_oracle accepts them, and the exact emulator agrees with it on them
    obs = {k: v.reshape((6, 10) + v.shape[1:]) for k, v in tr.items()}
    obs["agent_attr"] = rng.normal(0, 1, (6, 10, 83)).astype(np.float32)
    want, wval = oracle(weights, obs)
    assert np.isfinite(want).all() and np.isfinite(wval).all()
    lg, v = pfe.forward(pfe.packed(weights, rounding=False), obs, exact=True)
    np.testing.assert_allclose(lg.numpy(), want, rtol=0, atol=EXACT_ATOL)
    np.testing.assert_allclose(v.numpy(), wval, rtol=0, atol=EXACT_ATOL)
