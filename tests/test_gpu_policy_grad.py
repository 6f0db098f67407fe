"""GPU: the PPO loss and gradients of the fp32 network (fl_policy_ppo_grad_f32, PolicyLearner) against float64 autograd through
tests/policy_grad_oracle.py.

Tolerance.  Every one of the 46 gradients must satisfy ||g - g_ref||_2 <= 1e-4 ||g_ref||_2, and the statistics agree to 1e-5
relative (1e-6 absolute for those that are zero).  Both bounds were set before measuring.  Measured on one B200, the worst
per-tensor relative gradient error over the cases below is 1.05e-6 (Test_03 golden rows); each case prints its own (-s)."""
import numpy as np
import pytest
import torch

import policy_grad_oracle as pgo

pytestmark = pytest.mark.gpu
GRAD_RTOL = 1e-4
OBS = ("agent_attr", "forest", "adjacency", "node_order", "edge_order", "valid_actions")


@pytest.fixture(scope="module")
def learner():
    from flatland_marl_b200 import PolicyLearner
    return PolicyLearner(None, seed=0)


def dev(a, device):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device)


def golden_rows(golden, fixture, steps):
    g = golden(fixture)
    return {k: np.stack([g["obs%d_%s" % (s, "attr" if k == "agent_attr" else k)] for s in steps]) for k in OBS}


def live_rows(config, E, n_steps, seed=0, T=None):
    """Observations of a BatchedRailEnv after n_steps random steps (done agents, 0 / 1 valid actions, null tree nodes)."""
    import flatland_marl_b200 as fb
    from test_fork import short_worlds
    batch = fb.BatchedRailEnv(short_worlds(config, E, T=T), auto_reset=True)
    obs = batch.reset()
    rng = np.random.RandomState(seed)
    for _ in range(n_steps):
        obs, _, _ = batch.step(torch.from_numpy(rng.randint(0, 5, (E, batch.N)).astype(np.uint8)).to(batch.device))
    return {k: obs[k].cpu().numpy() for k in OBS}


def null_nodes(forest):
    """Null tree nodes: the observation's "no branch here" placeholder, a non-root node whose features are all -1 once +inf
    is replaced by -1 (eval_env.py:76; recognised by value in policy.cu's k_prep)."""
    f = np.where(np.isposinf(forest), -1.0, forest)
    return (f[..., 1:, :] == -1.0).all(-1)


def make_minibatch(learner, obs, seed, acted=None):
    """Actions and log pi sampled by the fp32 actor of the learner's parameters (so log pi_old is bit-equal to the loss
    kernel's log pi_new), then log pi_old moved by -log r for r in {1 (exact tie), 1.5, 0.6, 1.1} per agent; advantages of
    both signs and one exact 0."""
    actor = learner.actor("fp32")
    d = {k: dev(obs[k], learner.device) for k in OBS}
    logits, _ = actor.forward(d)
    a, lp = actor.sample_actions(logits, d["valid_actions"], seed, 0)
    E, N = obs["agent_attr"].shape[:2]
    rng = np.random.RandomState(seed)
    r = np.array([1.0, 1.5, 0.6, 1.1])[rng.randint(0, 4, (E, N))]
    old = (lp.cpu().numpy() - np.log(r).astype(np.float32)).astype(np.float32)
    old[r == 1.0] = lp.cpu().numpy()[r == 1.0]
    adv = (rng.randn(E) * 2).astype(np.float32)
    if E > 2:
        adv[0] = 0.0
    mb = dict(actions=a.cpu().numpy(), log_probs=old, advantages=adv, returns=(rng.randn(E) * 3).astype(np.float32),
              acted=np.ones(E, np.uint8) if acted is None else np.asarray(acted, np.uint8))
    return mb


def device_mb(learner, obs, mb):
    d = {k: dev(obs[k], learner.device) for k in ("agent_attr", "forest", "adjacency", "node_order", "valid_actions")}
    d.update({k: dev(v, learner.device) for k, v in mb.items()})
    return d


def check_against_oracle(learner, obs, mb, what, clip=0.2, vf=0.5, ent=0.01):
    stats = learner.ppo_grad(device_mb(learner, obs, mb), clip, vf, ent).cpu().numpy().astype(np.float64)
    w = {k: v.detach().cpu().numpy() for k, v in learner.named_parameters()}
    _, ref_stats, ref_logits, ref_val, ref_g = pgo.loss_and_grads(w, obs, mb, clip, vf, ent)
    logits, value = learner.last_outputs()
    np.testing.assert_allclose(logits.cpu().numpy(), ref_logits, rtol=0, atol=1e-4)
    np.testing.assert_allclose(value.cpu().numpy(), ref_val, rtol=0, atol=1e-4)
    worst = 0.0
    for name, p in learner.named_parameters():
        g, ref = p.grad.cpu().numpy().astype(np.float64), ref_g[name]
        err, nrm = np.linalg.norm(g - ref), np.linalg.norm(ref)
        assert np.isfinite(g).all(), name
        assert err <= GRAD_RTOL * nrm + 1e-12, "%s: %s |g - ref| = %.3e, |ref| = %.3e" % (what, name, err, nrm)
        if nrm > 0:
            worst = max(worst, err / nrm)
    np.testing.assert_allclose(stats, ref_stats, rtol=1e-5, atol=1e-6, err_msg=what)
    print("%s: worst relative gradient error %.2e, stats %s" % (what, worst, np.array2string(stats, precision=4)))
    return stats, worst


@pytest.mark.parametrize("fixture,steps", [("t00_l0_random", (3, 35)), ("t02_l0_forward", (119, 235)), ("t03_l0_random", (46, 89)),
                                           ("t08_l0_greedy", (0, 2)), ("t14_l0_forward", (1,))])
def test_golden_observations(learner, golden, fixture, steps):
    obs = golden_rows(golden, fixture, steps)
    mb = make_minibatch(learner, obs, seed=len(steps) + 7)
    stats, _ = check_against_oracle(learner, obs, mb, fixture)
    assert 0 < stats[4] < 1                                # both sides of the clip range and in-range agents occur


def test_live_rows_with_reset_rows_and_degenerate_agents(learner):
    obs = live_rows("Test_02", 6, 30, seed=4, T=25)
    assert null_nodes(obs["forest"]).any()
    # the valid-action mask only enters the loss: give some agents no valid action and some exactly one
    obs["valid_actions"][0, :3] = 0
    obs["valid_actions"][2, :4] = np.eye(5, dtype=np.uint8)[[0, 2, 3, 4]]
    nvalid = obs["valid_actions"].sum(-1)
    assert (nvalid == 0).any() and (nvalid == 1).any()
    mb = make_minibatch(learner, obs, seed=11, acted=[1, 0, 1, 1, 0, 1])
    stats, _ = check_against_oracle(learner, obs, mb, "live Test_02")
    assert stats[6] == 4


def test_test14_rows_long_attention(learner):
    obs = live_rows("Test_14", 2, 12, seed=2)
    assert obs["agent_attr"].shape[1] == 425
    mb = make_minibatch(learner, obs, seed=5)
    check_against_oracle(learner, obs, mb, "live Test_14")


def test_training_forward_is_the_fp32_forward_and_calls_are_deterministic(learner, golden):
    obs = golden_rows(golden, "t03_l0_random", (0, 46, 89, 133))
    mb = make_minibatch(learner, obs, seed=3, acted=[1, 1, 0, 1])
    d = device_mb(learner, obs, mb)
    runs = []
    for _ in range(2):
        stats = learner.ppo_grad(d).clone()
        logits, value = (t.clone() for t in learner.last_outputs())
        runs.append((stats, logits, value, [p.grad.clone() for p in learner.parameters()]))
    for a, b in zip(runs[0][:3], runs[1][:3]):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))
    for ga, gb in zip(runs[0][3], runs[1][3]):
        assert torch.equal(ga.view(torch.int32), gb.view(torch.int32))
    lf, vf = learner.forward({k: d[k] for k in ("agent_attr", "forest", "adjacency", "node_order")})
    assert torch.equal(lf.view(torch.int32), runs[0][1].view(torch.int32)) and torch.equal(vf.view(torch.int32), runs[0][2].view(torch.int32))
    ref = learner.actor("fp32").forward({k: d[k] for k in ("agent_attr", "forest", "adjacency", "node_order")})
    assert torch.equal(ref[0].view(torch.int32), runs[0][1].view(torch.int32))
    assert torch.equal(ref[1].view(torch.int32), runs[0][2].view(torch.int32))


def make_rollout(learner, E=16, T=24, precision="fp32"):
    import flatland_marl_b200 as fb
    from test_fork import short_worlds
    batch = fb.BatchedRailEnv(short_worlds("Test_02", E, T=20), auto_reset=True)
    batch.reset()
    ro = fb.Rollout(batch, learner.actor(precision), T=T, seed=7)
    ro.collect()
    ro.advantages(0.99, 0.95)
    return ro


def test_first_pass_over_an_fp32_rollout_has_ratio_one(learner):
    ro = make_rollout(learner)
    n = ro.T * ro.batch.E
    g = torch.Generator(device="cpu").manual_seed(1)
    perm = torch.randperm(n, generator=g)
    for ids in (perm[:64], perm[64:200], torch.arange(n)):
        stats = learner.ppo_grad(ro.minibatch(ids.tolist())).cpu().numpy()
        assert stats[3] == 0.0 and stats[4] == 0.0, stats
        assert stats[5] > 0 and np.isfinite(stats).all()
    mb = ro.minibatch(perm[:5].to(learner.device))
    assert mb["agent_attr"].shape == (5, ro.batch.N, 83) and mb["advantages"].shape == (5,)
    with pytest.raises(ValueError):
        ro.minibatch([n])


def test_sgd_step_lowers_the_loss(learner):
    ro = make_rollout(learner)
    mb = ro.minibatch(list(range(0, ro.T * ro.batch.E, 3)))
    L0 = float(learner.ppo_grad(mb)[7])
    saved = [p.detach().clone() for p in learner.parameters()]
    gnorm = float(torch.sqrt(sum((p.grad.double() ** 2).sum() for p in learner.parameters())))
    eta = 1e-3 / gnorm
    with torch.no_grad():
        for p in learner.parameters():
            p -= eta * p.grad
    L1 = float(learner.ppo_grad(mb)[7])
    with torch.no_grad():
        for p, s in zip(learner.parameters(), saved):
            p.copy_(s)
    assert L1 < L0 - 0.25 * eta * gnorm ** 2, (L0, L1, eta * gnorm ** 2)


def test_training_loop_no_torch_sync_no_nan():
    """collect -> advantages -> minibatches -> ppo_grad -> clip_grad_norm_ -> Adam.step, then a new actor; the torch side of
    an update makes no host synchronisation (the library's documented one per fp32 forward and per ppo_grad is inside the C
    call)."""
    import flatland_marl_b200 as fb
    from test_fork import short_worlds
    learner = fb.PolicyLearner(None, seed=1)
    opt = torch.optim.Adam(learner.parameters(), lr=1e-4)
    batch = fb.BatchedRailEnv(short_worlds("Test_02", 8, T=20), auto_reset=True)
    batch.reset()
    ro = fb.Rollout(batch, learner.actor(), T=16, seed=3)
    n = ro.T * batch.E
    for it in range(3):
        ro.collect()
        ro.advantages()
        perm = torch.randperm(n, device=learner.device)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            for k in range(0, n, 48):
                stats = learner.ppo_grad(ro.minibatch(perm[k:k + 48]))
                torch.nn.utils.clip_grad_norm_(learner.parameters(), 1.0)
                opt.step()
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert torch.isfinite(stats).all()
        ro.actor = learner.actor()
    assert all(torch.isfinite(p).all() for p in learner.parameters())
