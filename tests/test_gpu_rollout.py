"""GPU: PPO rollout collection on the device — seeded sampling with log-probabilities (fl_policy_sample_actions), GAE
(fl_policy_gae) and the Rollout trajectory buffer — against the numpy oracle and against replays on forked batches."""
import numpy as np
import pytest
import torch

import rollout_oracle as rorc
from test_fork import short_worlds

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def actor():
    from flatland_marl_b200.policy import BatchedActor
    return BatchedActor(None, seed=0)


def random_case(E=64, N=50, seed=5):
    rng = np.random.RandomState(seed)
    logits = (rng.randn(E, N, 5) * 2).astype(np.float32)
    valid = (rng.rand(E, N, 5) < 0.6).astype(np.uint8)
    valid[0, :5] = 0                                   # no valid action -> 0, log-probability 0
    valid[1, :5] = np.eye(5, dtype=np.uint8)           # one valid action -> that action, log-probability 0
    return logits, valid


def dev(a, actor):
    return torch.from_numpy(np.ascontiguousarray(a)).to(actor.device)


@pytest.mark.parametrize("seed,step,env_offset", [(0, 0, 0), (1234, 7, 0), (2 ** 40 + 3, 2 ** 33 + 1, 1000), (99, 5, 2 ** 32 - 64)])
def test_sample_actions_against_oracle(actor, seed, step, env_offset):
    logits, valid = random_case()
    a, lp = actor.sample_actions(dev(logits, actor), dev(valid, actor), seed, step, env_offset)
    a, lp = a.cpu().numpy(), lp.cpu().numpy()
    want, wlp, margin = rorc.sample_actions(logits, valid, seed, step, env_offset)
    ok = margin > 1e-6
    assert (~ok).sum() <= 5
    assert (a[ok] == want[ok]).all()
    np.testing.assert_allclose(lp[ok], wlp[ok], rtol=0, atol=1e-5)
    assert (a[0, :5] == 0).all() and (lp[0, :5] == 0).all()
    assert (a[1, :5] == np.arange(5)).all() and (lp[1, :5] == 0).all()
    chosen_valid = np.take_along_axis(valid, a[..., None].astype(np.int64), axis=2)[..., 0]
    assert ((chosen_valid == 1) | (valid.sum(axis=2) == 0)).all()


def test_sampling_distribution(actor):
    """204,800 draws of one logit row (64 x 50 agents x 64 steps): every action's frequency within 5 sigma of its softmax
    probability; the invalid action is never drawn."""
    row = np.array([0.3, -1.2, 2.0, 0.0, 0.9], np.float32)
    mask = np.array([1, 1, 1, 0, 1], np.uint8)
    logits = dev(np.broadcast_to(row, (64, 50, 5)), actor)
    valid = dev(np.broadcast_to(mask, (64, 50, 5)), actor)
    counts = np.zeros(5, np.int64)
    for step in range(64):
        a, _ = actor.sample_actions(logits, valid, 42, step)
        counts += np.bincount(a.cpu().numpy().ravel(), minlength=5)
    n = counts.sum()
    assert n == 204800 and counts[3] == 0
    p = np.where(mask == 1, np.exp(row - row.max()), 0.0)
    p /= p.sum()
    sigma = np.sqrt(n * p * (1 - p))
    assert (np.abs(counts - n * p) <= 5 * sigma).all(), (counts, n * p)


def test_shards_sample_what_one_device_samples(actor):
    logits, valid = random_case()
    a, lp = (t.clone() for t in actor.sample_actions(dev(logits, actor), dev(valid, actor), 77, 3, 0))
    a0, lp0 = (t.clone() for t in actor.sample_actions(dev(logits[:32], actor), dev(valid[:32], actor), 77, 3, 0))
    a1, lp1 = (t.clone() for t in actor.sample_actions(dev(logits[32:], actor), dev(valid[32:], actor), 77, 3, 32))
    assert torch.equal(a, torch.cat([a0, a1])) and torch.equal(lp, torch.cat([lp0, lp1]))


@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (1.0, 1.0), (0.0, 0.0)])
def test_gae_against_oracle(actor, gamma, lam):
    T, E, N = 37, 129, 7
    rng = np.random.RandomState(11)
    rewards = rng.randint(-40, 5, (T + 1, E, N)).astype(np.int32)
    dones = (rng.rand(T + 1, E, N + 1) < 0.05).astype(np.uint8)
    values = (rng.randn(T + 1, E) * 10).astype(np.float32)
    acted = (rng.rand(T, E) < 0.9).astype(np.uint8)
    adv, ret = (torch.empty((T, E), dtype=torch.float32, device=actor.device) for _ in range(2))
    d = [dev(x, actor) for x in (rewards, dones, values, acted)]
    rc = actor.lib.fl_policy_gae(*(x.data_ptr() for x in d), T, E, N, gamma, lam, adv.data_ptr(), ret.data_ptr(), actor._stream())
    assert rc == 0
    want_a, want_r = rorc.gae(rewards, dones, values, acted, gamma, lam)
    adv, ret = adv.cpu().numpy(), ret.cpu().numpy()
    np.testing.assert_allclose(adv, want_a, rtol=1e-6, atol=0)
    np.testing.assert_allclose(ret, want_r, rtol=1e-6, atol=0)
    assert (adv[acted == 0] == 0).all() and (ret[acted == 0] == 0).all()


OUT_KEYS = ("agent_attr", "forest", "adjacency", "node_order", "edge_order", "valid_actions", "dist_target", "rewards", "dones")


def outs(batch):
    d = dict(batch.obs)
    d["rewards"], d["dones"] = batch.rewards, batch.dones
    return d


def assert_row(buf, k, batch, what):
    for key in OUT_KEYS:
        got, want = buf[key][k], outs(batch)[key]
        assert torch.equal(got.view(torch.uint8) if got.is_floating_point() else got,
                           want.view(torch.uint8) if want.is_floating_point() else want), "%s: row %d %s" % (what, k, key)


def replay(fork, buf, T, what):
    """Steps `fork` (a copy taken before the collection) with the buffer's actions: every row must come out byte for byte;
    returns 1 - done_all before each step."""
    assert_row(buf, 0, fork, what)
    acted = []
    for k in range(T):
        acted.append((1 - fork.t["done_all"]).cpu().numpy())
        fork.step(buf["actions"][k].contiguous())
        assert_row(buf, k + 1, fork, what)
    return np.stack(acted)


def test_collect_end_to_end(actor):
    import flatland_marl_b200 as fb
    E, T, seed, step0 = 32, 48, 1234, 5
    batch = fb.BatchedRailEnv(short_worlds("Test_02", E, T=20), auto_reset=True)
    batch.reset()
    rng = np.random.RandomState(3)
    for _ in range(7):                                 # episodes out of phase: some environments end inside the window
        batch.step(torch.from_numpy(rng.randint(0, 5, (E, batch.N)).astype(np.uint8)).to(batch.device))
    forks = [fb.BatchedRailEnv.fork_of(batch, range(E)) for _ in range(3)]
    ro = fb.Rollout(batch, actor, T=T, seed=seed, step=step0)
    buf = {k: v.clone() for k, v in ro.collect().items()}
    assert ro.step == step0 + T
    # the rows are the ones the batch produced, and acted is 1 - done_all before each step
    acted = replay(forks[0], buf, T, "replay")
    assert (buf["acted"].cpu().numpy() == acted).all()
    assert (acted == 0).any(), "no reset step inside the window"
    # actions, log-probabilities and values are what forward + sample_actions give on the stored rows, bit for bit
    for k in range(T + 1):
        obs = {key: buf[key][k] for key in ("agent_attr", "forest", "adjacency", "node_order")}
        logits, value = actor.forward(obs)
        assert torch.equal(value, buf["values"][k]), k
        if k < T:
            a, lp = actor.sample_actions(logits, buf["valid_actions"][k], seed, step0 + k)
            assert torch.equal(a, buf["actions"][k]) and torch.equal(lp, buf["log_probs"][k]), k
    # GAE over the buffer
    adv, ret = ro.advantages(0.99, 0.95)
    h = {k: v.cpu().numpy() for k, v in buf.items()}
    want_a, want_r = rorc.gae(h["rewards"], h["dones"], h["values"], h["acted"], 0.99, 0.95)
    np.testing.assert_allclose(adv.cpu().numpy(), want_a, rtol=1e-6, atol=0)
    np.testing.assert_allclose(ret.cpu().numpy(), want_r, rtol=1e-6, atol=0)
    # same seed on a copy: the same buffer; another seed: other actions
    same = fb.Rollout(forks[1], actor, T=T, seed=seed, step=step0).collect()
    for k in buf:
        assert torch.equal(same[k], buf[k]), k
    other = fb.Rollout(forks[2], actor, T=T, seed=seed + 1, step=step0).collect()
    assert not torch.equal(other["actions"], buf["actions"])
    # the next collect continues the stream and the batch from where the last one stopped
    nxt = ro.collect()
    assert ro.step == step0 + 2 * T
    for key in OUT_KEYS:
        assert torch.equal(nxt[key][0], buf[key][T]), key


def test_collect_through_reset_pipeline(actor):
    import flatland_marl_b200 as fb
    E, T = 8, 40
    worlds = short_worlds("Test_02", E + 12, T=15)
    batch = fb.BatchedRailEnv(worlds[:E], auto_reset=True, reserve=1.0, min_slots=8)
    pipe = fb.ResetPipeline(batch, fb.PackSource(worlds[E:]))
    pipe.reset()
    fork = fb.BatchedRailEnv.fork_of(batch, range(E))
    fork_pipe = fb.ResetPipeline(fork, fb.PackSource(worlds[E:]))
    buf = fb.Rollout(pipe, actor, T=T, seed=9).collect()
    assert pipe.replaced > 0
    assert_row(buf, 0, fork, "pipeline")
    for k in range(T):
        assert (buf["acted"][k] == 1 - fork.t["done_all"]).all(), k
        fork_pipe.step(buf["actions"][k].contiguous())
        assert_row(buf, k + 1, fork, "pipeline")
    assert fork_pipe.replaced == pipe.replaced


def test_collect_makes_no_host_sync_and_one_copy_launch_per_step(actor):
    import flatland_marl_b200 as fb
    E, T = 16, 12
    batch = fb.BatchedRailEnv(short_worlds("Test_02", E, T=10), auto_reset=True)
    batch.reset()
    plain = fb.BatchedRailEnv.fork_of(batch, range(E))
    a = torch.zeros((E, batch.N), dtype=torch.uint8, device=batch.device)
    n0 = plain.launch_count()
    for _ in range(T):
        plain.step(a)
    per_steps = plain.launch_count() - n0
    ro = fb.Rollout(batch, actor, T=T, seed=1)
    ro.collect()                                       # first call: lazily created scratch may sync
    torch.cuda.synchronize()
    n0 = batch.launch_count()
    torch.cuda.set_sync_debug_mode("error")
    try:
        ro.collect()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert batch.launch_count() - n0 == per_steps + T + 1     # + one row copy per step, + row 0


def test_rollout_refuses_batch_without_auto_reset(actor):
    import flatland_marl_b200 as fb
    batch = fb.BatchedRailEnv(short_worlds("Test_02", 2))
    with pytest.raises(ValueError):
        fb.Rollout(batch, actor, T=4, seed=0)
