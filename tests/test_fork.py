"""Copies of environments on the device (fl_copy_envs, BatchedRailEnv.copy_from / fork_of / snapshot / restore, copy.deepcopy
of the façades).  A copy must be indistinguishable from its source: given the same actions it produces the same bytes
(observations, rewards, dones, agent state, elapsed steps, schedule position, status, stats), across in-place auto-resets too.
Integers and floats are compared bit-exactly."""
import copy
import ctypes as C

import numpy as np
import pytest

from test_cabi import lib  # noqa: F401  (fixture: builds and loads the library)
from test_gpu_parity import assert_same, compare_obs, compare_state, obs_plan  # noqa: F401

STATE = ["rc", "old_rc", "dir", "old_dir", "state", "ctr", "mal", "saved", "sig_mal", "deadlocked", "done", "nmal", "arrival",
         "elapsed", "sched_pos", "done_all", "status", "stats"]


def rows(obs, rewards, dones, t, e):
    """Everything a copy must reproduce of environment (row) e, as numpy."""
    d = {k: v[e] for k, v in obs.items()}
    d["rewards"], d["dones"] = rewards[e], dones[e]
    d.update({k: t[k][e] for k in STATE})
    return {k: v.cpu().numpy() for k, v in d.items()}


def slot(batch, e):
    return rows(batch.obs, batch.rewards, batch.dones, batch.t, e)


def assert_rows(got, want, what):
    for k in want:
        assert_same(got[k], want[k], "%s %s" % (what, k))


def random_actions(rng, n, N):
    return np.where(rng.rand(n, N) < 0.7, 2, rng.randint(0, 5, (n, N))).astype(np.uint8)


def short_worlds(config, n, T=None):
    import bench
    worlds = bench.load_worlds(config, n)
    if T:
        for w in worlds:
            w["T"] = T                          # short episodes: in-place resets happen within the test
    return worlds


def step(batch, a):
    import torch
    return batch.step(torch.from_numpy(np.ascontiguousarray(a)).to(batch.device))


def fork_and_follow(config, n_envs, src, dst, warm, T=None, max_steps=200):
    """Steps a batch `warm` times, copies slots src -> dst inside it, then gives each copy its source's actions until every
    source has been reset in place after an episode end, and five steps more: every step, copies equal sources and the
    other slots equal a control batch that was never copied into."""
    import flatland_marl_b200 as fb
    worlds = short_worlds(config, n_envs, T)
    batch = fb.BatchedRailEnv(worlds, auto_reset=True)
    control = fb.BatchedRailEnv(worlds, auto_reset=True)
    batch.reset(); control.reset()
    rng = np.random.RandomState(5)
    for _ in range(warm):
        a = random_actions(rng, n_envs, batch.N)
        step(batch, a); step(control, a)
    n0 = batch.launch_count()
    batch.copy_from(batch, src, dst)
    assert batch.launch_count() - n0 == 1
    others = [e for e in range(n_envs) if e not in dst]
    # the output rows come with the copy: no observe() in between
    for s, d in zip(src, dst):
        assert_rows(slot(batch, d), slot(batch, s), "copy %d <- %d" % (d, s))
    for e in others:
        assert_rows(slot(batch, e), slot(control, e), "untouched %d" % e)
    t, extra = 0, 5
    while t < max_steps and extra > 0:
        a = random_actions(rng, n_envs, batch.N)
        a[dst] = a[src]
        step(batch, a); step(control, a)
        t += 1
        for s, d in zip(src, dst):
            assert_rows(slot(batch, d), slot(batch, s), "step %d copy %d <- %d" % (t, d, s))
        for e in others:
            assert_rows(slot(batch, e), slot(control, e), "step %d untouched %d" % (t, e))
        if ((batch.t["status"][src] & fb._lib.ST_AUTO_RESET) != 0).all().item():
            extra -= 1
    assert extra == 0, "a source was never reset in place"
    return batch


# 1 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fork_and_follow_past_auto_reset():
    batch = fork_and_follow("Test_03", 8, [0, 1, 2], [5, 6, 7], warm=20, T=60)
    # the copies ran past an in-place reset: the schedule position went on past the first episode
    assert (batch.t["sched_pos"][[5, 6, 7]] > batch.t["elapsed"][[5, 6, 7]]).all().item()


# 2 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fork_and_diverge_matches_oracle():
    """Copies that then get their own actions equal an oracle that replays the source's actions up to the copy, then the
    copy's, with the same schedule rows."""
    import flatland_marl_b200 as fb
    from oracle import oracle as orc
    worlds = short_worlds("Test_03", 4)
    batch = fb.BatchedRailEnv(worlds)
    batch.reset()
    rng = np.random.RandomState(9)
    hist = []
    for _ in range(15):
        a = random_actions(rng, 4, batch.N)
        hist.append(a)
        step(batch, a)
    batch.copy_from(batch, [0, 1], [2, 3])
    oracles = {}
    for d, s in ((2, 0), (3, 1)):
        env = orc.OracleEnv(worlds[s])
        env.reset()
        for t, a in enumerate(hist):
            env.step(a[s], worlds[s]["sched"][t])
        oracles[d] = (env, s)
        compare_state(batch, d, env.state(), "copy %d at the fork" % d)
        compare_obs(batch, d, env.obs(), "copy %d at the fork obs" % d)
    for t in range(len(hist), len(hist) + 30):
        a = random_actions(rng, 4, batch.N)
        _, rew, don = step(batch, a)
        for d, (env, s) in oracles.items():
            orew, odon = env.step(a[d], worlds[s]["sched"][t])
            what = "copy %d step %d" % (d, t + 1)
            assert_same(rew[d].cpu().numpy(), orew, what + " rewards")
            assert_same(don[d].cpu().numpy(), odon, what + " dones")
            compare_state(batch, d, env.state(), what)
            compare_obs(batch, d, env.obs(), what + " obs")


# 3 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("caches", ["on", "off"])
def test_fork_across_worlds_equals_fresh_batch(obs_plan, caches):  # noqa: F811
    """The destination held another world (another number of unique targets, other walk-table sizes) with warm caches;
    after the copy it equals a fresh batch of the source's world stepped with the same actions."""
    import flatland_marl_b200 as fb
    from flatland_marl_b200.worlds import unique_target_slots
    if caches == "off":
        obs_plan({"treecache": 0, "pathcache": 0})
    worlds = short_worlds("Test_03", 4)
    batch = fb.BatchedRailEnv(worlds, reserve=0.5, min_slots=8)
    batch.reset()
    assert len(unique_target_slots(worlds[0])[0]) != len(unique_target_slots(worlds[1])[0])
    tot = batch.t["walk_total"].cpu().numpy()
    assert tuple(tot[0, :3]) != tuple(tot[1, :3])
    fresh = fb.BatchedRailEnv([worlds[0]], reserve=0.5, min_slots=8)
    fresh.reset()
    rng = np.random.RandomState(3)
    for _ in range(12):
        a = random_actions(rng, 4, batch.N)
        step(batch, a); step(fresh, a[:1])
    batch.copy_from(batch, [0], [1])
    assert batch.tokens[1] == batch.tokens[0]
    assert (batch.dist_numpy(1) == batch.dist_numpy(0)).all()
    for t in range(30):
        a = random_actions(rng, 4, batch.N)
        a[1] = a[0]
        step(batch, a); step(fresh, a[:1])
        assert_rows(slot(batch, 1), slot(fresh, 0), "step %d" % (t + 1))


# 4 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_fork_small_environments():
    """Test_00: 7 agents (the all-pairs MotionCheck, the fused observation kernel)."""
    fork_and_follow("Test_00", 4, [0, 1], [2, 3], warm=10, T=40)


@pytest.mark.gpu
def test_fork_large_environments():
    """Test_14: 425 agents (the split observation launch with its workspace, ~12 MB distance maps per environment)."""
    import flatland_marl_b200 as fb
    worlds = short_worlds("Test_14", 3)
    batch = fb.BatchedRailEnv(worlds, auto_reset=True)
    batch.reset()
    assert batch.observe_plan()["parts"] > 0
    rng = np.random.RandomState(14)
    for _ in range(10):
        step(batch, random_actions(rng, 3, batch.N))
    batch.copy_from(batch, [0], [2])
    assert (batch.dist_numpy(2) == batch.dist_numpy(0)).all()
    for t in range(25):
        a = random_actions(rng, 3, batch.N)
        a[2] = a[0]
        step(batch, a)
        assert_rows(slot(batch, 2), slot(batch, 0), "step %d" % (t + 1))


@pytest.mark.gpu
def test_fork_of_steps_alone():
    """fork_of into a second batch, then that batch stepped on its own equals its sources."""
    import flatland_marl_b200 as fb
    worlds = short_worlds("Test_03", 4, T=50)
    batch = fb.BatchedRailEnv(worlds, auto_reset=True)
    batch.reset()
    rng = np.random.RandomState(1)
    for _ in range(20):
        step(batch, random_actions(rng, 4, batch.N))
    n0 = batch.launch_count()
    fork = fb.BatchedRailEnv.fork_of(batch, [3, 1, 3])
    assert batch.launch_count() - n0 == 1                # no BFS, no walk tables: one copy launch
    assert fork.E == 3 and fork.auto_reset is True and fork.state_stride == batch.state_stride
    assert fork.tokens == [batch.tokens[3], batch.tokens[1], batch.tokens[3]]
    for k, s in enumerate([3, 1, 3]):
        assert_rows(slot(fork, k), slot(batch, s), "fork %d" % k)
    for t in range(45):
        a = random_actions(rng, 4, batch.N)
        b = a[[3, 1, 3]]
        b[2] = random_actions(rng, 1, batch.N)[0] if t >= 10 else b[2]   # the second copy of 3 diverges after 10 steps
        step(fork, b); step(batch, a)
        for k, s in enumerate([3, 1, 3][:2] if t >= 10 else [3, 1, 3]):
            assert_rows(slot(fork, k), slot(batch, s), "step %d fork %d" % (t + 1, k))
    assert (fork.t["stats"][:2, 0] >= 1).all().item()


# 5 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_snapshot_restore_replays_past_episode_end():
    import flatland_marl_b200 as fb
    worlds = short_worlds("Test_03", 4, T=40)
    batch = fb.BatchedRailEnv(worlds, auto_reset=True)
    batch.reset()
    rng = np.random.RandomState(2)
    for _ in range(10):
        step(batch, random_actions(rng, 4, batch.N))
    at_snap = [slot(batch, e) for e in range(4)]
    snap = batch.snapshot()
    assert isinstance(snap, fb.EnvSnapshot) and len(snap) == 4
    for e in range(4):
        assert_rows(rows(snap.obs, snap.rewards, snap.dones, snap.t, e), at_snap[e], "snapshot row %d" % e)
    acts = [random_actions(rng, 4, batch.N) for _ in range(50)]
    first = []
    for a in acts:
        step(batch, a)
        first.append([slot(batch, e) for e in range(4)])
    assert (batch.t["stats"][:, 0] >= 1).all().item()
    batch.restore(snap)
    for e in range(4):
        assert_rows(slot(batch, e), at_snap[e], "restored %d" % e)
    for t, a in enumerate(acts):
        step(batch, a)
        for e in range(4):
            assert_rows(slot(batch, e), first[t][e], "replay step %d env %d" % (t + 1, e))


@pytest.mark.gpu
def test_restore_one_row_into_branch_slots_and_token_guard():
    import flatland_marl_b200 as fb
    worlds = short_worlds("Test_03", 3)
    batch = fb.BatchedRailEnv(worlds + [worlds[0]] * 3)
    batch.reset()
    batch.copy_from(batch, [0, 0, 0], [3, 4, 5])            # branch slots 3..5 hold world 0
    rng = np.random.RandomState(4)
    for _ in range(8):
        step(batch, random_actions(rng, 6, batch.N))
    snap = batch.snapshot([0])
    want = rows(snap.obs, snap.rewards, snap.dones, snap.t, 0)
    for _ in range(5):
        step(batch, random_actions(rng, 6, batch.N))
    n0 = batch.launch_count()
    batch.restore(snap, rows=[0, 0, 0, 0], into=[0, 3, 4, 5])
    assert batch.launch_count() - n0 == 1
    for e in (0, 3, 4, 5):
        assert_rows(slot(batch, e), want, "restored into %d" % e)
    for t in range(10):
        a = random_actions(rng, 6, batch.N)
        a[[3, 4, 5]] = a[0]
        step(batch, a)
        for e in (3, 4, 5):
            assert_rows(slot(batch, e), slot(batch, 0), "branch %d step %d" % (e, t + 1))
    with pytest.raises(ValueError):
        batch.restore(snap, rows=[0], into=[1])             # slot 1 holds another world
    batch.replace_worlds([3], [worlds[0]])                   # same world dict, but uploaded again: a new token
    with pytest.raises(ValueError):
        batch.restore(snap, rows=[0], into=[3])
    batch.restore(snap, rows=[0], into=[4])


# 6 ---------------------------------------------------------------------------------------------------------------------
def facade_result(res):
    obs, rew, done, info = res
    attr, (forest, adj, norder, eorder) = obs
    return dict(attr=np.array(attr, np.float32), forest=np.array(forest, np.float32), adjacency=np.array(adj),
                node_order=np.array(norder), edge_order=np.array(eorder), rew=np.array([rew[i] for i in sorted(rew)]),
                done=np.array([done[k] for k in done if k != "__all__"] + [done["__all__"]]),
                info=np.array([[int(v[i]) if k != "speed" else v[i] for i in sorted(v)] for k, v in sorted(info.items())], np.float64))


def assert_facade(got, want, what):
    for k in want:
        assert_same(got[k], want[k], "%s %s" % (what, k))


def action_dict(rng, n):
    return {i: int(a) for i, a in enumerate(random_actions(rng, 1, n)[0])}


@pytest.mark.gpu
def test_deepcopy_facade_rail_env():
    import flatland_marl_b200 as fb
    w = short_worlds("Test_03", 1)[0]
    env, third = fb.RailEnv.from_world(w), fb.RailEnv.from_world(w)
    env.reset(); third.reset()
    rng = np.random.RandomState(6)
    for _ in range(12):
        a = action_dict(rng, env.get_num_agents())
        env.step(a); third.step(a)
    c = copy.deepcopy(env)
    assert c._batch is not env._batch and c._elapsed_steps == env._elapsed_steps and c.dones == env.dones
    for t in range(5):
        a = action_dict(rng, env.get_num_agents())
        r1, r2 = env.step(a), c.step(a)
        third.step(a)
        assert_facade(facade_result(r2), facade_result(r1), "step %d" % t)
    for t in range(10):                                        # the copy diverges; the original is unaffected
        a = action_dict(rng, env.get_num_agents())
        c.step(action_dict(rng, env.get_num_agents()))
        assert_facade(facade_result(env.step(a)), facade_result(third.step(a)), "original step %d" % t)


@pytest.mark.gpu
def test_deepcopy_of_view_and_of_batch():
    import torch
    import flatland_marl_b200 as fb
    worlds = short_worlds("Test_03", 3)
    batch = fb.BatchedRailEnv(worlds)
    control = fb.BatchedRailEnv(worlds)
    batch.reset(); control.reset()
    rng = np.random.RandomState(8)
    for _ in range(10):
        a = random_actions(rng, 3, batch.N)
        step(batch, a); step(control, a)
    view = fb.RailEnv.view(batch, worlds, 1)
    view.after_batch_step()
    c = copy.deepcopy(view)
    assert c._batch.E == 1
    for t in range(6):
        a = random_actions(rng, 3, batch.N)
        step(batch, a); step(control, a)
        got = c.step({i: int(x) for i, x in enumerate(a[1])})
        assert_facade(facade_result(got), facade_result(view.after_batch_step()), "view step %d" % t)
    b2 = copy.deepcopy(batch)
    assert b2.E == 3 and b2.tokens == batch.tokens
    for e in range(3):
        assert_rows(slot(b2, e), slot(batch, e), "deepcopy %d" % e)
    for t in range(6):
        a = random_actions(rng, 3, batch.N)
        step(b2, a); step(batch, a); step(control, a)
        for e in range(3):
            assert_rows(slot(b2, e), slot(batch, e), "deepcopy step %d env %d" % (t, e))
    for t in range(6):
        a = random_actions(rng, 3, batch.N)
        step(b2, random_actions(rng, 3, batch.N)); step(batch, a); step(control, a)
        for e in range(3):
            assert_rows(slot(batch, e), slot(control, e), "original step %d env %d" % (t, e))
    torch.cuda.synchronize()


# 7 ---------------------------------------------------------------------------------------------------------------------
def test_copy_envs_bad_arguments(lib):  # noqa: F811
    """Rejected with FL_ERR_BAD_ARG before any CUDA call (no device needed): the pointers below are never dereferenced."""
    import flatland_marl_b200 as fb

    def batch():
        b = fb._lib.FlBatch()
        b.E, b.N, b.H, b.W, b.n_slots, b.S = 4, 7, 30, 30, 3, 100
        b.grid_stride, b.dist_stride, b.ridx_stride = 904, 10800, 904
        b.state_stride, b.wlist_stride, b.whits_stride, b.pc_stride = 512, 2048, 256, 512
        for name in fb._lib._PTR:
            setattr(b, name, 1 << 20)
        return b
    ids = C.c_void_p(1 << 20)
    W, S = fb._lib.COPY_WORLD, fb._lib.COPY_STATE
    a, b = batch(), batch()

    def call(src, dst, n=2, parts=W | S, s_ids=ids, d_ids=ids, so=None, do=None):
        return lib.fl_copy_envs(src, dst, s_ids, d_ids, n, parts, so, do, None)
    assert call(None, C.byref(b)) == -1 and call(C.byref(a), None) == -1
    assert call(C.byref(a), C.byref(b), s_ids=None) == -1 and call(C.byref(a), C.byref(b), d_ids=None) == -1
    assert call(C.byref(a), C.byref(b), n=0) == -1 and call(C.byref(a), C.byref(b), n=5) == -1
    assert call(C.byref(a), C.byref(b), parts=4) == -1 and call(C.byref(a), C.byref(b), parts=0) == -1
    outs = fb._lib.FlObsBuffers()
    assert call(C.byref(a), C.byref(b), so=C.byref(outs)) == -1               # one output set only
    for field, value in (("N", 8), ("H", 31), ("n_slots", 4), ("S", 99), ("dist_stride", 10808), ("state_stride", 544),
                         ("wlist_stride", 2052), ("whits_stride", 260), ("pc_stride", 256), ("ridx_stride", 912)):
        c = batch()
        setattr(c, field, value)
        assert call(C.byref(a), C.byref(c)) == -1, field
    for name in ("grid", "sched", "dist", "gtab", "walk_total"):               # a world pointer NULL with FL_COPY_WORLD
        c = batch()
        setattr(c, name, None)
        assert call(C.byref(a), C.byref(c), parts=W) == -1, name
        assert call(C.byref(c), C.byref(a), parts=W) == -1, name
    c = batch()
    c.tree_cache = None                                                       # a cache in one batch only
    assert call(C.byref(a), C.byref(c), parts=W) == -1
    snap = fb._lib.FlBatch()                                                  # a snapshot store: state pointers only
    snap.E, snap.N = 2, 7
    assert call(C.byref(a), C.byref(snap), parts=W | S) == -1
    snap.rc = None
    assert call(C.byref(a), C.byref(snap), parts=S) == -1
    assert call(C.byref(a), C.byref(b), parts=S, so=C.byref(outs), do=C.byref(outs)) == -1   # NULL output rows


@pytest.mark.gpu
def test_copy_and_restore_reject_bad_ids():
    import flatland_marl_b200 as fb
    worlds = short_worlds("Test_03", 4)
    batch = fb.BatchedRailEnv(worlds)
    batch.reset()
    for s, d in (([0, 1], [1, 2]), ([0, 1], [2, 2]), ([0], [4]), ([-1], [2]), ([0, 1], [2])):
        with pytest.raises(ValueError):
            batch.copy_from(batch, s, d)
    other = fb.BatchedRailEnv(short_worlds("Test_00", 1))
    other.reset()
    with pytest.raises(ValueError):
        batch.copy_from(other, [0], [1])                     # another layout
    snap = batch.snapshot([0, 1])
    for r, d in (([2], [0]), ([0, 1], [3, 3]), ([0], [4])):
        with pytest.raises(ValueError):
            batch.restore(snap, rows=r, into=d)
    with pytest.raises(ValueError):
        batch.snapshot([4])
