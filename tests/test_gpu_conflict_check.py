"""The queued conflict check of k_observe's tree phase (observe.cuh, phase 4 stage 2) against the C oracle, bit for bit, over
whole episodes on the fused kernel and on the split launch, on a world made to reach the cases where the check's shortcuts
could differ from the three separate interval tests of treeobs.cpp:379-465:
  * windows cut at the horizon: a check at pt <= 1 (the window starts at row 0) and one at pt = 500 (post = pt);
  * trains slower than 1/8 (rows per cell > 8: the index entry refers to the agent record for its speed);
  * DONE agents while other trains are still moving;
  * long-lived entries (the last element of a path, occupied up to row 500) inside a checked window;
  * buckets of more than 16 entries.
The kernel counts the checks of each case in its debug counters (FlBatch.debug_clocks words 26-30); the test asserts from
those and from the oracle's states that every case occurred."""
import numpy as np
import pytest

from test_gpu_parity import compare_obs, compare_state, obs_plan  # noqa: F401

pytestmark = pytest.mark.gpu

DONE = 6
CASES = ["window from row 0", "window at row 500", "bucket above 16 entries", "long-lived entry visited", "train slower than 1/8"]


@pytest.fixture(scope="module")
def slow_world():
    """The Test_03 world of the golden fixtures (35 x 30, 50 agents) with a speed mix from 1 down to 1/50: trains slower
    than 1/8 (10, 20 and 50 rows per cell), whose trees reach the 500-row horizon within a few cells; its malfunction
    schedule is kept."""
    import os
    from conftest import GOLDEN_DIR
    with np.load(os.path.join(GOLDEN_DIR, "t03_l0_random.npz")) as z:
        w = {k: z[k] for k in ("H", "W", "N", "T", "grid", "init_pos", "init_dir", "target", "earliest", "latest", "sched")}
    w["speed"] = np.resize(np.array([0.1, 0.25, 1.0, 0.05, 0.5, 0.02, 1.0 / 3.0, 1.0]), int(w["N"])).astype(np.float64)
    w["T"] = np.int64(max(int(w["T"]), 700))
    assert (np.ceil(1.0 / w["speed"]) > 8).any()
    return w


def actions_of(N, T, seed):
    """Mostly forward, so that trains cross the map and finish; some stops and turns for contention."""
    rng = np.random.RandomState(seed)
    return np.where(rng.rand(T, N) < 0.75, 2, rng.randint(0, 5, size=(T, N))).astype(np.uint8)


@pytest.mark.parametrize("plan", [{"parts": 0}, {"parts": 2}], ids=["fused", "split"])
def test_conflict_check_matches_oracle_on_edge_cases(slow_world, obs_plan, plan):
    import torch
    import flatland_marl_b200 as fb
    from oracle import oracle as orc
    obs_plan(plan)
    w, N, sched = slow_world, int(slow_world["N"]), slow_world["sched"]
    T = int(w["T"])
    acts = [actions_of(N, T, 11), actions_of(N, T, 12)]
    batch = fb.BatchedRailEnv([dict(w), dict(w)], sched_rows=len(sched), debug_clocks=True)
    envs = [orc.OracleEnv(w), orc.OracleEnv(w)]
    batch.reset()
    for e, env in enumerate(envs):
        env.reset()
        compare_state(batch, e, env.state(), "env %d reset" % e)
        compare_obs(batch, e, env.obs(), "env %d reset obs" % e)
    counts = np.zeros(5, np.int64)
    done_while_moving = 0
    alive = [True, True]
    for t in range(T):
        act = np.stack([a[t] for a in acts])
        batch.step(torch.from_numpy(act).to(batch.device))
        counts += batch.debug_clocks[:, 26:31].sum(0).cpu().numpy()
        for e, env in enumerate(envs):
            if not alive[e]:
                continue
            _, odon = env.step(act[e], sched[t % len(sched)])
            what = "env %d step %d" % (e, t + 1)
            s = env.state()
            compare_state(batch, e, s, what)
            compare_obs(batch, e, env.obs(), what + " obs")
            done_while_moving += int((s["state"] == DONE).any() and (s["state"] == 3).any())
            alive[e] = not odon[-1]
        if not any(alive):
            break
    missing = [c for c, n in zip(CASES, counts) if n == 0]
    assert not missing, "cases never checked: %s (counts %s)" % (missing, counts.tolist())
    assert done_while_moving > 0, "no DONE agent while other trains moved"
