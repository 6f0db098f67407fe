"""numpy mirrors of the PPO rollout kernels — TEST INFRASTRUCTURE ONLY.

Restates fl_policy_sample_actions (Philox4x32-10 uniforms, the masked soft choice, log-probabilities) and fl_policy_gae of
include/flatland_policy_b200.h, so that tests can check the kernels bit for bit.  The choice is np.random.choice's cdf search
(oracle/policy_oracle.choose_actions) with the uniform as a parameter: with u = policy_oracle.CHOICE_U it gives
policy_oracle.choose_actions' actions (tests/test_rollout.py checks this).
"""
import numpy as np

F32 = np.float32
_M32 = 0xFFFFFFFF


def philox4x32_10(counter, key):
    """Philox4x32-10 (Random123): counter (4 words), key (2 words) -> 4 words, as Python ints."""
    c0, c1, c2, c3 = (int(x) & _M32 for x in counter)
    k0, k1 = (int(x) & _M32 for x in key)
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & _M32, p1 & _M32, ((p0 >> 32) ^ c3 ^ k1) & _M32, p0 & _M32
        k0, k1 = (k0 + 0x9E3779B9) & _M32, (k1 + 0xBB67AE85) & _M32
    return c0, c1, c2, c3


def uniform53(seed, step, env, agent):
    """The uniform of agent `agent` of global environment `env` at `step`: 53 bits of Philox output, in [0, 1)."""
    x0, x1, _, _ = philox4x32_10((step & _M32, (step >> 32) & _M32, env, agent), (seed & _M32, (seed >> 32) & _M32))
    return ((x0 >> 5) * 67108864.0 + (x1 >> 6)) / 9007199254740992.0


def soft_choice(x, nz, u):
    """np.random.choice(nz, p=softmax(x)) with its one uniform u, in the kernels' arithmetic (fp32 exponentials, float64 cdf);
    returns (action, float64 log-probability, distance of u from the nearest inner cdf step)."""
    x = np.asarray(x, F32)
    mx = x.max()
    e = np.exp(x - mx).astype(F32)
    s = F32(e.sum(dtype=F32))
    cdf = np.cumsum((e / s).astype(np.float64))
    cdf = cdf / cdf[-1]
    j = int(np.argmax(cdf > u)) if (cdf > u).any() else len(nz) - 1
    x64 = x.astype(np.float64)
    lp = (x64[j] - x64.max()) - np.log(np.exp(x64 - x64.max()).sum())
    margin = float(np.min(np.abs(cdf[:-1] - u))) if len(nz) > 1 else 1.0
    return int(nz[j]), lp, margin


def sample_actions(logits, valid, seed, step, env_offset=0):
    """fl_policy_sample_actions on logits [E,N,5], valid [E,N,5]: (actions u8 [E,N], log_probs f64 [E,N], margin [E,N]).
    margin: distance of the agent's uniform from the nearest cdf step (tests exclude agents below their float tolerance).
    policy_oracle.choose_actions is the special case u = CHOICE_U for every agent."""
    logits, valid = np.asarray(logits, F32), np.asarray(valid)
    E, N = logits.shape[:2]
    acts = np.zeros((E, N), np.uint8)
    lps = np.zeros((E, N), np.float64)
    margin = np.ones((E, N), np.float64)
    for e in range(E):
        for i in range(N):
            nz = valid[e, i].nonzero()[0]
            if nz.size == 0:
                continue
            acts[e, i], lps[e, i], margin[e, i] = soft_choice(logits[e, i][nz], nz, uniform53(seed, step, env_offset + e, i))
    return acts, lps, margin


def gae(rewards, dones, values, acted, gamma, lam):
    """fl_policy_gae in float64: rewards [T+1,E,N], dones [T+1,E,N+1] (column N read), values [T+1,E], acted [T,E] ->
    (advantages, returns) [T,E].  Row 0 of rewards and dones is not read."""
    rewards, dones = np.asarray(rewards), np.asarray(dones)
    values, acted = np.asarray(values, np.float64), np.asarray(acted)
    T, E = acted.shape
    g, lm = float(np.float32(gamma)), float(np.float32(lam))
    adv = np.zeros((T, E), np.float64)
    ret = np.zeros((T, E), np.float64)
    a_next = np.zeros(E, np.float64)
    for k in range(T - 1, -1, -1):
        live = 1.0 - (dones[k + 1, :, -1] != 0)
        r = rewards[k + 1].astype(np.int64).sum(axis=1) / rewards.shape[2]
        a = r + g * values[k + 1] * live - values[k] + g * lm * live * a_next
        a = np.where(acted[k] != 0, a, 0.0)
        adv[k], ret[k] = a, np.where(acted[k] != 0, a + values[k], 0.0)
        a_next = a
    return adv, ret
