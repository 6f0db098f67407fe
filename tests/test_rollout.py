"""PPO rollout pieces that need no GPU: the oracle's Philox4x32-10 and GAE against known answers, and the argument checks of
fl_policy_sample_actions / fl_policy_gae (include/flatland_policy_b200.h), which return codes before any CUDA call."""
import ctypes as C

import numpy as np
import pytest

import rollout_oracle as rorc
from oracle import policy_oracle as po
from test_cabi import lib  # noqa: F401  (fixture: builds and loads the libraries)


@pytest.mark.parametrize("counter,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(counter, key, want):
    """The Random123 known-answer vectors of Philox4x32-10."""
    assert rorc.philox4x32_10(counter, key) == want


def test_uniform53_rule():
    x0, x1, _, _ = rorc.philox4x32_10((7, 0, 3, 11), (1234, 0))
    u = rorc.uniform53(1234, 7, 3, 11)
    assert u == ((x0 >> 5) * 2.0 ** 26 + (x1 >> 6)) / 2.0 ** 53 and 0.0 <= u < 1.0
    assert rorc.uniform53(1234, 7, 3, 12) != u and rorc.uniform53(1235, 7, 3, 11) != u and rorc.uniform53(1234, 2 ** 32 + 7, 3, 11) != u


def test_sample_actions_oracle_special_cases():
    """No valid action -> 0 with log-probability 0; one valid action -> that action with log-probability 0; the log-probability
    is the masked log-softmax of the chosen action."""
    logits = np.array([[[1.0, 2.0, 3.0, 4.0, 5.0]] * 3], np.float32)
    valid = np.array([[[0, 0, 0, 0, 0], [0, 0, 1, 0, 0], [1, 1, 0, 1, 0]]], np.uint8)
    a, lp, _ = rorc.sample_actions(logits, valid, seed=3, step=0)
    assert a[0, 0] == 0 and lp[0, 0] == 0.0
    assert a[0, 1] == 2 and lp[0, 1] == 0.0
    x = np.array([1.0, 2.0, 4.0])
    assert a[0, 2] in (0, 1, 3)
    np.testing.assert_allclose(lp[0, 2], (x - np.log(np.exp(x).sum()))[[0, 1, 3].index(int(a[0, 2]))], rtol=0, atol=1e-12)


def test_choose_actions_is_the_fixed_uniform_case():
    """The reference's evaluation choice (np.random.choice after seed 42, policy_oracle.choose_actions) is the sampling rule
    with the one uniform it draws, as k_choose and k_sample share their choice code."""
    rng = np.random.RandomState(1)
    logits = (rng.randn(40, 50, 5) * 3).astype(np.float32)
    valid = (rng.rand(40, 50, 5) < 0.6).astype(np.uint8)
    want = po.choose_actions(logits, valid)
    for idx in np.ndindex(*logits.shape[:-1]):
        nz = valid[idx].nonzero()[0]
        got = rorc.soft_choice(logits[idx][nz], nz, po.CHOICE_U)[0] if nz.size else 0
        assert got == want[idx], idx


def gae_case():
    """T = 3, two environments of two agents.  Environment 0 ends its episode in step 1 (dones[2]["__all__"] = 1), so step 2
    only resets it (acted = 0); environment 1 runs through and is bootstrapped from V_3."""
    rewards = np.zeros((4, 2, 2), np.int32)
    dones = np.zeros((4, 2, 3), np.uint8)
    rewards[0] = 99                                    # row 0 is not read
    dones[0, :, 2] = 1
    rewards[1, 0], rewards[2, 0] = (1, 3), (4, 6)      # mean 2, then 5
    rewards[1:, 1] = (0, 2)                            # mean 1 every step
    dones[2, 0] = 1
    values = np.array([[0.5, 0.0], [1.0, 0.0], [2.0, 0.0], [3.0, 10.0]], np.float32)
    acted = np.array([[1, 1], [1, 1], [0, 1]], np.uint8)
    return rewards, dones, values, acted


def test_gae_oracle_hand_computed():
    rewards, dones, values, acted = gae_case()
    # gamma = lam = 1: returns are the plain reward sums up to the episode end (env 0) or up to T plus V_T (env 1)
    adv, ret = rorc.gae(rewards, dones, values, acted, 1.0, 1.0)
    np.testing.assert_array_equal(ret[:, 0], [7.0, 5.0, 0.0])
    np.testing.assert_array_equal(adv[:, 0], [6.5, 4.0, 0.0])
    np.testing.assert_array_equal(ret[:, 1], [13.0, 12.0, 11.0])
    # gamma = lam = 0.5, env 0: delta_1 = 5 - 1 (episode end: no V_2), delta_0 = 2 + 0.5 * 1 - 0.5, A_0 = 2 + 0.25 * 4
    adv, ret = rorc.gae(rewards, dones, values, acted, 0.5, 0.5)
    np.testing.assert_array_equal(adv[:, 0], [3.0, 4.0, 0.0])
    np.testing.assert_array_equal(ret[:, 0], [3.5, 5.0, 0.0])
    # env 1, values 0 until V_3 = 10: A_2 = 1 + 5, A_1 = 1 + 0.25 * 6, A_0 = 1 + 0.25 * 2.5
    np.testing.assert_array_equal(adv[:, 1], [1.625, 2.5, 6.0])


def test_sample_and_gae_bad_arguments(lib):  # noqa: F811
    from flatland_marl_b200 import policy
    L = policy.lib()
    buf = C.create_string_buffer(64)
    p = C.cast(buf, C.c_void_p)

    def sample(E=2, N=3, off=0, ptrs=(p, p, p, p)):
        return L.fl_policy_sample_actions(ptrs[0], ptrs[1], E, N, off, 1, 0, ptrs[2], ptrs[3], None)
    for k in range(4):
        ptrs = [p] * 4
        ptrs[k] = None
        assert sample(ptrs=ptrs) == -1
    assert sample(E=0) == -1 and sample(N=0) == -1 and sample(E=-1) == -1 and sample(off=-1) == -1
    assert sample(off=2 ** 32 - 1) == -1 and sample(E=2, off=2 ** 32 - 1) == -1
    assert sample(E=1, off=2 ** 32) == -1

    def gae(T=2, E=2, N=3, ptrs=(p,) * 6):
        return L.fl_policy_gae(ptrs[0], ptrs[1], ptrs[2], ptrs[3], T, E, N, 0.99, 0.95, ptrs[4], ptrs[5], None)
    for k in range(6):
        ptrs = [p] * 6
        ptrs[k] = None
        assert gae(ptrs=ptrs) == -1
    assert gae(T=0) == -1 and gae(E=0) == -1 and gae(N=0) == -1 and gae(T=-3) == -1
