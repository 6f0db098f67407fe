"""CPU: the bf16 learner's arithmetic contract as a float64 oracle (tests/policy_grad_oracle_bf16.py), and the argument
checks of fl_policy_ppo_grad_bf16, fl_policy_forward_train_bf16 and fl_policy_tc_product_bf16 (include/flatland_policy_b200.h),
which return codes before any CUDA call."""
import ctypes as C

import numpy as np
import torch

import policy_grad_oracle as pgo
import policy_grad_oracle_bf16 as pgb
from test_cabi import lib  # noqa: F401  (fixture: builds and loads the libraries)
from test_policy_grad import golden_obs, tiny_case
import flatland_marl_b200.policy_weights as pw


def test_tc_weights_are_the_twenty_matrices():
    names = [n for n, _, _ in pw.weight_spec()]
    assert len(pgb.TC_WEIGHTS) == 20 and len(set(pgb.TC_WEIGHTS)) == 20
    assert set(pgb.TC_WEIGHTS) <= set(names)


def test_without_rounding_it_is_the_float64_oracle_bit_for_bit():
    w, o, mb = tiny_case()
    cases = [(o, mb)]
    g = {k: v[:6][None] for k, v in golden_obs("t03_l0_random", 46).items()}
    rng = np.random.RandomState(0)
    cases.append((g, dict(actions=rng.randint(0, 5, (1, 6)).astype(np.uint8), log_probs=-rng.rand(1, 6), advantages=np.array([-0.4]),
                          returns=np.array([1.2]), acted=np.array([1], np.uint8))))
    for obs, m in cases:
        ref = pgo.loss_and_grads(w, obs, m)
        got = pgb.loss_and_grads(w, obs, m, rounding=False)
        assert ref[0] == got[0]
        for a, b in zip(ref[1:4], got[1:4]):
            assert np.array_equal(a, b)
        for name in ref[4]:
            assert np.array_equal(ref[4][name], got[4][name]), name


def test_with_rounding_the_products_are_hand_rounded_float64_products():
    rng = np.random.RandomState(1)
    x = torch.tensor(rng.randn(5, 7), dtype=torch.float64, requires_grad=True)
    w = torch.tensor(rng.randn(3, 7), dtype=torch.float64, requires_grad=True)
    b = torch.tensor(rng.randn(3), dtype=torch.float64, requires_grad=True)
    dy = torch.tensor(rng.randn(5, 3), dtype=torch.float64)

    def r(a):   # round to nearest even at bit 16 of the fp32 pattern, by hand
        u = a.detach().numpy().astype(np.float32).view(np.uint32).astype(np.uint64)
        u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
        return u.astype(np.uint32).view(np.float32).astype(np.float64)
    y = pgb.TcLinear.apply(x, w, b, True)
    y.backward(dy)
    X, W, DY = r(x), r(w), r(dy)
    assert not np.array_equal(X, x.detach().numpy())              # the case does round
    np.testing.assert_array_equal(y.detach().numpy(), X @ W.T + b.detach().numpy())
    np.testing.assert_array_equal(x.grad.numpy(), DY @ W)
    np.testing.assert_array_equal(w.grad.numpy(), DY.T @ X)
    np.testing.assert_array_equal(b.grad.numpy(), dy.numpy().sum(0))


def test_rounding_moves_the_gradients_only_by_bf16_amounts():
    w, o, mb = tiny_case()
    ref = pgo.loss_and_grads(w, o, mb)
    got = pgb.loss_and_grads(w, o, mb)
    assert np.abs(got[2] - ref[2]).max() < 5e-2
    total = np.concatenate([ref[4][n].ravel() for n in ref[4]])
    diff = np.concatenate([got[4][n].ravel() - ref[4][n].ravel() for n in ref[4]])
    assert 0 < np.linalg.norm(diff) < 5e-2 * np.linalg.norm(total)


def test_bf16_bad_arguments(lib):  # noqa: F811
    from flatland_marl_b200 import policy
    L = policy.lib()
    assert L.fl_policy_workspace_bytes_grad_bf16(0) == 0 and L.fl_policy_workspace_bytes_grad_bf16(-1) == 0
    assert L.fl_policy_workspace_bytes_grad_bf16(1000) == L.fl_policy_workspace_bytes_grad_f32(1000)
    buf = C.create_string_buffer(64)
    p = C.cast(buf, C.c_void_p)
    n_t = 46
    good = (C.c_void_p * n_t)(*([p.value] * n_t))
    ws_need = int(L.fl_policy_workspace_bytes_grad_bf16(6))

    def call(E=2, N=3, ptrs=None, wts=good, grads=good, ws_bytes=ws_need, clip=0.2, params=True):
        ptrs = ptrs or [p] * 14
        prm = policy.FlPpoParams(clip, 0.5, 0.01)
        return L.fl_policy_ppo_grad_bf16(wts, ptrs[0], ws_bytes, E, N, *ptrs[1:11], C.byref(prm) if params else None, grads,
                                         ptrs[11], ptrs[12], ptrs[13], None)
    for k in range(14):
        ptrs = [p] * 14
        ptrs[k] = None
        assert call(ptrs=ptrs) == -1, k
    assert call(wts=None) == -1 and call(grads=None) == -1 and call(params=False) == -1
    for k in (0, 17, 45):
        bad = (C.c_void_p * n_t)(*([p.value] * n_t))
        bad[k] = None
        assert call(wts=bad) == -1 and call(grads=bad) == -1
    assert call(E=0) == -1 and call(N=0) == -1 and call(E=-1) == -1
    assert call(ws_bytes=ws_need - 1) == -1 and call(clip=0.0) == -1 and call(clip=float("nan")) == -1
    assert call(E=2 ** 40, N=2 ** 30) == -1

    def fwd(E=2, N=3, k=None, ws_bytes=ws_need, wts=good):
        ptrs = [p] * 7
        if k is not None:
            ptrs[k] = None
        return L.fl_policy_forward_train_bf16(wts, ptrs[0], ws_bytes, E, N, *ptrs[1:7], None)
    for k in range(7):
        assert fwd(k=k) == -1, k
    assert fwd(wts=None) == -1 and fwd(E=0) == -1 and fwd(ws_bytes=ws_need - 1) == -1

    def prod(**kw):
        t = policy.FlTcProduct(kind=0, M=4, N=128, K=64, x1=p, ldx1=64, K1=64, w=p, c=p, ldc=128)
        for k, v in kw.items():
            setattr(t, k, v)
        return L.fl_policy_tc_product_bf16(C.byref(t), p, 64, None)
    assert L.fl_policy_tc_product_bf16(None, None, 0, None) == -1
    assert prod(kind=3) == -1 and prod(x1=None) == -1 and prod(w=None) == -1 and prod(c=None) == -1
    assert prod(K1=60) == -1 and prod(K2=4) == -1 and prod(M=-1) == -1 and prod(N=0) == -1
    assert prod(kind=1) == -1                                     # dX without dY
    assert prod(kind=2, dy=p) == -1                               # dW partials do not fit 64 bytes
