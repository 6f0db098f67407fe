"""CPU: the argument checks of fl_policy_forward_f32 and the size of its workspace (include/flatland_policy_b200.h).  Every
rejected call below has exactly one bad argument and returns FL_ERR_BAD_ARG before any CUDA call."""
import ctypes as C

from test_cabi import lib  # noqa: F401  (fixture: builds and loads the libraries)

N_T = 46


def test_f32_workspace_bytes(lib):  # noqa: F811
    from flatland_marl_b200 import policy
    L = policy.lib()
    assert L.fl_policy_workspace_bytes_f32(0) == 0 and L.fl_policy_workspace_bytes_f32(-1) == 0
    sizes = [L.fl_policy_workspace_bytes_f32(n) for n in (1, 2, 1000, 51200)]
    assert 0 < sizes[0] < sizes[1] < sizes[2] < sizes[3]
    for n in (1, 1000, 51200):
        assert L.fl_policy_workspace_bytes_f32(n) < L.fl_policy_workspace_bytes_grad_f32(n)


def test_f32_forward_bad_arguments(lib):  # noqa: F811
    from flatland_marl_b200 import policy
    L = policy.lib()
    buf = C.create_string_buffer(64)
    p = C.cast(buf, C.c_void_p)
    good = (C.c_void_p * N_T)(*([p.value] * N_T))
    ws_need = int(L.fl_policy_workspace_bytes_f32(6))

    def fwd(E=2, N=3, k=None, ws_bytes=ws_need, wts=good):
        ptrs = [p] * 7                     # workspace, agent_attr, forest, adjacency, node_order, logits, value
        if k is not None:
            ptrs[k] = None
        return L.fl_policy_forward_f32(wts, ptrs[0], ws_bytes, E, N, *ptrs[1:7], None)
    for k in range(7):
        assert fwd(k=k) == -1, k
    assert fwd(wts=None) == -1
    for k in range(N_T):
        bad = (C.c_void_p * N_T)(*([p.value] * N_T))
        bad[k] = None
        assert fwd(wts=bad) == -1, k
    assert fwd(E=0) == -1 and fwd(N=0) == -1 and fwd(E=-1) == -1 and fwd(N=-3) == -1
    assert fwd(ws_bytes=ws_need - 1) == -1
    assert fwd(E=2 ** 40, N=2 ** 30) == -1                         # E * N * 31 node ids do not fit 32 bits
