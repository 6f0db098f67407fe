"""BatchedActor — the reference's `Actor` (solution/plfActor.py:7-74) for a whole lock-step batch on one B200.

Host side of the policy forward pass (SURVEY.md §8 f1): owns the packed bf16 parameters and the device scratch,
and calls the tcgen05 kernels through the C ABI of include/flatland_policy_b200.h.  It consumes the observation
tensors of `BatchedRailEnv.observe()` where they lie on the device.  No CPU fallback: the CUDA library and a
CUDA device are required.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import policy_weights as pw
from ._lib import FlatlandB200Error

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "policy", "libflatland_policy_b200.so")
LAYERS = pw.N_TRANSFORMER

EXPORTS = ["fl_policy_abi_version", "fl_policy_workspace_bytes", "fl_policy_forward", "fl_policy_workspace_bytes_f32",
           "fl_policy_forward_f32", "fl_policy_workspace_bytes_grad_f32", "fl_policy_ppo_grad_f32", "fl_policy_workspace_bytes_grad_bf16",
           "fl_policy_ppo_grad_bf16", "fl_policy_forward_train_bf16", "fl_policy_tc_product_bf16", "fl_policy_ppo_counts",
           "fl_policy_ppo_grad_shard_f32", "fl_policy_ppo_grad_shard_bf16", "fl_policy_ppo_moments", "fl_policy_ppo_grad_ex_f32",
           "fl_policy_ppo_grad_ex_bf16", "fl_policy_choose_actions",
           "fl_policy_sample_actions", "fl_policy_gae",
           "fl_policy_linear", "fl_policy_linear_debug", "fl_policy_debug_clocks", "fl_policy_launch_count"]


class FlPolicyWeights(C.Structure):
    """Mirror of `struct FlPolicyWeights` (include/flatland_policy_b200.h)."""
    _fields_ = [(n, C.c_void_p) for n in ("tree_uiou", "tree_wiou", "tree_wc", "tree_ufwf", "tree_b_iou", "tree_b_c", "tree_b_f")] + \
               [("attr_w", C.c_void_p * 4), ("attr_b", C.c_void_p * 4),
                ("tf_wqkv", C.c_void_p * LAYERS), ("tf_bqkv", C.c_void_p * LAYERS), ("tf_wo", C.c_void_p * LAYERS),
                ("tf_bo", C.c_void_p * LAYERS), ("tf_wm", C.c_void_p * LAYERS), ("tf_bm", C.c_void_p * LAYERS)] + \
               [(n, C.c_void_p) for n in ("head_w1", "head_b1", "head_w2a", "head_w2c", "head_b2", "head_w3", "head_b3")]


class FlPpoParams(C.Structure):
    """Mirror of `struct FlPpoParams` (include/flatland_policy_b200.h)."""
    _fields_ = [("clip_eps", C.c_float), ("vf_coef", C.c_float), ("ent_coef", C.c_float)]


class FlPpoOptions(C.Structure):
    """Mirror of `struct FlPpoOptions` (include/flatland_policy_b200.h): clipped value loss and advantage normalisation."""
    _fields_ = [("vf_clip", C.c_float), ("norm_adv", C.c_int32), ("adv_eps", C.c_float)]


class FlTcProduct(C.Structure):
    """Mirror of `struct FlTcProduct` (include/flatland_policy_b200.h): one tensor-core product of the bf16 learner."""
    _fields_ = [("kind", C.c_int32), ("M", C.c_int64), ("N", C.c_int32), ("K", C.c_int32),
                ("x1", C.c_void_p), ("idx", C.c_void_p), ("ldx1", C.c_int64), ("K1", C.c_int32),
                ("x2", C.c_void_p), ("ldx2", C.c_int64), ("K2", C.c_int32),
                ("dy", C.c_void_p), ("lddy", C.c_int64),
                ("w", C.c_void_p), ("ldw", C.c_int64), ("bias", C.c_void_p),
                ("c", C.c_void_p), ("cidx", C.c_void_p), ("ldc", C.c_int64),
                ("add", C.c_void_p), ("ldadd", C.c_int64), ("accum", C.c_int32),
                ("pre", C.c_void_p), ("act", C.c_int32),
                ("gpre", C.c_void_p), ("ldgpre", C.c_int64),
                ("db", C.c_void_p)]


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FlatlandB200Error("CUDA library %s is not built (run `python __graft_entry__.py build`); "
                                "there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    P = C.c_void_p
    L.fl_policy_abi_version.restype = C.c_int
    L.fl_policy_launch_count.restype = C.c_uint64
    L.fl_policy_workspace_bytes.restype = C.c_size_t
    L.fl_policy_workspace_bytes.argtypes = [C.c_int64]
    L.fl_policy_forward.restype = C.c_int
    L.fl_policy_forward.argtypes = [C.POINTER(FlPolicyWeights), P, C.c_size_t, C.c_int64, C.c_int64, P, P, P, P, P, P, P]
    L.fl_policy_workspace_bytes_f32.restype = C.c_size_t
    L.fl_policy_workspace_bytes_f32.argtypes = [C.c_int64]
    L.fl_policy_forward_f32.restype = C.c_int
    L.fl_policy_forward_f32.argtypes = [P, P, C.c_size_t, C.c_int64, C.c_int64, P, P, P, P, P, P, P]
    L.fl_policy_workspace_bytes_grad_f32.restype = C.c_size_t
    L.fl_policy_workspace_bytes_grad_f32.argtypes = [C.c_int64]
    L.fl_policy_ppo_grad_f32.restype = C.c_int
    L.fl_policy_ppo_grad_f32.argtypes = [P, P, C.c_size_t, C.c_int64, C.c_int64] + [P] * 10 + [C.POINTER(FlPpoParams), P, P, P, P, P]
    L.fl_policy_workspace_bytes_grad_bf16.restype = C.c_size_t
    L.fl_policy_workspace_bytes_grad_bf16.argtypes = [C.c_int64]
    L.fl_policy_ppo_grad_bf16.restype = C.c_int
    L.fl_policy_ppo_grad_bf16.argtypes = [P, P, C.c_size_t, C.c_int64, C.c_int64] + [P] * 10 + [C.POINTER(FlPpoParams), P, P, P, P, P]
    L.fl_policy_forward_train_bf16.restype = C.c_int
    L.fl_policy_forward_train_bf16.argtypes = [P, P, C.c_size_t, C.c_int64, C.c_int64, P, P, P, P, P, P, P]
    L.fl_policy_ppo_counts.restype = C.c_int
    L.fl_policy_ppo_counts.argtypes = [C.c_int64, C.c_int64, P, P, P, P]
    for name in ("fl_policy_ppo_grad_shard_f32", "fl_policy_ppo_grad_shard_bf16"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = [P, P, C.c_size_t, C.c_int64, C.c_int64] + [P] * 11 + [C.POINTER(FlPpoParams), P, P, P, P, P]
    L.fl_policy_ppo_moments.restype = C.c_int
    L.fl_policy_ppo_moments.argtypes = [C.c_int64, C.c_int64, P, P, P, P, P]
    for name in ("fl_policy_ppo_grad_ex_f32", "fl_policy_ppo_grad_ex_bf16"):
        getattr(L, name).restype = C.c_int
        getattr(L, name).argtypes = [P, P, C.c_size_t, C.c_int64, C.c_int64] + [P] * 11 + [C.POINTER(FlPpoParams), P, P, P, P, P] + \
            [P, P, C.POINTER(FlPpoOptions)]
    L.fl_policy_tc_product_bf16.restype = C.c_int
    L.fl_policy_tc_product_bf16.argtypes = [C.POINTER(FlTcProduct), P, C.c_size_t, P]
    L.fl_policy_choose_actions.restype = C.c_int
    L.fl_policy_choose_actions.argtypes = [P, P, P, C.c_int64, P]
    L.fl_policy_sample_actions.restype = C.c_int
    L.fl_policy_sample_actions.argtypes = [P, P, C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.c_uint64, P, P, P]
    L.fl_policy_gae.restype = C.c_int
    L.fl_policy_gae.argtypes = [P, P, P, P, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_float, P, P, P]
    L.fl_policy_linear.restype = C.c_int
    L.fl_policy_linear.argtypes = [P, C.c_int64, P, P, P, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, P]
    L.fl_policy_debug_clocks.restype = None
    L.fl_policy_debug_clocks.argtypes = [P]
    L.fl_policy_linear_debug.restype = C.c_int
    L.fl_policy_linear_debug.argtypes = [P, C.c_int64, P, P, P, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, P, P]
    _lib = L
    return L


def _check(rc, what):
    if rc != 0:
        raise FlatlandB200Error("%s failed (code %d: %s)" % (what, rc, "bad argument" if rc < 0 else "CUDA error"))


def pack_weights(w):
    """Reference state_dict (numpy float32) -> {field: numpy array} in the layouts of FlPolicyWeights
    (matrices float32 here, cast to bf16 on upload; `in` dimension zero-padded)."""
    pw.check_weights(w)

    def pad_in(m, k):
        out = np.zeros((m.shape[0], k), np.float32)
        out[:, : m.shape[1]] = m
        return out

    # Tree-LSTM: biases become column 12 of the node-feature weights (the kernels feed a constant 1 there), and the
    # sigmoid gates' rows are halved: sigmoid(2z) = 0.5 tanh(z) + 0.5 (see include/flatland_policy_b200.h)
    wiou = pad_in(w["tree_lstm.W_iou.weight"], 16)
    wiou[:, 12] = w["tree_lstm.W_iou.bias"]
    uiou = w["tree_lstm.U_iou.weight"].copy()
    wiou[:256] *= 0.5
    uiou[:256] *= 0.5
    wf = pad_in(w["tree_lstm.W_f.weight"], 16)
    wf[:, 12] = w["tree_lstm.W_f.bias"]
    d = {
        "tree_uiou": uiou, "tree_wiou": wiou,
        "tree_wc": w["tree_lstm.W_c.weight"],
        "tree_ufwf": 0.5 * np.concatenate([w["tree_lstm.U_f.weight"], wf], axis=1),
        "tree_b_iou": w["tree_lstm.W_iou.bias"], "tree_b_c": w["tree_lstm.W_c.bias"], "tree_b_f": w["tree_lstm.W_f.bias"],
        "head_w1": np.concatenate([w["actor_net.0.weight"], w["critic_net.0.weight"]], axis=0),
        "head_b1": np.concatenate([w["actor_net.0.bias"], w["critic_net.0.bias"]]),
        "head_w2a": w["actor_net.2.weight"], "head_w2c": w["critic_net.2.weight"],
        "head_b2": np.concatenate([w["actor_net.2.bias"], w["critic_net.2.bias"]]),
        "head_w3": np.concatenate([w["actor_net.4.weight"], w["critic_net.4.weight"]], axis=0),
        "head_b3": np.concatenate([w["actor_net.4.bias"], w["critic_net.4.bias"]]),
    }
    for i in range(4):
        m = w["attr_embedding.%d.weight" % (2 * i)]
        d["attr_w%d" % i] = pad_in(m, 128) if i == 0 else m
        d["attr_b%d" % i] = w["attr_embedding.%d.bias" % (2 * i)]
    for l in range(LAYERS):
        p = "transformer.%d." % l
        d["tf_wqkv%d" % l], d["tf_bqkv%d" % l] = w[p + "attention.in_proj_weight"], w[p + "attention.in_proj_bias"]
        wo, bo = w[p + "attention.out_proj.weight"].astype(np.float64), w[p + "attention.out_proj.bias"].astype(np.float64)
        wm, bm = w[p + "att_mlp.0.weight"].astype(np.float64), w[p + "att_mlp.0.bias"].astype(np.float64)
        d["tf_wo%d" % l], d["tf_bo%d" % l] = wo, bo
        # Transformer.forward (net_tree.py:20-32) applies att_mlp to cat(input, out_proj(heads)) with nothing in between:
        # cat(x, a Wo^T + bo) [W1 | W2]^T = x W1^T + a (W2 Wo)^T + (bm + W2 bo) — the out-projection is folded into the
        # second half of att_mlp's weights here, in float64, and the kernels run one layer instead of two
        e = wo.shape[0]
        d["tf_wm%d" % l] = np.concatenate([wm[:, :e], wm[:, e:] @ wo], axis=1)
        d["tf_bm%d" % l] = bm + wm[:, e:] @ bo
    return {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in d.items()}


def weights_dict(weights, seed=0):
    """A weight source -> reference state_dict as numpy float32: a checkpoint path (.pt state_dict or .npz), a state_dict-like
    dict of arrays or tensors, or None for `init_weights(seed)`."""
    if weights is None:
        return pw.init_weights(seed)
    if isinstance(weights, (str, os.PathLike)):
        return pw.load_weights(weights)
    return {k: (v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)).astype(np.float32) for k, v in weights.items()}


_FP32_FIELDS = ("head_w3",)


class BatchedActor:
    """`Actor(model_path)` of the reference for E environments x N agents.

    weights: a reference checkpoint path (.pt state_dict or .npz), a state_dict-like dict of arrays, or None for
    `init_weights(seed)`."""

    def __init__(self, weights=None, device="cuda:0", seed=0, precision="bf16"):
        """precision: "bf16" — bf16 operands, fp32 accumulation on the tensor cores (the fast path; logits within about 1e-2
        of the reference network); "fp32" — the reference's own arithmetic on the CUDA cores (fl_policy_forward_f32: logits
        within summation-order rounding of the reference, about ten times slower)."""
        if precision not in ("bf16", "fp32"):
            raise ValueError("precision must be 'bf16' or 'fp32'")
        self.precision = precision
        if not torch.cuda.is_available():
            raise FlatlandB200Error("BatchedActor needs a CUDA device (no CPU fallback on the policy path)")
        self.lib = lib()
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        self.weights = weights = weights_dict(weights, seed)
        packed = pack_weights(weights)
        self.t = {}
        for k, v in packed.items():
            is_matrix = v.ndim == 2 and k not in _FP32_FIELDS
            tt = torch.from_numpy(v).to(self.device)
            self.t[k] = tt.to(torch.bfloat16).contiguous() if is_matrix else tt.contiguous()
        s = self.struct = FlPolicyWeights()
        for name, _ in FlPolicyWeights._fields_:
            if name in ("attr_w", "attr_b"):
                for i in range(4):
                    getattr(s, name)[i] = self.t["%s%d" % (name, i)].data_ptr()
            elif name.startswith("tf_"):
                for l in range(LAYERS):
                    getattr(s, name)[l] = self.t["%s%d" % (name, l)].data_ptr()
            else:
                setattr(s, name, self.t[name].data_ptr())
        # fp32 path: the reference state_dict as it is, in registration order
        self._f32 = None
        if precision == "fp32":
            tens = [torch.from_numpy(np.ascontiguousarray(weights[name], dtype=np.float32)).to(self.device) for name, _, _ in pw.weight_spec()]
            ptrs = (C.c_void_p * len(tens))(*[t.data_ptr() for t in tens])
            self._f32 = (tens, ptrs)
        self._ws = None
        self._out = None
        self._sampled = None

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _buffers(self, E, N):
        need = int((self.lib.fl_policy_workspace_bytes_f32 if self.precision == "fp32" else self.lib.fl_policy_workspace_bytes)(E * N))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        if self._out is None or self._out[0].shape[:2] != (E, N):
            self._out = (torch.empty((E, N, 5), dtype=torch.float32, device=self.device),
                         torch.empty((E,), dtype=torch.float32, device=self.device),
                         torch.empty((E, N), dtype=torch.uint8, device=self.device))
        return self._ws, self._out

    def forward(self, obs):
        """Network.forward (net_tree.py:73-98) on device tensors agent_attr [E,N,83] f32, forest [E,N,31,12] f32
        (+inf allowed: replaced by -1 as eval_env.py:76 does), adjacency [E,N,30,3] i32, node_order [E,N,31] i32.
        Returns (logits [E,N,5] f32, value [E] f32), valid until the next call."""
        a, f, adj, no = obs["agent_attr"], obs["forest"], obs["adjacency"], obs["node_order"]
        for name, tns, dt in (("agent_attr", a, torch.float32), ("forest", f, torch.float32), ("adjacency", adj, torch.int32),
                              ("node_order", no, torch.int32)):
            if tns.device != self.device or tns.dtype != dt or not tns.is_contiguous():
                raise ValueError("%s must be a contiguous %s tensor on %s" % (name, dt, self.device))
        E, N = int(a.shape[0]), int(a.shape[1])
        ws, (logits, value, _) = self._buffers(E, N)
        if self.precision == "fp32":
            _check(self.lib.fl_policy_forward_f32(self._f32[1], ws.data_ptr(), ws.numel(), E, N, a.data_ptr(), f.data_ptr(),
                                                  adj.data_ptr(), no.data_ptr(), logits.data_ptr(), value.data_ptr(), self._stream()),
                   "fl_policy_forward_f32")
            return logits, value
        _check(self.lib.fl_policy_forward(C.byref(self.struct), ws.data_ptr(), ws.numel(), E, N, a.data_ptr(), f.data_ptr(),
                                          adj.data_ptr(), no.data_ptr(), logits.data_ptr(), value.data_ptr(), self._stream()),
               "fl_policy_forward")
        return logits, value

    def choose_actions(self, logits, valid_actions):
        """Actor._choose_action, soft mode (plfActor.py:27-44), for every agent: uint8 [E,N] device tensor."""
        E, N = int(logits.shape[0]), int(logits.shape[1])
        _, (_, _, actions) = self._buffers(E, N)
        va = self._valid_u8(valid_actions)
        _check(self.lib.fl_policy_choose_actions(logits.data_ptr(), va.data_ptr(), actions.data_ptr(), E * N, self._stream()),
               "fl_policy_choose_actions")
        return actions

    def _valid_u8(self, valid_actions):
        va = valid_actions.to(torch.uint8) if valid_actions.dtype == torch.bool else valid_actions
        if va.device != self.device or va.dtype != torch.uint8 or not va.is_contiguous():
            raise ValueError("valid_actions must be a contiguous uint8/bool tensor on %s" % self.device)
        return va

    def sample_actions(self, logits, valid_actions, seed, step, env_offset=0):
        """Exploration for PPO rollouts (fl_policy_sample_actions): the soft choice of choose_actions with a seeded uniform
        per agent, drawn from Philox4x32-10 at counter (step, env_offset + e, agent) and key `seed`, so that the draw of an
        agent depends only on (seed, step, global environment id, agent).  A shard of a multi-GPU sweep passes env_offset =
        its first global environment id (shard_range).  Returns (actions uint8 [E,N], log_probs float32 [E,N]): the chosen
        actions and their log-probabilities under the masked softmax of `logits` (log pi_old of the PPO ratio), device
        tensors reused by the next call."""
        E, N = int(logits.shape[0]), int(logits.shape[1])
        if self._sampled is None or self._sampled[0].shape != (E, N):
            self._sampled = (torch.empty((E, N), dtype=torch.uint8, device=self.device),
                             torch.empty((E, N), dtype=torch.float32, device=self.device))
        self._sample_into(logits, valid_actions, seed, step, env_offset, *self._sampled)
        return self._sampled

    def _sample_into(self, logits, valid_actions, seed, step, env_offset, actions, log_probs):
        if logits.device != self.device or logits.dtype != torch.float32 or not logits.is_contiguous() or logits.shape[2:] != (5,):
            raise ValueError("logits must be a contiguous float32 [E,N,5] tensor on %s" % self.device)
        va = self._valid_u8(valid_actions)
        E, N = int(logits.shape[0]), int(logits.shape[1])
        if tuple(va.shape) != (E, N, 5):
            raise ValueError("valid_actions must be [E,N,5] like logits")
        _check(self.lib.fl_policy_sample_actions(logits.data_ptr(), va.data_ptr(), E, N, int(env_offset), int(seed) & (2 ** 64 - 1),
                                                 int(step) & (2 ** 64 - 1), actions.data_ptr(), log_probs.data_ptr(), self._stream()),
               "fl_policy_sample_actions")

    def get_actions(self, obs, valid_actions=None):
        """Actor.get_actions (plfActor.py:15-25) for the whole batch: observation dict -> actions uint8 [E,N]
        (device tensor that `BatchedRailEnv.step` takes as is)."""
        logits, _ = self.forward(obs)
        return self.choose_actions(logits, obs["valid_actions"] if valid_actions is None else valid_actions)

    def linear(self, a, w, bias, act=0, out=None):
        """One dense layer on the tensor-core path (tests): a [M,K] bf16, w [N,K] bf16, bias [N] f32."""
        M, K = a.shape
        Nn = w.shape[0]
        if out is None:
            out = torch.empty((M, Nn), dtype=torch.bfloat16, device=self.device)
        _check(self.lib.fl_policy_linear(a.data_ptr(), a.stride(0), w.data_ptr(), bias.data_ptr(), out.data_ptr(), out.stride(0),
                                         M, Nn, K, int(act), self._stream()), "fl_policy_linear")
        return out

    def launch_count(self):
        return int(self.lib.fl_policy_launch_count())
