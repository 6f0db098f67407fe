"""The arithmetic contract of fl_policy_ppo_grad_bf16 (include/flatland_policy_b200.h) restated in float64 torch — TEST
INFRASTRUCTURE ONLY.  tests/policy_grad_oracle.py with one change: the 20 tensor-core layers go through TcLinear, whose
forward X W^T, input gradient dY W and weight gradient dY^T X multiply operands rounded to bf16 (from their fp32 value, round
to nearest even, as the kernels round the fp32 activations they stage) and accumulate in float64; the bias gradient is the
sum of the unrounded dY.  Everything else is the float64 restatement as it stands."""
import contextlib

import numpy as np
import torch

import policy_grad_oracle as pgo

# weights whose products run on the tensor cores (their biases are added in fp32)
TC_WEIGHTS = (["tree_lstm.U_iou.weight", "tree_lstm.U_f.weight", "tree_lstm.W_c.weight"] +
              ["attr_embedding.%d.weight" % i for i in (0, 2, 4, 6)] +
              ["transformer.%d.%s" % (l, n) for l in range(3)
               for n in ("attention.in_proj_weight", "attention.out_proj.weight", "att_mlp.0.weight")] +
              ["%s.%d.weight" % (h, i) for h in ("actor_net", "critic_net") for i in (0, 2)])


def bf16(t):
    """float64 -> fp32 -> bf16 (round to nearest even) -> float64."""
    return t.to(torch.float32).to(torch.bfloat16).to(t.dtype)


class TcLinear(torch.autograd.Function):
    """y = r(x) r(w)^T + b; dx = r(dy) r(w); dw = r(dy)^T r(x); db = sum of dy; r = bf16 when `rounding`, else the identity.
    With rounding off, every product is the one autograd computes for policy_grad_oracle.linear (same operands, same
    layouts), so the results are bit-identical to it."""

    @staticmethod
    def forward(ctx, x, w, b, rounding):
        ctx.save_for_backward(x, w)
        ctx.rounding = rounding
        ctx.has_bias = b is not None
        r = bf16 if rounding else (lambda t: t)
        y = r(x) @ r(w).t()
        return y + b if b is not None else y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        r = bf16 if ctx.rounding else (lambda t: t)
        dx = r(dy).mm(r(w)) if ctx.needs_input_grad[0] else None
        dw = r(dy).t().mm(r(x)) if ctx.needs_input_grad[1] else None
        db = dy.sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dw, db, None


@contextlib.contextmanager
def tensor_core_layers(p, rounding=True):
    """While active, policy_grad_oracle's network sends the TC_WEIGHTS of parameter dict p through TcLinear."""
    tc = {id(p[n]) for n in TC_WEIGHTS}
    plain = pgo.linear

    def linear(x, w, b=None):
        return TcLinear.apply(x, w, b, rounding) if id(w) in tc else plain(x, w, b)

    pgo.linear = linear
    try:
        yield
    finally:
        pgo.linear = plain


def loss_and_grads(w, obs, mb, clip_eps=0.2, vf_coef=0.5, ent_coef=0.01, rounding=True, dtype=torch.float64):
    """policy_grad_oracle.loss_and_grads under the bf16 learner's contract (rounding=False: the float64 restatement).
    dtype=torch.float32 evaluates the same contract in fp32: where it and the float64 evaluation disagree, the case is
    sensitive to which side of a bf16 rounding boundary an activation falls on, whatever computes it."""
    p = pgo.params(w, dtype=dtype)
    with tensor_core_layers(p, rounding):
        logits, value = pgo.forward(p, obs["agent_attr"], obs["forest"], obs["adjacency"], obs["node_order"], obs["edge_order"])
        L, stats = pgo.ppo_loss(logits, value, obs["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"],
                                mb["returns"], mb["acted"], clip_eps, vf_coef, ent_coef)
        L.backward()
    grads = {k: (v.grad.double().numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in p.items()}
    return float(L.detach()), stats, logits.detach().double().numpy(), value.detach().double().numpy(), grads
