"""The PPO loss with its options (FlPpoOptions, include/flatland_policy_b200.h: clipped value loss and advantage normalisation
over the whole minibatch) restated in float64 torch — TEST INFRASTRUCTURE ONLY.  It calls the forwards and the loss of
tests/policy_grad_oracle.py (and, for the bf16 learner, the tensor-core layers of tests/policy_grad_oracle_bf16.py) and
changes only what the options change: the advantages the policy term sees and the value term."""
import numpy as np
import torch

import policy_grad_oracle as pgo
import policy_grad_oracle_bf16 as pgb


def agent_set(valid, acted):
    """S as a bool [E, N] array: agents of acted rows with at least one valid action."""
    return (np.asarray(valid) != 0).any(-1) & (np.asarray(acted) != 0)[:, None]


def moments(valid, acted, advantages):
    """[sum_S A, sum_S A^2] in float64, each row's A once per agent of S (fl_policy_ppo_moments)."""
    n = agent_set(valid, acted).sum(-1).astype(np.float64)
    a = np.asarray(advantages, np.float32).astype(np.float64)
    return np.array([(n * a).sum(), (n * (a * a)).sum()])


def normalised_advantages(advantages, n_s, mom, adv_eps):
    """A_hat of every row from the minibatch's |S| and moments: (A - mu) / (sigma + adv_eps) formed in float64 and rounded once
    to fp32 (returned as float64); 0 where sigma + adv_eps = 0."""
    a = np.asarray(advantages, np.float32).astype(np.float64)
    n, s, q = float(n_s), float(mom[0]), float(mom[1])
    mu = s / n if n_s > 0 else 0.0
    var = max(0.0, (q - s * s / n) / (n - 1.0)) if n_s > 1 else 0.0
    den = np.sqrt(var) + float(np.float32(adv_eps))
    if not den > 0:
        return np.zeros_like(a)
    return ((a - mu) / den).astype(np.float32).astype(np.float64)


def ppo_loss_ex(logits, value, valid, actions, old_log_probs, advantages, returns, acted, clip_eps, vf_coef, ent_coef,
                vf_clip=0.0, norm_adv=False, adv_eps=1e-8, old_values=None, n_s=None, mom=None):
    """The loss with the options, and its 8 statistics (numpy float64).  n_s, mom: |S| and the moments of the whole
    minibatch (default: these rows').  With both options off this is policy_grad_oracle.ppo_loss, bit for bit."""
    if not norm_adv and not vf_clip > 0:
        return pgo.ppo_loss(logits, value, valid, actions, old_log_probs, advantages, returns, acted, clip_eps, vf_coef,
                            ent_coef)
    if norm_adv:
        n_s = int(agent_set(valid, acted).sum()) if n_s is None else n_s
        mom = moments(valid, acted, advantages) if mom is None else mom
        advantages = normalised_advantages(advantages, n_s, mom, adv_eps)
    # the policy term and its statistics with A_hat; the value term added below (0 * L_val + vf_coef * L_val' leaves the
    # order of the additions of policy_grad_oracle.ppo_loss: (L_pol - ent L_ent) + vf L_val)
    L0, stats = pgo.ppo_loss(logits, value, valid, actions, old_log_probs, advantages, returns, acted, clip_eps, 0.0, ent_coef)
    dt, dv = logits.dtype, logits.device
    act = torch.as_tensor(np.asarray(acted) != 0, device=dv)
    R = torch.as_tensor(np.asarray(returns, np.float64), dtype=dt, device=dv)
    u = (value - R) ** 2
    if vf_clip > 0:
        Vo = torch.as_tensor(np.asarray(old_values, np.float64), dtype=dt, device=dv)
        Vc = Vo + torch.clamp(value - Vo, -float(np.float32(vf_clip)), float(np.float32(vf_clip)))
        uc = (Vc - R) ** 2
        u = torch.where(u >= uc, u, uc)             # ties take the unclipped square (torch.max would split the gradient)
    nR = int(act.sum())
    L_val = torch.where(act, u, torch.zeros_like(u)).sum() / nR if nR else torch.zeros((), dtype=dt, device=dv)
    L = L0 + vf_coef * L_val
    stats = stats.copy()
    stats[1], stats[7] = float(L_val.detach()), float(L.detach())
    return L, stats


def loss_and_grads(w, obs, mb, clip_eps=0.2, vf_coef=0.5, ent_coef=0.01, vf_clip=0.0, norm_adv=False, adv_eps=1e-8,
                   precision="fp32", dtype=torch.float64, n_s=None, mom=None):
    """policy_grad_oracle.loss_and_grads with the options (mb["values"]: V_old).  precision="bf16" evaluates the bf16 learner's
    contract (policy_grad_oracle_bf16's tensor-core layers); dtype=torch.float32 the same contract in fp32."""
    import contextlib
    p = pgo.params(w, dtype=dtype)
    ctx = pgb.tensor_core_layers(p) if precision == "bf16" else contextlib.nullcontext()
    with ctx:
        logits, value = pgo.forward(p, obs["agent_attr"], obs["forest"], obs["adjacency"], obs["node_order"], obs["edge_order"])
        L, stats = ppo_loss_ex(logits, value, obs["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"],
                               mb["returns"], mb["acted"], clip_eps, vf_coef, ent_coef, vf_clip, norm_adv, adv_eps,
                               mb.get("values"), n_s, mom)
        L.backward()
    grads = {k: (v.grad.double().numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in p.items()}
    return float(L.detach()), stats, logits.detach().double().numpy(), value.detach().double().numpy(), grads
