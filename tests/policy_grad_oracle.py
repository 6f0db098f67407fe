"""Float64 torch restatement of the reference network (oracle/policy_oracle.forward) and of the PPO loss of
fl_policy_ppo_grad_f32 (include/flatland_policy_b200.h) — TEST INFRASTRUCTURE ONLY.  Autograd through it is the yardstick of
the library's gradients: tests/test_policy_grad.py pins its forward to policy_oracle.forward, tests/test_gpu_policy_grad.py
compares the CUDA gradients with its own."""
import numpy as np
import torch
import torch.nn.functional as F

from flatland_marl_b200 import policy_weights as pw

D = torch.float64


def params(w, requires_grad=True, dtype=D, device="cpu"):
    """Reference state_dict (numpy) -> {name: leaf tensor} in weight_spec order (float64 on the CPU unless asked otherwise;
    tools/learner_bench.py runs the restatement in fp32 on the GPU as the autograd yardstick)."""
    return {name: torch.tensor(np.asarray(w[name], np.float64), dtype=dtype, device=device, requires_grad=requires_grad)
            for name, _, _ in pw.weight_spec()}


def linear(x, w, b=None):
    y = x @ w.t()
    return y + b if b is not None else y


def tree_lstm(p, forest, adjacency, node_order, edge_order):
    """policy_oracle.tree_lstm in torch: forest [B,N,31,12] tensor (cleaned), index arrays as numpy."""
    B, N, M, nf = forest.shape
    adj = np.asarray(adjacency, np.int64).copy()
    tree_id = np.arange(B * N, dtype=np.int64).reshape(B, N, 1)
    adj[adj == -2] = -B * N * M
    adj[..., 0] += tree_id * M
    adj[..., 1] += tree_id * M
    adj[adj < 0] = -2
    adj = adj.reshape(-1, 3)
    no = np.asarray(node_order).reshape(-1)
    eo = np.asarray(edge_order).reshape(-1)
    x_all = forest.reshape(-1, nf)
    T = p["tree_lstm.U_f.weight"].shape[0]
    h = torch.zeros((x_all.shape[0], T), dtype=x_all.dtype, device=x_all.device)
    c = torch.zeros_like(h)
    for it in range(int(no.max()) + 1):
        nm = torch.from_numpy(np.nonzero(no == it)[0]).to(x_all.device)
        x = x_all[nm]
        iou = linear(x, p["tree_lstm.W_iou.weight"], p["tree_lstm.W_iou.bias"])
        if it > 0:
            a = adj[eo == it]
            par, chi = torch.from_numpy(a[:, 0]).to(x_all.device), torch.from_numpy(a[:, 1]).to(x_all.device)
            ch, cc = h[chi], c[chi]
            iou = iou + linear(ch.reshape(ch.shape[0] // 3, 3 * T), p["tree_lstm.U_iou.weight"])
        i, o, u = torch.sigmoid(iou[:, :T]), torch.sigmoid(iou[:, T:2 * T]), torch.tanh(iou[:, 2 * T:])
        cn = i * u
        if it > 0:
            f = torch.sigmoid(linear(x_all[par], p["tree_lstm.W_f.weight"], p["tree_lstm.W_f.bias"]) + linear(ch, p["tree_lstm.U_f.weight"]))
            cn = cn + linear((f * cc).reshape(ch.shape[0] // 3, 3 * T), p["tree_lstm.W_c.weight"], p["tree_lstm.W_c.bias"])
        c = c.index_put((nm,), cn)
        h = h.index_put((nm,), o * torch.tanh(cn))
    return h


def attention_block(p, pre, x, heads=4):
    B, N, E = x.shape
    d = E // heads
    qkv = linear(x.reshape(B * N, E), p[pre + "attention.in_proj_weight"], p[pre + "attention.in_proj_bias"]).reshape(B, N, 3, heads, d)
    q = qkv[:, :, 0].transpose(1, 2) / np.sqrt(d)
    k = qkv[:, :, 1].transpose(1, 2)
    v = qkv[:, :, 2].transpose(1, 2)
    a = torch.softmax(q @ k.transpose(-1, -2), dim=-1)
    o = (a @ v).transpose(1, 2).reshape(B * N, E)
    o = linear(o, p[pre + "attention.out_proj.weight"], p[pre + "attention.out_proj.bias"])
    y = linear(torch.cat([x.reshape(B * N, E), o], dim=1), p[pre + "att_mlp.0.weight"], p[pre + "att_mlp.0.bias"])
    return F.gelu(y).reshape(B, N, E)


def forward(p, agent_attr, forest, adjacency, node_order, edge_order):
    """policy_oracle.forward: agent_attr [B,N,83], forest [B,N,31,12] (+inf allowed: cleaned here), index arrays numpy.
    Returns (logits [B,N,5], value [B]) tensors of the parameters' dtype and device."""
    dt, dv = p["tree_lstm.U_f.weight"].dtype, p["tree_lstm.U_f.weight"].device
    f = np.array(forest, np.float64, copy=True)
    f[f == np.inf] = -1
    forest = torch.as_tensor(f, dtype=dt, device=dv)
    B, N, M, _ = forest.shape
    h = tree_lstm(p, forest, adjacency, node_order, edge_order)
    tree_emb = h.reshape(B, N, M, -1)[:, :, 0, :]
    a = torch.as_tensor(np.asarray(agent_attr, np.float64), dtype=dt, device=dv).reshape(B * N, -1)
    for i in range(4):
        a = F.gelu(linear(a, p["attr_embedding.%d.weight" % (2 * i)], p["attr_embedding.%d.bias" % (2 * i)]))
    emb = torch.cat([a.reshape(B, N, -1), tree_emb], dim=2)
    att = emb
    for l in range(3):
        att = attention_block(p, "transformer.%d." % l, att)
    z = torch.cat([emb, att], dim=-1).reshape(B * N, -1)

    def head(name):
        y = F.gelu(linear(z, p[name + ".0.weight"], p[name + ".0.bias"]))
        y = F.gelu(linear(y, p[name + ".2.weight"], p[name + ".2.bias"]))
        return linear(y, p[name + ".4.weight"], p[name + ".4.bias"])

    return head("actor_net").reshape(B, N, -1), head("critic_net").reshape(B, N).mean(dim=1)


def log_probs(logits, valid, actions):
    """Masked log-softmax of the taken action; 0 for agents with no valid action."""
    valid = torch.as_tensor(np.asarray(valid) != 0, device=logits.device)
    xm = torch.where(valid, logits, torch.full_like(logits, -1e30))
    logp = xm - torch.logsumexp(xm, dim=-1, keepdim=True)
    lp = logp.gather(-1, torch.as_tensor(np.asarray(actions, np.int64), device=logits.device)[..., None])[..., 0]
    return torch.where(valid.any(-1), lp, torch.zeros_like(lp)), logp, valid


def ppo_loss(logits, value, valid, actions, old_log_probs, advantages, returns, acted, clip_eps, vf_coef, ent_coef):
    """The loss of fl_policy_ppo_grad_f32 (header comment) and its 8 statistics (numpy float64), in the logits' dtype."""
    lp, logp, valid = log_probs(logits, valid, actions)
    dt, dv = logits.dtype, logits.device
    acted = torch.as_tensor(np.asarray(acted) != 0, device=dv)
    S = valid.any(-1) & acted[:, None]
    old = torch.as_tensor(np.asarray(old_log_probs, np.float64), dtype=dt, device=dv)
    A = torch.as_tensor(np.asarray(advantages, np.float64), dtype=dt, device=dv)[:, None]
    R = torch.as_tensor(np.asarray(returns, np.float64), dtype=dt, device=dv)
    r = torch.exp(lp - old)
    s1, s2 = r * A, torch.clamp(r, 1 - clip_eps, 1 + clip_eps) * A
    pol = -torch.where(s1 <= s2, s1, s2)                 # the gradient flows through r A on ties
    p = torch.where(valid, logp.exp(), torch.zeros_like(logp))
    H = -torch.where(valid, p * logp, torch.zeros_like(logp)).sum(-1)
    nS, nR = int(S.sum()), int(acted.sum())
    zero = torch.zeros((), dtype=dt, device=dv)

    def mean_S(t):
        return torch.where(S, t, torch.zeros_like(t)).sum() / nS if nS else zero
    L_pol, L_ent = mean_S(pol), mean_S(H)
    L_val = torch.where(acted, (value - R) ** 2, torch.zeros_like(value)).sum() / nR if nR else zero
    L = L_pol - ent_coef * L_ent + vf_coef * L_val
    stats = [L_pol, L_val, L_ent, mean_S(old - lp), mean_S(((r - 1).abs() > clip_eps).to(dt)), nS, nR, L]
    return L, np.array([float(s.detach()) if torch.is_tensor(s) else float(s) for s in stats])


def loss_and_grads(w, obs, mb, clip_eps=0.2, vf_coef=0.5, ent_coef=0.01):
    """Float64 loss, stats, logits, values and {name: gradient} for reference weights w (numpy) on a minibatch of numpy arrays
    (obs keys as Rollout.minibatch, plus edge_order)."""
    p = params(w)
    logits, value = forward(p, obs["agent_attr"], obs["forest"], obs["adjacency"], obs["node_order"], obs["edge_order"])
    L, stats = ppo_loss(logits, value, obs["valid_actions"], mb["actions"], mb["log_probs"], mb["advantages"], mb["returns"],
                        mb["acted"], clip_eps, vf_coef, ent_coef)
    L.backward()
    grads = {k: (v.grad.numpy() if v.grad is not None else np.zeros(v.shape)) for k, v in p.items()}
    return float(L.detach()), stats, logits.detach().numpy(), value.detach().numpy(), grads
