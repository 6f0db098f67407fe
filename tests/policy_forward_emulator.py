"""The arithmetic of fl_policy_forward (the bf16 tensor-core forward, policy.cu) restated in float64 torch — TEST
INFRASTRUCTURE ONLY.

One function per kernel.  Each takes its inputs as the kernel reads them (bf16 values held in float64, packed weights
exactly as `BatchedActor.t` uploads them: halved sigmoid-gate rows, the Tree-LSTM biases in column 12 / 140 of the node
weights, the folded att_mlp `[W1 | W2 Wo]`, fp32 `head_w3`) and returns the value before the kernel's final bf16 store.
Products accumulate in float64; the kernels accumulate the same bf16 operands in fp32 on the tensor cores, so the two
differ by summation order and by the kernels' approximate tanh (tanh.approx, about 2^-11 relative).

`exact=True` switches to the reference arithmetic: no bf16 rounding anywhere, the erf form of GELU and exact tanh
(the halved gates make 0.5 tanh(z) + 0.5 exactly sigmoid(2z)).  With fp32 packed weights, `forward(..., exact=True)` is
oracle/policy_oracle.forward in float64, which pins every function here to the reference network.

`random_trees` generates valid observation trees in fl_observe's numbering (observe.cuh): 31 slots filled breadth-first,
the children of a node are three consecutive nodes, adjacency row n-1 = (parent, n, ad), node_order = height above the
leaves (-2 for unused slots), edge_order[n-1] = node_order[parent]."""
import math

import numpy as np
import torch

NODES = 32            # node slots per tree in the kernels' scratch (31 used)
NULL_COPIES = 1024    # copies of the shared null-node row (policy.cu)
MAX_LEVELS = 11
# the kernels' GELU: 0.5 x (1 + tanh(x P(x^2))), x^2 clamped at 49 (csrc/policy/umma.cuh, test_gelu_fit_used_by_the_kernels)
GELU_P = (7.97507884e-1, 3.70056460e-2, -3.51516783e-4)


def bf16(t):
    """float64 -> fp32 -> bf16 (round to nearest even) -> float64: the kernels' pack_bf16 of an fp32 value."""
    return t.to(torch.float32).to(torch.bfloat16).to(torch.float64)


def f32(t):
    return t.to(torch.float32).to(torch.float64)


def ulp(t):
    """One bf16 unit in the last place of |t| (the spacing of bf16 values at t; normal range)."""
    a = t.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


def _r(t, exact):
    return t if exact else bf16(t)


def gelu(x, exact=False):
    if exact:
        return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))
    x = f32(x)
    u = torch.clamp(x * x, max=49.0)
    p = GELU_P[0] + u * (GELU_P[1] + u * GELU_P[2])
    return 0.5 * x * (1.0 + torch.tanh(x * p))


def weights64(t, device=None):
    """Packed weights (BatchedActor.t or pack_weights' fp32 numpy dict) -> float64 torch tensors."""
    out = {}
    for k, v in t.items():
        v = torch.as_tensor(v) if not isinstance(v, torch.Tensor) else v
        out[k] = v.to(device=device if device is not None else v.device).to(torch.float64)
    return out


# ---- k_prep -------------------------------------------------------------------------------------------------------
def prep(agent_attr, forest, exact=False):
    """agent_attr [M,83], forest [M,31,12] (fp32, +inf allowed) -> (attr [M,128], x [M+1024,32,16], nullmask [M] int64).
    x: +inf -> -1, column 12 = 1 on real nodes, slot 31 zero; trees M.. carry the null-node features in node 1.
    nullmask bit v: non-root node v whose twelve features are all -1 (after +inf -> -1)."""
    attr = torch.as_tensor(agent_attr).to(torch.float64)
    fo = torch.as_tensor(forest).to(torch.float64)
    M = attr.shape[0]
    a = torch.zeros((M, 128), dtype=torch.float64, device=attr.device)
    a[:, :83] = _r(attr, exact)
    fo = torch.where(torch.isposinf(fo), torch.full_like(fo, -1.0), fo)
    x = torch.zeros((M + NULL_COPIES, NODES, 16), dtype=torch.float64, device=attr.device)
    x[:M, :31, :12] = _r(fo, exact)
    x[:M, :31, 12] = 1.0
    x[M:, 1, :12] = -1.0
    x[M:, 1, 12] = 1.0
    null = (fo == -1.0).all(-1)
    null[:, 0] = False
    bits = torch.tensor([1 << v for v in range(31)], dtype=torch.int64, device=attr.device)
    nullmask = (null.to(torch.int64) * bits).sum(-1)
    return a, x, nullmask


# ---- the Tree-LSTM kernels ------------------------------------------------------------------------------------------
def leaf(x, wiou, exact=False):
    """k_tree_leaf: x [R,16] (bias column 12 = 1), wiou [384,16] (rows 0..255 halved) -> (h, c) [R,128].
    c = 0.5 tu ti + 0.5 tu, h = 0.5 tc to + 0.5 tc, t* = tanh of the (halved) pre-activations, tc = tanh(c unrounded)."""
    iou = x @ wiou.t()
    ti, to, tu = torch.tanh(iou[:, :128]), torch.tanh(iou[:, 128:256]), torch.tanh(iou[:, 256:])
    c = 0.5 * tu * ti + 0.5 * tu
    tc = torch.tanh(c if exact else f32(c))
    return 0.5 * tc * to + 0.5 * tc, c


def forget(h_child, x_parent, c_child, ufwf):
    """k_lin<MODE_TREE_F>: one row per child: acc = [h_child | x_parent] ufwf^T (halved: b_f rides in column 140),
    fc = 0.5 c tanh(acc) + 0.5 c = sigmoid(f) c_child."""
    acc = torch.cat([h_child, x_parent], 1) @ ufwf.t()
    return 0.5 * c_child * torch.tanh(acc) + 0.5 * c_child


def parent(h3, x, fc3, uiou, wiou, wc, b_c, exact=False):
    """k_tree_p: h3 = [h0|h1|h2] [R,384] of the children, x [R,16], fc3 [R,384] -> (h, c) [R,128].
    iou = h3 U_iou^T + x W_iou^T; c = 0.5 tu ti + 0.5 tu + fc3 W_c^T + b_c; h from the unrounded c."""
    iou = h3 @ uiou.t() + x @ wiou.t()
    ti, to, tu = torch.tanh(iou[:, :128]), torch.tanh(iou[:, 128:256]), torch.tanh(iou[:, 256:])
    acc_c = fc3 @ wc.t()
    c = 0.5 * tu * ti + 0.5 * tu
    c = c + (acc_c + b_c if exact else f32(f32(acc_c) + b_c))
    tc = torch.tanh(c if exact else f32(c))
    return 0.5 * tc * to + 0.5 * tc, c


# ---- dense layers, attention, head ----------------------------------------------------------------------------------
def dense(srcs, w, b, act, exact=False):
    """k_lin<MODE_LINEAR>: [src0 | src1] w^T + b (fp32 bias), then the kernels' GELU when act (erf GELU when exact)."""
    a = torch.cat(srcs, 1) if len(srcs) > 1 else srcs[0]
    y = a @ w.t() + b
    return gelu(y, exact) if act else y


def attention(qkv, E, N, exact=False):
    """k_attn_mma: qkv [M,768] = q | k | v, 4 heads of 64; per (row, head) the keys of the row's own environment only.
    P = bf16(exp(S/8 - max)), den = the sum of the rounded P, O = sum P V / den.  Returns [M,256]."""
    q = qkv[:, :256].reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    k = qkv[:, 256:512].reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    v = qkv[:, 512:].reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    s = q @ k.transpose(-1, -2)
    s = s * 0.125 if exact else f32(f32(s) * 0.125)
    p = torch.exp(s - s.amax(-1, keepdim=True))
    if not exact:
        p = bf16(p)
    o = (p @ v) / p.sum(-1, keepdim=True)
    return o.permute(0, 2, 1, 3).reshape(E * N, 256)


def head_final(y2, w3, b3, E, N):
    """k_head_final: logits = y2[:, :128] w3[:5]^T + b3[:5]; value = mean over the N agents of y2[:, 128:] w3[5] + b3[5]."""
    logits = y2[:, :128] @ w3[:5].t() + b3[:5]
    crit = y2[:, 128:] @ w3[5] + b3[5]
    return logits.reshape(E, N, 5), crit.reshape(E, N).sum(1) / N


# ---- tree structure -----------------------------------------------------------------------------------------------
def levels(adjacency, node_order, nullmask):
    """The Tree-LSTM's schedule with the reference's child semantics.  Returns (leaves, inner, shared):
    leaves = (tree, node) index tensors of the computed leaves (node_order 0, not a null leaf);
    inner[L] = (tree, node, first child) of the nodes with node_order L >= 1;
    shared [M,31] bool = the null leaves, whose state is the shared null row (equal features give equal states)."""
    adj = torch.as_tensor(adjacency).to(torch.int64)
    no = torch.as_tensor(node_order).to(torch.int64)
    M = no.shape[0]
    dev = no.device
    bits = torch.tensor([1 << v for v in range(31)], dtype=torch.int64, device=dev)
    null = (nullmask.to(dev)[:, None] & bits) != 0
    shared = null & (no == 0)
    t_all = torch.arange(M, device=dev)[:, None].expand(M, 31)
    v_all = torch.arange(31, device=dev)[None, :].expand(M, 31)
    lm = (no == 0) & ~shared
    leaves = (t_all[lm], v_all[lm])
    child0 = torch.zeros((M, 31), dtype=torch.int64, device=dev)
    par = adj[:, 0::3, 0]                                         # parent of nodes 3g+1 .. 3g+3
    g = torch.arange(10, device=dev)[None, :].expand(M, 10)
    ok = (par >= 0) & (par < 31)
    child0[t_all[:, :10][ok], par[ok]] = 3 * g[ok] + 1
    inner = {}
    for L in range(1, MAX_LEVELS):
        m = no == L
        if bool(m.any()):
            inner[L] = (t_all[m], v_all[m], child0[m])
    return leaves, inner, shared


def forward(t, obs, exact=False, stages=None):
    """The whole forward on packed weights `t` (weights64) and observation tensors [E,N,...] -> (logits [E,N,5], value [E]).
    Every stage rounds its output as the kernel stores it (unless exact).  `stages`, a dict, receives the intermediate
    tensors under the names of the workspace buffers (x, h, c, fc, attr, a1/a2 as left by the last layers, emb, ...)."""
    a_in = torch.as_tensor(obs["agent_attr"])
    E, N = int(a_in.shape[0]), int(a_in.shape[1])
    M = E * N
    dev = t["tree_wiou"].device
    r = (lambda z: z) if exact else bf16
    attr, x, nm = prep(a_in.reshape(M, 83).to(dev), torch.as_tensor(obs["forest"]).reshape(M, 31, 12).to(dev), exact)
    leaves, inner, shared = levels(torch.as_tensor(obs["adjacency"]).reshape(M, 30, 3).to(dev),
                                   torch.as_tensor(obs["node_order"]).reshape(M, 31).to(dev), nm)
    h = torch.zeros((M, NODES, 128), dtype=torch.float64, device=dev)
    c = torch.zeros_like(h)
    fc = torch.zeros_like(h)
    nh, nc = leaf(x[M, 1][None], t["tree_wiou"], exact)
    nh, nc = r(nh[0]), r(nc[0])
    ti, vi = leaves
    hh, cc = leaf(x[ti, vi], t["tree_wiou"], exact)
    h[ti, vi], c[ti, vi] = r(hh), r(cc)

    def state(tt, ch, buf, nullrow):
        s = buf[tt, ch]
        sh = shared[tt, ch]
        return torch.where(sh[:, None], nullrow[None, :], s)

    for L in sorted(inner):
        tt, vv, c0 = inner[L]
        h3, fc3 = [], []
        for j in range(3):
            hj, cj = state(tt, c0 + j, h, nh), state(tt, c0 + j, c, nc)
            fj = r(forget(hj, x[tt, vv], cj, t["tree_ufwf"]))
            fc[tt, c0 + j] = fj
            h3.append(hj)
            fc3.append(fj)
        hp, cp = parent(torch.cat(h3, 1), x[tt, vv], torch.cat(fc3, 1), t["tree_uiou"], t["tree_wiou"], t["tree_wc"], t["tree_b_c"], exact)
        h[tt, vv], c[tt, vv] = r(hp), r(cp)
    no = torch.as_tensor(obs["node_order"]).reshape(M, 31).to(dev)
    emb = torch.zeros((M, 256), dtype=torch.float64, device=dev)
    emb[:, 128:] = torch.where((no[:, 0] >= 0)[:, None], h[:, 0], torch.zeros_like(h[:, 0]))
    a = attr
    outs = []
    for i in range(4):
        a = r(dense([a], t["attr_w%d" % i], t["attr_b%d" % i], True, exact))
        outs.append(a)
    emb[:, :128] = a
    tin = emb
    touts = []
    for l in range(3):
        qkv = r(dense([tin], t["tf_wqkv%d" % l], t["tf_bqkv%d" % l], False, exact))
        atto = r(attention(qkv, E, N, exact))
        tin = r(dense([tin, atto], t["tf_wm%d" % l], t["tf_bm%d" % l], True, exact))
        touts.append(tin)
    y1 = r(dense([emb, tin], t["head_w1"], t["head_b1"], True, exact))
    y2 = torch.cat([r(dense([y1[:, :256]], t["head_w2a"], t["head_b2"][:128], True, exact)),
                    r(dense([y1[:, 256:]], t["head_w2c"], t["head_b2"][128:], True, exact))], 1)
    logits, value = head_final(y2, t["head_w3"], t["head_b3"], E, N)
    if stages is not None:
        stages.update(x=x, h=h, c=c, fc=fc, null_h=nh, null_c=nc, attr=attr, a2=outs[1], a1=outs[2], emb=emb, qkv=qkv, atto=atto,
                      tb=touts[1], ta=touts[2], y1=y1, y2=y2, nullmask=nm, shared=shared)
    return logits, value


# ---- random observation trees ---------------------------------------------------------------------------------------
def random_trees(rng, n, p_null=0.3, p_inf=0.1, null_inner=False, kinds=None):
    """n random observation trees in fl_observe's numbering -> dict forest [n,31,12] f32, adjacency [n,30,3] i32,
    node_order [n,31] i32, edge_order [n,30] i32.  kinds (per tree, default random): "random" (each node breadth-first
    expands with a per-tree probability while slots remain), "deep" (a chain: height 10), "full" (31 nodes),
    "root" (a single root leaf), "empty" (no edge: node_order -2 everywhere).  Null leaves (all -1, partly written
    as +inf as the observation does) appear with probability p_null among non-root leaves; other nodes get random
    features with some +inf entries.  null_inner=True makes one inner non-root node null-featured in every tree
    that has one (the observation never does: null nodes are leaves there)."""
    kinds = kinds or [rng.choice(["random", "random", "random", "deep", "full", "root", "empty"]) for _ in range(n)]
    forest = np.zeros((n, 31, 12), np.float32)
    adjacency = np.full((n, 30, 3), -2, np.int32)
    node_order = np.full((n, 31), -2, np.int32)
    edge_order = np.full((n, 30), -2, np.int32)
    for i, kind in enumerate(kinds):
        children = {}
        count = 1
        if kind == "deep":                                    # a chain: one node of every new group expands
            v = 0
            for _ in range(int(rng.randint(5, 11))):
                children[v] = count
                for j in range(3):
                    adjacency[i, count - 1 + j] = (v, count + j, j - 1)
                v = count + int(rng.randint(0, 3))
                count += 3
        elif kind in ("random", "full"):                      # breadth-first, as fl_observe numbers the nodes
            queue = [0]
            p = rng.uniform(0.3, 0.9)
            while queue and count + 3 <= 31:
                v = queue.pop(0)
                if kind == "full" or v == 0 or rng.rand() < p:
                    children[v] = count
                    for j in range(3):
                        adjacency[i, count - 1 + j] = (v, count + j, j - 1)
                    queue += [count, count + 1, count + 2]
                    count += 3
        if kind != "empty":
            order = np.full(31, -2, np.int64)
            for v in range(count - 1, -1, -1):
                order[v] = 0 if v not in children else 1 + max(order[children[v] + j] for j in range(3))
            node_order[i] = order
            for n1 in range(1, count):
                edge_order[i, n1 - 1] = order[adjacency[i, n1 - 1, 0]]
        feats = rng.uniform(-1.0, 3.0, (31, 12)).astype(np.float32)
        feats[rng.rand(31, 12) < p_inf] = np.inf
        feats[count:] = rng.uniform(-1.0, 3.0, (31 - count, 12))          # unused slots: arbitrary values
        for v in range(1, count):
            if v not in children and rng.rand() < p_null:
                feats[v] = -1.0
                feats[v, rng.rand(12) < 0.6] = np.inf
        if null_inner:
            inner = [v for v in children if v != 0]
            if inner:
                v = inner[int(rng.randint(0, len(inner)))]
                feats[v] = -1.0
                feats[v, :7] = np.inf
        forest[i] = feats
    return dict(forest=forest, adjacency=adjacency, node_order=node_order, edge_order=edge_order)


def random_obs(rng, E, N, **kw):
    """random_trees for E x N agents plus agent attributes -> observation dict of numpy arrays shaped [E,N,...]."""
    tr = random_trees(rng, E * N, **kw)
    out = {k: v.reshape((E, N) + v.shape[1:]) for k, v in tr.items()}
    out["agent_attr"] = rng.normal(0.0, 1.0, (E, N, 83)).astype(np.float32)
    return out


def packed(weights, rounding=True, device="cpu"):
    """Reference state_dict -> the packed weights as BatchedActor uploads them (matrices bf16 except head_w3, vectors
    fp32), in float64; rounding=False keeps the fp32 packing (for exact=True)."""
    from flatland_marl_b200.policy import pack_weights
    out = {}
    for k, v in pack_weights(weights).items():
        tt = torch.from_numpy(v).to(device).to(torch.float64)
        out[k] = bf16(tt) if rounding and v.ndim == 2 and k != "head_w3" else tt
    return out
