"""GPU: every stage of the bf16 tensor-core forward (fl_policy_forward) against the float64 restatement of its arithmetic
(tests/policy_forward_emulator.py), at the shapes where tiles and attention groups end part-way.

`BatchedActor.forward` runs with its workspace first filled with 0xFF (bf16 NaN), so that a row no kernel wrote shows up;
the stages are then read back from the workspace (`carve` below mirrors policy.cu's `carve`).  Every stage is emulated
from the inputs the kernels themselves stored, so an error is charged to the stage that made it and does not compound.

Bounds.  `ulp` is one bf16 unit in the last place of the emulated value.  Two were revised after the first B200 run, for
causes that are not kernel errors: the GELU layers' bit-equal fraction was 0.70, and att_mlp of block 2 measured 0.648 -
0.75 under the sharp weights, whose pre-activations reach far into GELU's negative tail, where 1 + tanh is small and the
2^-11 error of tanh.approx is a large part of it (0.82 - 0.92 with the default weights); and the attention bound had no
term for probabilities that round to the other bf16 neighbour, which one element in 13 million needed (60 ulp of an
output near zero by cancellation, at Test_03's 1024 x 50).
  * Exact bytes: k_prep (attr, the node rows x, nullmask), the 1024 shared null rows of h / c (all identical), and
    emb[:, 128:] (the bytes of the root's h row, 0 for a tree with no edge).
  * Tree-LSTM rows (every computed leaf, every child's f * c, every parent), the dense layers (attribute layers 2 and 3,
    layer 1 from `attr` through one emulated bf16 intermediate, QKV and att_mlp of attention block 2, head layers 1 and 2):
        |kernel - emulated| <= ulp + err,
    err = the first-order effect of tanh.approx (2^-10 relative, twice its documented 2^-11, on every tanh value; for the
    GELU of the dense layers half |x| 2^-9, tanh.approx.f16x2 rounding its input and output to f16) plus 2^-18 of the
    sum of |products| of every fp32 accumulation.  Layer 1 adds 3 sqrt(sum_k (ulp(a1_k) w_k)^2) for its rounded
    intermediate.  And at least a fixed fraction of the elements bit-equal: 0.98 for QKV (no activation: summation order
    only), 0.60 for the GELU layers, 0.50 for the Tree-LSTM rows and layer 1 (several tanh.approx per element).
  * Attention of block 2: every element within one ulp (+ 2^-18 of sum |P V| / den, + what two probabilities rounded to
    the neighbouring bf16 value move O by: see pflip_err), and at least 0.99 bit-equal, which is what catches a
    systematic error of a fraction of an ulp.
  * Logits and values: within 1e-5 of the sum of |terms| of k_head_final's fp32 dot products and mean.
Above 20000 agents the Tree-LSTM rows are checked on a seeded sample of trees that holds the first and last row of every
128-row tile, the last environment and the 128-agent boundaries inside an environment; every other stage is checked
whole.  Every check prints what it measured (-s)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

import policy_forward_emulator as pfe

pytestmark = pytest.mark.gpu

EPS_T = 2.0 ** -10        # tanh.approx.f32 / .f16x2 relative error allowance
ACC = 2.0 ** -18          # fp32 accumulation, relative to the sum of |products|
FRAC_LIN, FRAC_GELU, FRAC_TREE, FRAC_ATTN = 0.98, 0.60, 0.50, 0.99
HEAD_RTOL = 1e-5
SAMPLE_ABOVE = 20000      # agents: above this the Tree-LSTM rows are checked on a seeded sample of trees
FP32_REL, FP32_ABS = 3e-2, 1e-2   # bf16 vs fp32 path (tests/test_gpu_policy.py)
OBS = ("agent_attr", "forest", "adjacency", "node_order", "edge_order")

# (E, N): G = 128 // N environments per attention tile when N <= 128, else 128-row query tiles of one environment
SHAPES = [(300, 1), (7, 3), (5, 50), (1024, 50), (3, 64), (5, 127), (4, 128), (3, 129), (2, 255), (2, 256), (2, 257),
          (2, 425), (1, 1000), (8192, 20)]


# ---- workspace layout (policy.cu: carve) ----------------------------------------------------------------------------
def carve(M):
    """name -> (byte offset, bytes) of fl_policy_forward's workspace for M agents, and the total."""
    out, off = {}, 0
    levels_rows = (21 + 10 * (pfe.MAX_LEVELS - 1)) * M + pfe.NULL_COPIES
    for name, n in (("counts", 64 * 4), ("lists", levels_rows * 4), ("nullmask", (M + 1) * 4), ("eflags", levels_rows),
                    ("x", (M + pfe.NULL_COPIES) * pfe.NODES * 16 * 2), ("h", (M + pfe.NULL_COPIES) * pfe.NODES * 128 * 2),
                    ("c", (M + pfe.NULL_COPIES) * pfe.NODES * 128 * 2), ("fc", M * pfe.NODES * 128 * 2), ("attr", M * 128 * 2),
                    ("a1", M * 256 * 2), ("a2", M * 256 * 2), ("emb", M * 256 * 2), ("qkv", M * 768 * 2), ("atto", M * 256 * 2),
                    ("proj", M * 256 * 2), ("ta", M * 256 * 2), ("tb", M * 256 * 2), ("y1", M * 512 * 2), ("y2", M * 256 * 2)):
        out[name] = (off, n)
        off += (n + 255) & ~255
    return out, off


def buf(ws, lay, name, dtype, shape):
    off, n = lay[name]
    return ws[off:off + n].view(dtype).reshape(shape)


# ---- fixtures -------------------------------------------------------------------------------------------------------
def sharp_weights(seed=0):
    """init_weights with the q/k rows of every in_proj scaled 8x (peaked attention) and the Tree-LSTM gate rows 3x
    (saturating gates)."""
    from flatland_marl_b200 import policy_weights as pw
    w = {k: v.copy() for k, v in pw.init_weights(seed).items()}
    for l in range(3):
        w["transformer.%d.attention.in_proj_weight" % l][:512] *= 8.0
        w["transformer.%d.attention.in_proj_bias" % l][:512] *= 8.0
    for n in ("tree_lstm.W_iou.weight", "tree_lstm.U_iou.weight", "tree_lstm.W_iou.bias"):
        w[n][:256] *= 3.0
    for n in ("tree_lstm.W_f.weight", "tree_lstm.U_f.weight", "tree_lstm.W_f.bias"):
        w[n] *= 3.0
    return w


@pytest.fixture(scope="module")
def actors():
    from flatland_marl_b200.policy import BatchedActor
    return {"default": BatchedActor(None, seed=0), "sharp": BatchedActor(sharp_weights(0))}


@pytest.fixture(scope="module")
def actor_f32():
    from flatland_marl_b200.policy import BatchedActor
    return BatchedActor(None, seed=0, precision="fp32")


@pytest.fixture(scope="module")
def pool():
    """Agent rows of live observations: done agents, null leaves, trees of every depth the simulator makes."""
    from test_gpu_policy_grad import live_rows
    obs = live_rows("Test_03", 8, 30)
    return {k: obs[k].reshape((-1,) + obs[k].shape[2:]) for k in OBS}


def make_obs(pool, E, N, seed, **kw):
    """E x N agents: live rows redistributed over (E, N), every other one replaced by a generated tree."""
    rng = np.random.RandomState(seed)
    M = E * N
    idx = rng.randint(0, pool["agent_attr"].shape[0], M)
    obs = {k: pool[k][idx].copy() for k in OBS}
    ng = min(M // 2 + 1, 4096)
    gen = pfe.random_obs(rng, ng, 1, **kw)
    sel = rng.permutation(M)[:M // 2 + 1]
    for k in OBS:
        g = gen[k].reshape((ng,) + gen[k].shape[2:])
        obs[k][sel] = g[np.arange(sel.size) % ng]
    return {k: v.reshape((E, N) + v.shape[1:]) for k, v in obs.items()}


def to_dev(obs, dev):
    return {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in obs.items()}


def run(actor, d):
    """The forward on a workspace filled with 0xFF; returns (logits, value, workspace, layout) — copies."""
    E, N = int(d["agent_attr"].shape[0]), int(d["agent_attr"].shape[1])
    ws, _ = actor._buffers(E, N)
    ws.fill_(0xFF)
    logits, value = actor.forward(d)
    torch.cuda.synchronize()
    lay, total = carve(E * N)
    return logits.clone(), value.clone(), ws, lay


# ---- comparison helpers ---------------------------------------------------------------------------------------------
class Report:
    def __init__(self, tag):
        self.tag, self.lines = tag, []

    def close(self, name, got, emu, err, frac_min):
        """|got - emu| <= ulp(emu) + err everywhere and at least frac_min of got bit-equal to bf16(emu)."""
        got = got.to(torch.float64).reshape(-1)
        emu = emu.reshape(-1)
        err = err.reshape(-1) if torch.is_tensor(err) else torch.full_like(emu, float(err))
        assert got.numel() == emu.numel() and got.numel() > 0, name
        assert bool(torch.isfinite(got).all()), "%s %s: non-finite values (a row no kernel wrote?)" % (self.tag, name)
        d = (got - emu).abs()
        u = pfe.ulp(emu)
        ratio = float((d / (u + err)).max())
        eq = float((got == pfe.bf16(emu)).double().mean())
        worst_ulps = float((d / u).max())
        self.lines.append("%-28s n=%-9d worst %.3g ulp (%.3f of bound)  bit-equal %.4f (min %.2f)" %
                          (name, got.numel(), worst_ulps, ratio, eq, frac_min))
        print("  %s %s" % (self.tag, self.lines[-1]))
        i = int((d / (u + err)).argmax())
        assert ratio <= 1.0, "%s %s: |d| = %.3g at %d (emulated %.6g, kernel %.6g, bound %.3g)" % (
            self.tag, name, float(d[i]), i, float(emu[i]), float(got[i]), float(u[i] + err[i]))
        assert eq >= frac_min, "%s %s: only %.4f bit-equal" % (self.tag, name, eq)


def bits_equal(a, b):
    return torch.equal(a.contiguous().view(torch.int16), b.contiguous().view(torch.int16))


def tobf(t):
    return t.to(torch.float32).to(torch.bfloat16)


def tree_gates(iou, acc_err, c_add=None, c_add_err=0.0):
    """Error allowance of c and h from the gate accumulators (first order): tanh.approx and accumulation errors."""
    ti, to, tu = torch.tanh(iou[:, :128]), torch.tanh(iou[:, 128:256]), torch.tanh(iou[:, 256:])
    di, do, du = (EPS_T * t.abs() + e for t, e in ((ti, acc_err[:, :128]), (to, acc_err[:, 128:256]), (tu, acc_err[:, 256:])))
    c = 0.5 * tu * ti + 0.5 * tu + (c_add if c_add is not None else 0.0)
    ec = 0.5 * du * (1 + ti.abs()) + 0.5 * tu.abs() * di + c_add_err
    tc = torch.tanh(c)
    dtc = EPS_T * tc.abs() + (1 - tc * tc) * ec
    eh = 0.5 * dtc * (1 + to.abs()) + 0.5 * tc.abs() * do
    return ec, eh


def pflip_err(qkv, ao, E, N):
    """What two bf16 probabilities rounded the other way move O = sum P V / den by: the kernel's S (fp32 tensor-core sums)
    and __expf differ from the float64 S and exp in the last bits, so a P near a bf16 rounding boundary may round to the
    neighbouring value; each such P moves the numerator by 2^-8 P |v| and den by 2^-8 P.  P = 1 (the row maximum) is exact
    and never moves.  Matters where O is small by cancellation, so that its own ulp is far below that of the P V terms."""
    q = qkv[:, :256].reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    k = qkv[:, 256:512].reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    v = qkv[:, 512:].abs().reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    o = ao.abs().reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    out = torch.empty_like(o)
    for hd in range(4):
        s = pfe.f32(pfe.f32(q[:, hd] @ k[:, hd].transpose(-1, -2)) * 0.125)
        p = pfe.bf16(torch.exp(s - s.amax(-1, keepdim=True)))
        den = p.sum(-1, keepdim=True)
        p = torch.where(p < 1.0, p, torch.zeros_like(p))
        pv = torch.stack([(p * v[:, hd, None, :, d]).amax(-1) for d in range(64)], -1)
        out[:, hd] = 2.0 ** -7 * (pv + p.amax(-1, keepdim=True) * o[:, hd]) / den
    return out.permute(0, 2, 1, 3).reshape(E * N, 256)


def dense_err(srcs, w, b, act):
    a = torch.cat(srcs, 1) if len(srcs) > 1 else srcs[0]
    y = a @ w.t() + b
    dy = ACC * (a.abs() @ w.abs().t() + b.abs())
    if not act:
        return dy
    return 0.5 * y.abs() * 2.0 ** -9 + 1.2 * dy


# ---- the stage checks -----------------------------------------------------------------------------------------------
def check_stages(actor, d, tag):
    """Runs the forward and checks every stage (module docstring); returns (logits, value)."""
    t = pfe.weights64(actor.t)
    E, N = int(d["agent_attr"].shape[0]), int(d["agent_attr"].shape[1])
    M = E * N
    logits, value, ws, lay = run(actor, d)
    rep = Report("%s E=%d N=%d" % (tag, E, N))
    B = torch.bfloat16
    X = buf(ws, lay, "x", B, (M + pfe.NULL_COPIES, pfe.NODES, 16))
    H = buf(ws, lay, "h", B, (M + pfe.NULL_COPIES, pfe.NODES, 128))
    Cc = buf(ws, lay, "c", B, (M + pfe.NULL_COPIES, pfe.NODES, 128))
    FC = buf(ws, lay, "fc", B, (M, pfe.NODES, 128))
    A = buf(ws, lay, "attr", B, (M, 128))
    EMB = buf(ws, lay, "emb", B, (M, 256))

    # k_prep: exact bytes
    attr_e, x_e, nm_e = pfe.prep(d["agent_attr"].reshape(M, 83), d["forest"].reshape(M, 31, 12))
    assert bits_equal(A, tobf(attr_e)), rep.tag + " attr"
    assert bits_equal(X, tobf(x_e)), rep.tag + " x"
    nm = buf(ws, lay, "nullmask", torch.int32, (M + 1,))[:M].to(torch.int64) & 0xFFFFFFFF
    assert torch.equal(nm, nm_e), rep.tag + " nullmask"
    x = X.to(torch.float64)

    # the shared null rows: identical bytes, and the leaf of the null features
    nh, ncr = H[M:, 1], Cc[M:, 1]
    assert bits_equal(nh, nh[:1].expand_as(nh)) and bits_equal(ncr, ncr[:1].expand_as(ncr)), rep.tag + " null rows differ"
    leaves, inner, shared = pfe.levels(d["adjacency"].reshape(M, 30, 3), d["node_order"].reshape(M, 31), nm_e)
    if M > SAMPLE_ABOVE:
        # a seeded sample of the trees: the first and last row of every 128-row tile, the last environment, the rows at
        # 128-agent boundaries inside an environment, and 4096 more
        keep = torch.zeros(M, dtype=torch.bool, device=X.device)
        keep[0::128] = True
        keep[127::128] = True
        keep[M - N:] = True
        for b0 in range(128, N, 128):
            keep[b0::N] = True
            keep[b0 - 1::N] = True
        keep[torch.from_numpy(np.random.RandomState(M).randint(0, M, 4096)).to(X.device)] = True
        leaves = tuple(z[keep[leaves[0]]] for z in leaves)
        inner = {L: tuple(z[keep[v[0]]] for z in v) for L, v in inner.items()}
    xl = torch.cat([x[M, 1][None], x[leaves[0], leaves[1]]])
    he, ce = pfe.leaf(xl, t["tree_wiou"])
    acc_err = ACC * (xl.abs() @ t["tree_wiou"].abs().t())
    ec, eh = tree_gates(xl @ t["tree_wiou"].t(), acc_err)
    gh = torch.cat([nh[:1], H[leaves[0], leaves[1]]])
    gc = torch.cat([ncr[:1], Cc[leaves[0], leaves[1]]])
    rep.close("leaf h", gh, he, eh, FRAC_TREE)
    rep.close("leaf c", gc, ce, ec, FRAC_TREE)

    # inner levels: forget gates of every child, then the parent, from the stored child rows
    h64, c64 = H.to(torch.float64), Cc.to(torch.float64)
    nullh, nullc = h64[M, 1], c64[M, 1]
    fcs, fce, fcerr, ph, pc, phe, pce, pherr, pcerr = [], [], [], [], [], [], [], [], []
    for L in sorted(inner):
        tt, vv, c0 = inner[L]
        h3, f3 = [], []
        for j in range(3):
            ch = c0 + j
            sh = shared[tt, ch][:, None]
            hj = torch.where(sh, nullh[None], h64[tt, ch])
            cj = torch.where(sh, nullc[None], c64[tt, ch])
            inp = torch.cat([hj, x[tt, vv]], 1)
            acc = inp @ t["tree_ufwf"].t()
            th = torch.tanh(acc)
            fcs.append(FC[tt, ch])
            fce.append(pfe.forget(hj, x[tt, vv], cj, t["tree_ufwf"]))
            fcerr.append(0.5 * cj.abs() * (EPS_T * th.abs() + ACC * (inp.abs() @ t["tree_ufwf"].abs().t())))
            h3.append(hj)
            f3.append(FC[tt, ch].to(torch.float64))
        h3, f3 = torch.cat(h3, 1), torch.cat(f3, 1)
        hp, cp = pfe.parent(h3, x[tt, vv], f3, t["tree_uiou"], t["tree_wiou"], t["tree_wc"], t["tree_b_c"])
        iou = h3 @ t["tree_uiou"].t() + x[tt, vv] @ t["tree_wiou"].t()
        ierr = ACC * (h3.abs() @ t["tree_uiou"].abs().t() + x[tt, vv].abs() @ t["tree_wiou"].abs().t())
        cadd = f3 @ t["tree_wc"].t() + t["tree_b_c"]
        caerr = ACC * (f3.abs() @ t["tree_wc"].abs().t() + t["tree_b_c"].abs())
        ecp, ehp = tree_gates(iou, ierr, cadd, caerr)
        ph.append(H[tt, vv]); pc.append(Cc[tt, vv]); phe.append(hp); pce.append(cp); pherr.append(ehp); pcerr.append(ecp)
    if fcs:
        rep.close("forget f*c", torch.cat(fcs), torch.cat(fce), torch.cat(fcerr), FRAC_TREE)
        rep.close("parent h", torch.cat(ph), torch.cat(phe), torch.cat(pherr), FRAC_TREE)
        rep.close("parent c", torch.cat(pc), torch.cat(pce), torch.cat(pcerr), FRAC_TREE)

    # emb[:, 128:]: the root's h row, 0 for a tree with no edge
    root = d["node_order"].reshape(M, 31)[:, 0] >= 0
    want = torch.where(root[:, None], H[:M, 0].view(torch.int16), torch.zeros_like(H[:M, 0].view(torch.int16)))
    assert torch.equal(EMB[:, 128:].contiguous().view(torch.int16), want), rep.tag + " emb[:, 128:]"

    # attribute MLP: layer 1 through an emulated bf16 intermediate, layers 2 and 3 from the stored inputs
    a = A.to(torch.float64)
    a2 = buf(ws, lay, "a2", B, (M, 256))
    a1 = buf(ws, lay, "a1", B, (M, 256))
    i1 = pfe.bf16(pfe.dense([a], t["attr_w0"], t["attr_b0"], True))
    prop = 3.0 * torch.sqrt((pfe.ulp(i1) ** 2) @ (t["attr_w1"] ** 2).t())
    rep.close("attr layer 1 (via a0)", a2, pfe.dense([i1], t["attr_w1"], t["attr_b1"], True),
              dense_err([i1], t["attr_w1"], t["attr_b1"], True) + prop, FRAC_TREE)
    a2d = a2.to(torch.float64)
    rep.close("attr layer 2", a1, pfe.dense([a2d], t["attr_w2"], t["attr_b2"], True), dense_err([a2d], t["attr_w2"], t["attr_b2"], True), FRAC_GELU)
    a1d = a1.to(torch.float64)
    rep.close("attr layer 3", EMB[:, :128], pfe.dense([a1d], t["attr_w3"], t["attr_b3"], True),
              dense_err([a1d], t["attr_w3"], t["attr_b3"], True), FRAC_GELU)

    # attention block 2 (the last): QKV from tb, attention from the stored qkv, att_mlp from [tb | atto]
    tb = buf(ws, lay, "tb", B, (M, 256)).to(torch.float64)
    qkv = buf(ws, lay, "qkv", B, (M, 768))
    atto = buf(ws, lay, "atto", B, (M, 256))
    rep.close("block 2 qkv", qkv, pfe.dense([tb], t["tf_wqkv2"], t["tf_bqkv2"], False), dense_err([tb], t["tf_wqkv2"], t["tf_bqkv2"], False), FRAC_LIN)
    q = qkv.to(torch.float64)
    ao = pfe.attention(q, E, N)
    # fp32 accumulation of S (through exp, scaled by 1/8) and of P V: relative to the largest |v| of the environment
    qh = q[:, :256].abs().reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    kh = q[:, 256:512].abs().reshape(E, N, 4, 64).permute(0, 2, 1, 3)
    vmax = q[:, 512:].abs().reshape(E, N, 4, 64).permute(0, 2, 1, 3).amax(2, keepdim=True)
    smax = (qh @ kh.transpose(-1, -2)).amax(-1, keepdim=True) * 0.125
    aerr = (ACC * (1.0 + 2.0 * smax) * vmax).expand(E, 4, N, 64).permute(0, 2, 1, 3).reshape(M, 256)
    aerr = aerr + pflip_err(q, ao, E, N)
    rep.close("block 2 attention", atto, ao, aerr, FRAC_ATTN)
    ad = atto.to(torch.float64)
    rep.close("block 2 att_mlp", buf(ws, lay, "ta", B, (M, 256)), pfe.dense([tb, ad], t["tf_wm2"], t["tf_bm2"], True),
              dense_err([tb, ad], t["tf_wm2"], t["tf_bm2"], True), FRAC_GELU)

    # heads
    emb = EMB.to(torch.float64)
    ta = buf(ws, lay, "ta", B, (M, 256)).to(torch.float64)
    y1 = buf(ws, lay, "y1", B, (M, 512))
    rep.close("head layer 1", y1, pfe.dense([emb, ta], t["head_w1"], t["head_b1"], True),
              dense_err([emb, ta], t["head_w1"], t["head_b1"], True), FRAC_GELU)
    y1d = y1.to(torch.float64)
    y2 = buf(ws, lay, "y2", B, (M, 256))
    e2 = torch.cat([pfe.dense([y1d[:, :256]], t["head_w2a"], t["head_b2"][:128], True),
                    pfe.dense([y1d[:, 256:]], t["head_w2c"], t["head_b2"][128:], True)], 1)
    r2 = torch.cat([dense_err([y1d[:, :256]], t["head_w2a"], t["head_b2"][:128], True),
                    dense_err([y1d[:, 256:]], t["head_w2c"], t["head_b2"][128:], True)], 1)
    rep.close("head layer 2", y2, e2, r2, FRAC_GELU)
    y2d = y2.to(torch.float64)
    le, ve = pfe.head_final(y2d, t["head_w3"], t["head_b3"], E, N)
    lsc = (y2d[:, :128].abs() @ t["head_w3"][:5].abs().t() + t["head_b3"][:5].abs()).reshape(E, N, 5)
    vsc = (y2d[:, 128:].abs() @ t["head_w3"][5].abs() + t["head_b3"][5].abs()).reshape(E, N).sum(1) / N
    lr = float(((logits.double() - le).abs() / lsc).max())
    vr = float(((value.double() - ve).abs() / vsc).max())
    print("  %s head_final: logits %.2e, value %.2e of the |terms| (bound %.0e)" % (rep.tag, lr, vr, HEAD_RTOL))
    assert lr <= HEAD_RTOL and vr <= HEAD_RTOL, "%s head_final: %.3g / %.3g" % (rep.tag, lr, vr)
    return logits, value


@pytest.mark.parametrize("weights", ["default", "sharp"])
@pytest.mark.parametrize("E,N", SHAPES)
def test_stages(actors, pool, E, N, weights):
    if weights == "sharp" and E * N > 100000:
        pytest.skip("the sharp weights run at the shapes with partial tiles; the BASELINE batch uses the default weights")
    d = to_dev(make_obs(pool, E, N, seed=E * 1000 + N), actors[weights].device)
    check_stages(actors[weights], d, weights)


@pytest.mark.parametrize("E,N", SHAPES)
def test_batch_permutation_and_fp32_agreement(actors, actor_f32, pool, E, N):
    """A permuted batch gives every environment its bytes when the permutation keeps each environment in the same slot of its
    attention tile (G = 128 // N environments share one when N <= 128: environment e sits at keys (e mod G) N ..).  Across
    slots the bytes may differ: the P V product sums the environment's keys in 16-key tensor-core steps whose boundaries
    depend on the slot, so the fp32 sums round differently; that difference is printed and held to 2^-8 of the largest
    |logit|.  And the bf16 path stays within 3e-2 of the largest |logit| (+1e-2) of the fp32 path (tests/test_gpu_policy.py)."""
    actor = actors["default"]
    obs = make_obs(pool, E, N, seed=E * 1000 + N + 1)
    d = to_dev(obs, actor.device)
    lg, v = actor.forward(d)
    lg, v = lg.clone(), v.clone()
    rng = np.random.RandomState(E + N)
    G = 128 // N if N <= 128 else 1
    # slot-preserving: environments permuted among those with the same e mod G
    perm = np.arange(E)
    for g in range(G):
        idx = np.arange(g, E, G)
        perm[idx] = idx[rng.permutation(idx.size)]
    lp, vp = actor.forward(to_dev({k: o[perm] for k, o in obs.items()}, actor.device))
    assert torch.equal(lp, lg[perm]) and torch.equal(vp, v[perm])
    perm = rng.permutation(E)
    lp, vp = actor.forward(to_dev({k: o[perm] for k, o in obs.items()}, actor.device))
    scale = float(lg.abs().max())
    dl, dv = float((lp - lg[perm]).abs().max()), float((vp - v[perm]).abs().max())
    print("  E=%d N=%d any permutation: logits %.2e, values %.2e (2^-8 |logit| = %.2e)" % (E, N, dl, dv, scale * 2 ** -8))
    assert dl <= 2 ** -8 * scale and dv <= 2 ** -8 * scale
    if G == 1:
        assert torch.equal(lp, lg[perm]) and torch.equal(vp, v[perm])
    lf, vf = actor_f32.forward(to_dev(obs, actor_f32.device))
    scale = float(lf.abs().max())
    dl, dv = float((lg - lf).abs().max()), float((v - vf).abs().max())
    print("  E=%d N=%d bf16 vs fp32: logits %.2e, values %.2e (|logit| up to %.2f)" % (E, N, dl, dv, scale))
    assert dl <= FP32_REL * scale + FP32_ABS and dv <= FP32_REL * max(scale, float(vf.abs().max())) + FP32_ABS


@pytest.mark.parametrize("M", [1, 127, 128, 129, 4099, 163840])
def test_workspace_layout(M):
    from flatland_marl_b200.policy import lib
    lay, total = carve(M)
    assert int(lib().fl_policy_workspace_bytes(M)) == total


def test_argument_errors(actors):
    actor = actors["default"]
    L = actor.lib
    E, N = 2, 3
    obs = to_dev(pfe.random_obs(np.random.RandomState(0), E, N), actor.device)
    ws, (logits, value, _) = actor._buffers(E, N)
    ptrs = [obs[k].data_ptr() for k in ("agent_attr", "forest", "adjacency", "node_order")] + [logits.data_ptr(), value.data_ptr()]
    need = int(L.fl_policy_workspace_bytes(E * N))
    st = actor._stream()
    assert L.fl_policy_forward(C.byref(actor.struct), ws.data_ptr(), need - 1, E, N, *ptrs, st) == -1
    assert L.fl_policy_forward(None, ws.data_ptr(), need, E, N, *ptrs, st) == -1
    big = 0x3FFFFF - pfe.NULL_COPIES + 1
    assert L.fl_policy_forward(C.byref(actor.struct), ws.data_ptr(), 1 << 62, big, 1, *ptrs, st) == -1
    assert L.fl_policy_forward(C.byref(actor.struct), ws.data_ptr(), need, E, N, *ptrs, st) == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("weights", ["default", "sharp"])
def test_null_featured_inner_node(actors, actor_f32, weights):
    """A node whose twelve features are all -1 but which has children is not a null leaf: its state depends on its subtree,
    and its parent must read its own row, not the shared null row (the reference's child semantics)."""
    actor = actors[weights]
    rng = np.random.RandomState(7)
    obs = pfe.random_obs(rng, 4, 16, null_inner=True, kinds=(["random"] * 3 + ["deep"]) * 16)
    d = to_dev(obs, actor.device)
    lg, v = check_stages(actor, d, weights + " null-inner")
    if weights == "default":
        lf, vf = actor_f32.forward(to_dev(obs, actor_f32.device))
        scale = float(lf.abs().max())
        assert float((lg - lf).abs().max()) <= FP32_REL * scale + FP32_ABS
