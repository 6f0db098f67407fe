"""Cost of one PPO minibatch update's loss and gradients on the device (PolicyLearner.ppo_grad, fl_policy_ppo_grad_f32 and,
with --bf16, fl_policy_ppo_grad_bf16: the dense products on the tensor cores), on a B200, against two yardsticks:
  - the fp32 forward alone (fl_policy_forward_f32, what the training forward costs without keeping activations);
  - torch autograd on the GPU over the test suite's torch restatement of the network and loss (tests/policy_grad_oracle.py,
    fp32, TF32 off), forward + loss + backward.  Its tree index lists are built on the host per call, as the restatement does.
All are alternated call by call so that they see the same clocks and neighbours; the working sets (GBs of
activations) are far larger than the 126 MB L2.

With --bf16 the bf16 learner (same parameters) joins the alternation, and the report adds its workspace, the PPO-ratio
spread of the bf16 behaviour policy against the bf16 learner, a per-kernel time table of both learners from a separate
torch.profiler run (two calls each, after the timed ones), and the achieved rate of the tensor-core products: their FLOPs,
counted from the layer shapes and the minibatch's actual per-level node counts, over the profiled time of k_tc_gemm.

Shapes: Test_03 x 1024 rows (51,200 agents) and a Test_02-shape minibatch of 8192 rows x 20 agents (163,840 agents).  The
rows come from a Rollout collected with the bf16 actor, so the first pass also measures the spread of the PPO ratio r between
the bf16 behaviour policy and the fp32 learner.  The card's name and power limit are read in the same run.

    python tools/learner_bench.py --out profiles/learner_bench_b200.json [--calls 5]
    python tools/learner_bench.py --bf16 --out profiles/learner_bench_bf16_b200.json

With --options the run times, instead, the loss options of ppo_grad: options off against norm_adv=True, vf_clip=0.2 on the
same minibatch (mb["values"] the behaviour critic's), alternated call by call, for the fp32 and the bf16 learner at both
shapes.  The difference is the moments launch and the options' arithmetic in the loss kernel.

    python tools/learner_bench.py --options --out profiles/learner_bench_options_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import bench  # noqa: E402
import flatland_marl_b200 as fb  # noqa: E402
import policy_grad_oracle as pgo  # noqa: E402

CASES = [("Test_03", 1024, 2), ("Test_02", 8192, 2)]      # config, rows per minibatch (= environments collected), T


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def ratio_spread(mb, logits, eps=0.2):
    """r = exp(log pi_new - log pi_old) over S (acted rows, agents with a valid action), in torch (measurement only)."""
    valid = mb["valid_actions"].bool()
    xm = torch.where(valid, logits, torch.full_like(logits, -1e30))
    lp = (xm - torch.logsumexp(xm, -1, keepdim=True)).gather(-1, mb["actions"].long()[..., None])[..., 0]
    S = valid.any(-1) & mb["acted"].bool()[:, None]
    d = (lp - mb["log_probs"])[S].double()
    r = d.exp()
    q = torch.quantile((r - 1).abs().float(), torch.tensor([0.5, 0.9, 0.99], device=r.device)).tolist()
    return dict(agents=int(S.sum()), abs_r_minus_1_p50=q[0], abs_r_minus_1_p90=q[1], abs_r_minus_1_p99=q[2],
                abs_r_minus_1_max=float((r - 1).abs().max()), r_min=float(r.min()), r_max=float(r.max()),
                approx_kl=float((-d).mean()), clip_fraction=float(((r - 1).abs() > eps).double().mean()))


def tc_flops(node_order, T):
    """FLOPs (2 per multiply-add) of the tensor-core products of one fl_policy_ppo_grad_bf16 call: forward, dW for the 20
    matrices, dX for all but attr_embedding.0 (its input is the observation).  node_order [T][31] (host): inner nodes are
    those with node_order >= 1; each costs U_iou (384 x 384), U_f (3 x 128 x 128) and W_c (128 x 384) per product."""
    n_in = int((node_order >= 1).sum())
    tree = n_in * (384 * 384 + 3 * 128 * 128 + 128 * 384)
    attr0 = T * 83 * 256
    rest = T * (256 * 256 * 2 + 256 * 128 + 3 * (256 * 768 + 256 * 256 + 512 * 256) + 2 * (512 * 256 + 256 * 128))
    fwd = tree + attr0 + rest
    return 2 * (fwd + fwd + (fwd - attr0)), n_in


def kernel_table(fn, calls=2):
    """{kernel name: mean device ms per call} of fn over `calls` calls, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "self_device_time_total", 0) or 0
        if t <= 0:
            continue
        name = e.key.replace("void ", "").split("(")[0]
        out[name] = out.get(name, 0.0) + t / 1000.0 / calls
    return dict(sorted(((k, round(v, 4)) for k, v in out.items()), key=lambda kv: -kv[1]))


def run_case(config, E, T, calls, with_bf16=False):
    learner = fb.PolicyLearner(None, seed=0)
    batch = fb.BatchedRailEnv(bench.load_worlds(config, E), auto_reset=True)
    batch.reset()
    actor = learner.actor("bf16")
    for _ in range(10):                                   # past the first steps' cold caches
        batch.step(actor.get_actions(batch.obs))
    ro = fb.Rollout(batch, actor, T=T, seed=1234)
    ro.collect()
    ro.advantages()
    ids = list(range(E))                                  # one minibatch = the E rows of step 0
    mb = ro.minibatch(ids)
    N = batch.N
    edge_order = ro.buffer["edge_order"][:T].reshape((T * E, N, 30))[:E].cpu().numpy()
    obs_keys = ("agent_attr", "forest", "adjacency", "node_order")
    stats = learner.ppo_grad(mb).cpu().numpy()
    spread = ratio_spread(mb, learner.last_outputs()[0])
    # torch yardstick: the restatement in fp32 on the GPU, TF32 off
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    w = {k: v.detach().cpu().numpy() for k, v in learner.named_parameters()}
    tp = pgo.params(w, requires_grad=True, dtype=torch.float32, device=learner.device)
    host = {k: mb[k].cpu().numpy() for k in obs_keys + ("valid_actions", "actions", "log_probs", "advantages", "returns", "acted")}

    def torch_step():
        for p in tp.values():
            p.grad = None
        logits, value = pgo.forward(tp, host["agent_attr"], host["forest"], host["adjacency"], host["node_order"], edge_order)
        L, _ = pgo.ppo_loss(logits, value, host["valid_actions"], host["actions"], host["log_probs"], host["advantages"],
                            host["returns"], host["acted"], 0.2, 0.5, 0.01)
        L.backward()
    fwd = {k: mb[k] for k in obs_keys}
    torch_ok = True
    try:
        torch_step()
    except torch.cuda.OutOfMemoryError:
        torch_ok = False
        torch.cuda.empty_cache()
    learner.ppo_grad(mb)
    learner.forward(fwd)
    lb = None
    if with_bf16:
        lb = fb.PolicyLearner(learner.state_dict(), seed=0, precision="bf16")
        lb.ppo_grad(mb)
        spread_bf16 = ratio_spread(mb, lb.last_outputs()[0])
        stats_bf16 = lb.ppo_grad(mb).cpu().numpy()
    ours, f32, tor, bf = [], [], [], []
    for _ in range(calls):
        ours.append(timed(lambda: learner.ppo_grad(mb)))
        if lb is not None:
            bf.append(timed(lambda: lb.ppo_grad(mb)))
        f32.append(timed(lambda: learner.forward(fwd)))
        if torch_ok:
            tor.append(timed(torch_step))
    med = lambda x: round(float(np.median(x)), 3) if x else None
    r = dict(config=config, rows=E, agents_per_row=N, agents=E * N,
             workspace_bytes=int(learner.lib.fl_policy_workspace_bytes_grad_f32(E * N)),
             ppo_grad_ms=med(ours), fp32_forward_ms=med(f32), torch_autograd_fp32_ms=med(tor) if torch_ok else "out of memory",
             ppo_grad_ms_calls=[round(x, 3) for x in ours], fp32_forward_ms_calls=[round(x, 3) for x in f32],
             torch_autograd_fp32_ms_calls=[round(x, 3) for x in tor],
             ppo_grad_over_forward=round(med(ours) / med(f32), 3),
             first_pass_stats=dict(zip(("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction", "S", "acted_rows",
                                        "loss"), [float(x) for x in stats])),
             ratio_bf16_behaviour_fp32_learner=spread)
    if lb is not None:
        flops, n_in = tc_flops(host["node_order"], E * N)
        tab32 = kernel_table(lambda: learner.ppo_grad(mb))
        tab16 = kernel_table(lambda: lb.ppo_grad(mb))
        tc_ms = sum(v for k, v in tab16.items() if "k_tc_gemm" in k)
        r.update(bf16_ppo_grad_ms=med(bf), bf16_ppo_grad_ms_calls=[round(x, 3) for x in bf],
                 bf16_speedup_over_fp32=round(med(ours) / med(bf), 2),
                 bf16_workspace_bytes=int(lb.lib.fl_policy_workspace_bytes_grad_bf16(E * N)),
                 bf16_first_pass_stats=dict(zip(("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction", "S",
                                                 "acted_rows", "loss"), [float(x) for x in stats_bf16])),
                 ratio_bf16_behaviour_bf16_learner=spread_bf16,
                 inner_nodes=n_in, tc_product_gflop=round(flops / 1e9, 2), tc_kernel_ms=round(tc_ms, 3),
                 tc_achieved_tflops=round(flops / (tc_ms * 1e-3) / 1e12, 1) if tc_ms > 0 else None,
                 kernels_fp32_ms_per_call=tab32, kernels_bf16_ms_per_call=tab16)
    print(json.dumps(r), flush=True)
    del ro, batch, learner, tp, lb
    torch.cuda.empty_cache()
    return r


def run_options_case(config, E, T, calls):
    """ppo_grad with the options off and on (norm_adv, vf_clip = 0.2), alternated call by call, both precisions."""
    learner = fb.PolicyLearner(None, seed=0)
    batch = fb.BatchedRailEnv(bench.load_worlds(config, E), auto_reset=True)
    batch.reset()
    actor = learner.actor("bf16")
    for _ in range(10):
        batch.step(actor.get_actions(batch.obs))
    ro = fb.Rollout(batch, actor, T=T, seed=1234)
    ro.collect()
    ro.advantages()
    mb = ro.minibatch(list(range(E)))
    r = dict(config=config, rows=E, agents_per_row=batch.N, agents=E * batch.N)
    names = ("policy_loss", "value_loss", "entropy", "approx_kl", "clip_fraction", "S", "acted_rows", "loss")
    for prec in ("fp32", "bf16"):
        lr = learner if prec == "fp32" else fb.PolicyLearner(learner.state_dict(), seed=0, precision="bf16")
        off = lambda: lr.ppo_grad(mb)
        on = lambda: lr.ppo_grad(mb, vf_clip=0.2, norm_adv=True)
        s_off, s_on = off().cpu().numpy(), on().cpu().numpy()
        t_off, t_on = [], []
        for _ in range(calls):
            t_off.append(timed(off))
            t_on.append(timed(on))
        med = lambda x: round(float(np.median(x)), 3)
        r[prec] = dict(off_ms=med(t_off), on_ms=med(t_on), on_minus_off_ms=round(med(t_on) - med(t_off), 3),
                       off_ms_calls=[round(x, 3) for x in t_off], on_ms_calls=[round(x, 3) for x in t_on],
                       stats_off=dict(zip(names, [float(x) for x in s_off])), stats_on=dict(zip(names, [float(x) for x in s_on])))
        if lr is not learner:
            del lr
    print(json.dumps(r), flush=True)
    del ro, batch, learner
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5, help="alternated timed calls per implementation")
    ap.add_argument("--bf16", action="store_true", help="also time the bf16 learner and profile both")
    ap.add_argument("--options", action="store_true", help="time ppo_grad's loss options off against on, both precisions")
    ap.add_argument("--out", required=True, help="JSON file the results are written to (its directory is created)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("learner_bench needs a CUDA device")
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    out = dict(gpu=torch.cuda.get_device_name(0), power_limit=power, calls=args.calls)
    print(json.dumps(out), flush=True)
    if args.options:
        out["cases"] = [run_options_case(config, E, T, args.calls) for config, E, T in CASES]
    else:
        out["cases"] = [run_case(config, E, T, args.calls, args.bf16) for config, E, T in CASES]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
