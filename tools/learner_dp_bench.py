"""Data-parallel PPO learner on the GPUs of one box (PolicyLearner(group=...), DESIGN.md §4.9): one global minibatch split by
rows over G ranks, every rank computing its share with fl_policy_ppo_grad_shard_* and the gradient summed by one NCCL
all-reduce.  Run under torchrun, one rank per GPU:

    python -m torch.distributed.run --nproc-per-node G tools/learner_dp_bench.py --out profiles/learner_dp_bench_b200.json

For every group size g in 1, 2, 4, ... up to G (the first g ranks; the others wait), both precisions and both shapes of
tools/learner_bench.py — Test_03 with 1024 rows in total and the Test_02 shape with 8192 rows of 20 agents — it reports:
  - ppo_grad_ms: the time of one ppo_grad call (counts, their all-reduce, the shard call, the gradient all-reduce), the
    maximum over the group's ranks of each call's CUDA-event time, median over --calls calls;
  - allreduce_ms: the all-reduce of the flat gradient buffer alone (1,918,470 + 8 floats), same statistic;
  - rows_per_rank, and speed-up and efficiency against g = 1 measured in the same run.
Rank r of a group of g collects its own rows: environments shard_range(rows, r, g) of the global batch, in a Rollout with
env_offset = the first of them, 10 untimed steps of the bf16 actor, then one collected step; its share of the minibatch is
those rows.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import flatland_marl_b200 as fb  # noqa: E402
from flatland_marl_b200.policy import BatchedActor  # noqa: E402

CASES = [("Test_03", 1024), ("Test_02", 8192)]


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def max_over(group, values, dev):
    t = torch.tensor(values, dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return t.tolist()


def share(config, rows, rank, g, dev, weights):
    """This rank's rows of the global minibatch, from its own Rollout (collected with the bf16 actor of `weights`)."""
    lo, hi = fb.shard_range(rows, rank, g)
    batch = fb.BatchedRailEnv(bench.load_worlds(config, hi - lo, offset=lo), device=dev, auto_reset=True)
    batch.reset()
    actor = BatchedActor(weights, device=dev, precision="bf16")
    for _ in range(10):
        batch.step(actor.get_actions(batch.obs))
    ro = fb.Rollout(batch, actor, T=1, seed=1234, env_offset=lo)
    ro.collect()
    ro.advantages()
    mb = ro.minibatch(torch.arange(hi - lo, device=dev))
    return mb, batch, ro


def run(config, rows, g, precision, calls, rank, dev, weights):
    group = dist.new_group(list(range(g)))                          # every rank takes part in creating it
    out = None
    if rank < g:
        mb, batch, ro = share(config, rows, rank, g, dev, weights)
        learner = fb.PolicyLearner(weights, device=dev, precision=precision, group=group)
        learner.ppo_grad(mb)                                        # warm-up: workspace, modules, NCCL channels
        dist.all_reduce(learner._flat, group=group)
        torch.cuda.synchronize()
        t_call, t_ar = [], []
        for _ in range(calls):
            dist.barrier(group=group)
            t_call.append(event_ms(lambda: learner.ppo_grad(mb)))
            dist.barrier(group=group)
            t_ar.append(event_ms(lambda: dist.all_reduce(learner._flat, group=group)))
        t_call, t_ar = max_over(group, t_call, dev), max_over(group, t_ar, dev)
        stats = learner.ppo_grad(mb).cpu().tolist()
        plain = None
        if g == 1:                                                  # the learner without a group, on the same rows
            lp = fb.PolicyLearner(weights, device=dev, precision=precision)
            lp.ppo_grad(mb)
            plain = round(float(np.median([event_ms(lambda: lp.ppo_grad(mb)) for _ in range(calls)])), 3)
            del lp
        out = dict(config=config, rows=rows, ranks=g, precision=precision, rows_per_rank=[
            fb.shard_range(rows, r, g)[1] - fb.shard_range(rows, r, g)[0] for r in range(g)], agents_per_row=batch.N,
            ppo_grad_ms=round(float(np.median(t_call)), 3), ppo_grad_ms_calls=[round(x, 3) for x in t_call],
            allreduce_ms=round(float(np.median(t_ar)), 4), allreduce_ms_calls=[round(x, 4) for x in t_ar],
            allreduce_bytes=learner._flat.numel() * 4, stats=stats, ungrouped_ppo_grad_ms=plain)
        del learner, mb, batch, ro
        torch.cuda.empty_cache()
    dist.barrier()
    dist.destroy_process_group(group)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=7, help="timed calls per measurement (median reported)")
    ap.add_argument("--out", required=True, help="JSON file rank 0 writes the results to (its directory is created)")
    ap.add_argument("--precisions", default="bf16,fp32")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("learner_dp_bench needs CUDA devices")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if "MASTER_ADDR" not in os.environ:                              # started without torchrun: one rank
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT="29531", RANK="0", WORLD_SIZE="1")
    dist.init_process_group("nccl", device_id=dev)
    weights = fb.PolicyLearner(None, device=dev, seed=0).state_dict()
    sizes = [g for g in (1, 2, 4, 8, 16) if g <= world]
    if world not in sizes:
        sizes.append(world)
    out = None
    if rank == 0:
        try:
            power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                                   capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        except (OSError, subprocess.SubprocessError):
            power = ["unknown"]
        out = dict(gpu=torch.cuda.get_device_name(dev), gpus_name_power_limit=power, world=world, calls=args.calls, cases=[])
        print(json.dumps(out), flush=True)
    for config, rows in CASES:
        for precision in args.precisions.split(","):
            base = None
            for g in sizes:
                r = run(config, rows, g, precision, args.calls, rank, dev, weights)
                if rank == 0:
                    base = base or r["ppo_grad_ms"]
                    r["speedup_vs_1"] = round(base / r["ppo_grad_ms"], 3)
                    r["efficiency"] = round(base / r["ppo_grad_ms"] / g, 3)
                    print(json.dumps({k: v for k, v in r.items() if not k.endswith("_calls")}), flush=True)
                    out["cases"].append(r)
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
        print("wrote", args.out)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
