"""Cost of collecting PPO rollouts on the device (Rollout: forward -> seeded sampling -> step -> one row copy per step), on a
B200, against the plain on-device loop `obs = batch.step(actor.get_actions(obs))` of the same batch.

Shapes: Test_03 x 1024 environments with T = 64, and the PPO sweep shape, Test_02 x 8192, with T = 32, on one GPU.  For each:
  - ms per collected step and per plain step: whole T-step windows timed with CUDA events, the two loops alternated window by
    window so that both see the same clocks and neighbours; the working sets (GBs of rows) are far larger than the 126 MB L2;
  - the shares of a collected step, from CUDA events recorded between its phases in a separate, instrumented window
    (forward + value copy, sampling + acted flags, step + observe, row copy), and the step / observe / copy kernels' device
    time from fl_profile_* in a third window;
  - the GAE time over the whole buffer (fl_policy_gae), and the buffer's size.
The card's name and power limit are read in the same run.

    python tools/rollout_bench.py --out profiles/rollout_bench_b200.json [--windows 5]
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

import bench  # noqa: E402
import flatland_marl_b200 as fb  # noqa: E402
from flatland_marl_b200.policy import BatchedActor  # noqa: E402

CASES = [("Test_03", 1024, 64), ("Test_02", 8192, 32)]
PHASES = ("forward", "sample", "step_observe", "row_copy")


def event():
    return torch.cuda.Event(enable_timing=True)


def window_ms(fn):
    a, b = event(), event()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def instrumented_collect(ro):
    """Rollout.collect with an event between every phase of every step: {phase: total ms}."""
    b, buf, T = ro.batch, ro.buffer, ro.T
    marks = []
    ro._copy_row(0)
    for k in range(T):
        ev = [event() for _ in range(5)]
        ev[0].record()
        logits = ro._forward(k)
        ev[1].record()
        ro.actor._sample_into(logits, b.obs["valid_actions"], ro.seed, ro.step + k, ro.env_offset, buf["actions"][k], buf["log_probs"][k])
        torch.bitwise_xor(b.t["done_all"], 1, out=buf["acted"][k])
        ev[2].record()
        ro.env.step(buf["actions"][k])
        ev[3].record()
        ro._copy_row(k + 1)
        ev[4].record()
        marks.append(ev)
    ro._forward(T)
    ro.step += T
    torch.cuda.synchronize()
    return {p: sum(ev[i].elapsed_time(ev[i + 1]) for ev in marks) for i, p in enumerate(PHASES)}


def run_case(actor, config, E, T, windows):
    batch = fb.BatchedRailEnv(bench.load_worlds(config, E), auto_reset=True)
    obs = batch.reset()
    for _ in range(10):                                   # past the first steps' cold caches
        obs, _, _ = batch.step(actor.get_actions(obs))
    ro = fb.Rollout(batch, actor, T=T, seed=1234)
    buffer_bytes = sum(v.numel() * v.element_size() for v in ro.buffer.values())

    def plain():
        o = batch.obs
        for _ in range(T):
            o, _, _ = batch.step(actor.get_actions(o))
    ro.collect()                                          # warm-up of both loops
    plain()
    torch.cuda.synchronize()
    col, pl = [], []
    for _ in range(windows):
        col.append(window_ms(ro.collect) / T)
        pl.append(window_ms(plain) / T)
    phases = instrumented_collect(ro)
    batch.profile(True)
    batch.profile_collect(reset=True)
    ro.collect()
    torch.cuda.synchronize()
    kern = {k: v for k, v in batch.profile_collect(reset=True).items() if v[1]}
    batch.profile(False)
    ro.advantages()
    gae = [window_ms(lambda: ro.advantages(0.99, 0.95)) for _ in range(20)]
    c, p = float(np.median(col)), float(np.median(pl))
    phase_total = sum(phases.values())
    r = dict(config=config, envs=E, agents=batch.N, T=T, buffer_bytes=buffer_bytes,
             buffer_bytes_per_agent_row=round(buffer_bytes / ((T + 1) * E * batch.N), 1),
             collect_ms_per_step=round(c, 4), plain_ms_per_step=round(p, 4), overhead=round(c / p - 1.0, 4),
             collect_ms_per_step_windows=[round(x, 4) for x in col], plain_ms_per_step_windows=[round(x, 4) for x in pl],
             phase_ms_per_step={k: round(v / T, 4) for k, v in phases.items()},
             phase_share={k: round(v / phase_total, 4) for k, v in phases.items()},
             kernel_ms_per_step={k: round(v[0] / T, 4) for k, v in kern.items()},
             kernel_launches_per_step={k: round(v[1] / T, 3) for k, v in kern.items()},
             gae_ms=round(float(np.median(gae)), 4))
    print(json.dumps(r), flush=True)
    del ro, batch
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=5, help="alternated timing windows of T steps per loop")
    ap.add_argument("--out", required=True, help="JSON file the results are written to (its directory is created)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rollout_bench needs a CUDA device")
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    out = dict(gpu=torch.cuda.get_device_name(0), power_limit=power, windows=args.windows, actor="bf16 tensor-core forward")
    print(json.dumps(out), flush=True)
    actor = BatchedActor(None, seed=0)
    out["cases"] = [run_case(actor, config, E, T, args.windows) for config, E, T in CASES]
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
