"""Cost of copying environments on the device (fl_copy_envs), on a B200.

Cases: (a) a full fork (world + state + output rows) of 512 Test_03 environments onto the other 512 of a 1024 batch;
(b) state + output rows only (destination already holds the world) for 1024 Test_03 environments into a second batch;
(c) snapshot and restore of 1024 Test_03 environments; (d) a full fork of 32 Test_14 environments onto the other 32 of a
64 batch.  Each case is timed with CUDA events, one launch per timed interval, with the 126 MB L2 overwritten before every
interval (the working sets are about L2-sized), and reported with the bytes it moves (from the shapes), its rate and its
share of the device-to-device copy peak measured in the same run (a 2 GiB tensor copy), beside the same copy done as one
index_select + index_copy_ pair per tensor and beside one lock-step step of the batch.  The caches (tree_cache,
path_cache) travel with the world; the last section measures the alternative, invalidating them and paying the cache misses
in the next observe().

    python tools/fork_bench.py --out results/fork_bench.json [--iters 30]
"""
import argparse
import ctypes as C
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
from flatland_marl_b200 import _lib  # noqa: E402
from flatland_marl_b200.batch import STATIC_ARRAYS, _state_tensors  # noqa: E402

WORLD_EXTRA = ("dist", "ridx", "srec", "wrec", "whoff", "wlist", "whits", "kcls", "sdist", "gtab", "walk_total", "tree_cache",
               "path_cache")
STATE = tuple(_state_tensors(1, 1, "cpu").keys())
FLUSH = torch.empty(0)


def timed(fn, iters):
    """Mean device time of fn() in ms: one event pair per call, L2 overwritten before each."""
    for _ in range(3):
        fn()
    total = 0.0
    for _ in range(iters):
        FLUSH.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
    return total / iters


def copy_peak(iters):
    n = 2 << 30
    x, y = torch.empty(n, dtype=torch.uint8, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda")
    ms = timed(lambda: y.copy_(x), iters)
    return n / ms / 1e6                                                          # GB/s copied (read once, written once)


def part_names(parts, outs):
    names = []
    if parts & _lib.COPY_WORLD:
        names += list(STATIC_ARRAYS) + list(WORLD_EXTRA)
    if parts & _lib.COPY_STATE:
        names += list(STATE)
    return names, outs


def bytes_per_env(batch, names, outs):
    n = sum(batch.t[k][0].numel() * batch.t[k].element_size() for k in names)
    if outs:
        n += sum(v[0].numel() * v.element_size() for v in list(batch.obs.values()) + [batch.rewards, batch.dones])
    return n


def raw_copy(src, dst, s_ids, d_ids, parts, outs=True):
    """The fl_copy_envs call of copy_from / snapshot / restore with the ids already on the device."""
    ids = torch.tensor([list(s_ids), list(d_ids)], dtype=torch.int32, device=dst.device)
    sp, dp = src._bp, dst._bp
    so, do = (C.byref(src._outs), C.byref(dst._outs)) if outs else (None, None)
    L = fb._lib.lib()

    def fn():
        _lib.check(L.fl_copy_envs(sp, dp, ids[0].data_ptr(), ids[1].data_ptr(), len(d_ids), parts, so, do,
                                  C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    return fn


def per_tensor_copy(src_t, dst_t, src_obs, dst_obs, s_ids, d_ids, names):
    """The same copy as index_select + index_copy_ per tensor (two launches each)."""
    si = torch.tensor(list(s_ids), dtype=torch.long, device="cuda")
    di = torch.tensor(list(d_ids), dtype=torch.long, device="cuda")
    pairs = [(src_t[k], dst_t[k]) for k in names] + [(src_obs[k], dst_obs[k]) for k in src_obs]

    def fn():
        for s, d in pairs:
            d.index_copy_(0, di, s.index_select(0, si))
    return fn, 2 * len(pairs)


def step_fn(batch, rng):
    a = torch.from_numpy(np.where(rng.rand(batch.E, batch.N) < 0.7, 2, rng.randint(0, 5, (batch.E, batch.N))).astype(np.uint8)).cuda()
    return lambda: batch.step(a)


def outs_of(b):
    d = dict(b.obs)
    d["rewards"], d["dones"] = b.rewards, b.dones
    return d


def report(name, n_envs, per_env, ms, peak, ms_tensor, launches_tensor, ms_step):
    moved = n_envs * per_env
    gbs = moved / ms / 1e6
    r = dict(case=name, envs=n_envs, bytes_per_env=per_env, bytes_moved=moved, ms=round(ms, 4), gb_s=round(gbs, 1),
             share_of_copy_peak=round(gbs / peak, 3), index_copy_ms=round(ms_tensor, 4), index_copy_launches=launches_tensor,
             step_ms=round(ms_step, 4))
    print(json.dumps(r), flush=True)
    return r


def main():
    global FLUSH
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--out", required=True, help="JSON file the results are written to (its directory is created)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fork_bench needs a CUDA device")
    FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    rng = np.random.RandomState(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    out = dict(gpu=torch.cuda.get_device_name(0), power_limit=power, l2_flushed_between_intervals=True, iters=args.iters)
    peak = copy_peak(args.iters)
    out["copy_peak_gb_s"] = round(peak, 1)
    print(json.dumps(out), flush=True)
    cases = []
    W, S = _lib.COPY_WORLD, _lib.COPY_STATE

    # Test_03, 1024 environments
    a = fb.BatchedRailEnv(bench.load_worlds("Test_03", 1024), auto_reset=True)
    a.reset()
    st = step_fn(a, rng)
    for _ in range(20):
        st()
    ms_step = timed(st, args.iters)
    half = list(range(512)), list(range(512, 1024))
    names, _ = part_names(W | S, True)
    fn_t, nl = per_tensor_copy(a.t, a.t, outs_of(a), outs_of(a), half[0], half[1], names)
    cases.append(report("a: full fork 512 -> 512, Test_03", 512, bytes_per_env(a, names, True),
                        timed(raw_copy(a, a, half[0], half[1], W | S), args.iters), peak, timed(fn_t, args.iters), nl, ms_step))
    b = fb.BatchedRailEnv.fork_of(a, range(1024))
    names, _ = part_names(S, True)
    ids = list(range(1024))
    fn_t, nl = per_tensor_copy(a.t, b.t, outs_of(a), outs_of(b), ids, ids, names)
    cases.append(report("b: state + output rows, 1024, Test_03", 1024, bytes_per_env(a, names, True),
                        timed(raw_copy(a, b, ids, ids, S), args.iters), peak, timed(fn_t, args.iters), nl, ms_step))
    snap = a.snapshot()
    fn_t1, nl = per_tensor_copy(a.t, snap.t, outs_of(a), dict(snap.obs, rewards=snap.rewards, dones=snap.dones), ids, ids, names)
    fn_t2, _ = per_tensor_copy(snap.t, a.t, dict(snap.obs, rewards=snap.rewards, dones=snap.dones), outs_of(a), ids, ids, names)
    snap_fn, rest_fn = raw_copy(a, snap, ids, ids, S), raw_copy(snap, a, ids, ids, S)

    def both():
        snap_fn(); rest_fn()

    def both_t():
        fn_t1(); fn_t2()
    cases.append(report("c: snapshot + restore, 1024, Test_03", 2048, bytes_per_env(a, names, True), timed(both, args.iters), peak,
                        timed(both_t, args.iters), 2 * nl, ms_step))

    # caches: copied with the world (case a) against invalidated + the next observe() paying the misses
    names_w, _ = part_names(W | S, True)
    nocache_src = _lib.FlBatch()
    C.memmove(C.byref(nocache_src), a._bp, C.sizeof(_lib.FlBatch))
    nocache_src.tree_cache, nocache_src.path_cache = None, None

    class _Shim:
        pass
    shim = _Shim()
    shim._bp, shim._outs, shim.device = C.byref(nocache_src), a._outs, a.device
    cache_bytes = sum(a.t[k][0].numel() * a.t[k].element_size() for k in ("tree_cache", "path_cache"))
    ms_full = timed(raw_copy(a, a, half[0], half[1], W | S), args.iters)
    ms_nocache = timed(raw_copy(shim, shim, half[0], half[1], W | S), args.iters)
    di = torch.tensor(half[1], dtype=torch.long, device="cuda")

    def invalidate():
        a.t["tree_cache"][di, :, 31] = 0
        a.t["path_cache"][di, :, 0, :] = 0
    ms_inval = timed(invalidate, args.iters)
    ms_obs_warm = timed(a.observe, args.iters)

    def cold_observe():
        invalidate()
        a.observe()
    ms_obs_cold = timed(cold_observe, args.iters) - ms_inval
    out["caches"] = dict(cache_bytes_per_env=cache_bytes, full_fork_ms=round(ms_full, 4), fork_without_caches_ms=round(ms_nocache, 4),
                         invalidate_ms=round(ms_inval, 4), observe_warm_ms=round(ms_obs_warm, 4),
                         observe_after_invalidating_512_ms=round(ms_obs_cold, 4),
                         copy_caches_total_ms=round(ms_full, 4),
                         invalidate_then_miss_total_ms=round(ms_nocache + ms_inval + ms_obs_cold - ms_obs_warm, 4))
    print(json.dumps(out["caches"]), flush=True)
    del a, b, snap
    torch.cuda.empty_cache()

    # Test_14, 64 environments
    c = fb.BatchedRailEnv(bench.load_worlds("Test_14", 64), auto_reset=True)
    c.reset()
    st = step_fn(c, rng)
    for _ in range(5):
        st()
    ms_step = timed(st, max(5, args.iters // 3))
    half = list(range(32)), list(range(32, 64))
    fn_t, nl = per_tensor_copy(c.t, c.t, outs_of(c), outs_of(c), half[0], half[1], names_w)
    cases.append(report("d: full fork 32 -> 32, Test_14", 32, bytes_per_env(c, names_w, True),
                        timed(raw_copy(c, c, half[0], half[1], W | S), args.iters), peak, timed(fn_t, args.iters), nl, ms_step))
    out["cases"] = cases
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
