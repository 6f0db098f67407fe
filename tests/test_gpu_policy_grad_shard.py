"""GPU: the data-parallel learner — fl_policy_ppo_counts, fl_policy_ppo_grad_shard_f32 / _bf16 (include/flatland_policy_b200.h)
and PolicyLearner(group=...).

One process, one GPU:
  - a shard call given its own counts writes the bytes of fl_policy_ppo_grad_f32 / _bf16 (gradients, statistics, logits,
    values), on golden and on live rows;
  - a live minibatch split into 2, 3 and 8 shards, the counts and gradients summed in torch, against the unsplit call.
    Logits and values of every row are bit-identical (the forward and the dX products of a row do not depend on the other
    rows); the counts are exact; the gradients differ only in the order of the weight-gradient sums (fixed row chunks whose
    bounds depend on the row count).  Bound per tensor: ||sum_k g_k - g|| <= 1e-4 (||g|| + sum_k ||g_k||), set before
    measuring; each case prints its worst measured value (-s).  The summed statistics match the full call to rounding.
Two or more GPUs (skipped with fewer): ranks started with torch.multiprocessing, a FileStore in tmp_path and NCCL.  After
ppo_grad the gradients and statistics are byte-identical across ranks and match the single-GPU call on the union of the rows
within the bound above; two calls give the same bytes; a rank with an empty share works; a sharded Rollout + Adam loop keeps
the parameters byte-identical across ranks with no torch-side host synchronisation.  The same checks also run with two ranks
sharing one GPU over gloo (which stages CUDA tensors through the host, so the no-sync check is NCCL's only)."""
import os

import numpy as np
import pytest
import torch

from test_gpu_policy_grad import device_mb, golden_rows, live_rows, make_minibatch

pytestmark = pytest.mark.gpu
REL = 1e-4
ROW_KEYS = ("advantages", "returns", "acted")


@pytest.fixture(scope="module", params=["fp32", "bf16"])
def learner(request):
    from flatland_marl_b200 import PolicyLearner
    return PolicyLearner(None, seed=0, precision=request.param)


def rows(d, lo, hi):
    return {k: v[lo:hi].contiguous() for k, v in d.items()}


def counts_of(learner, d):
    import ctypes as C
    from flatland_marl_b200.policy import _check
    E, N = d["agent_attr"].shape[:2]
    out = torch.full((2,), -1, dtype=torch.int64, device=learner.device)
    _check(learner.lib.fl_policy_ppo_counts(E, N, d["valid_actions"].data_ptr(), d["acted"].data_ptr(), out.data_ptr(),
                                            C.c_void_p(torch.cuda.current_stream(learner.device).cuda_stream)),
           "fl_policy_ppo_counts")
    return out


def call(learner, d, gcounts=None):
    """fl_policy_ppo_grad_<precision>, or with gcounts its shard call, on the rows of d: (stats, logits, value, grads), new
    tensors."""
    import ctypes as C
    from flatland_marl_b200.learner import MB_KEYS
    from flatland_marl_b200.policy import FlPpoParams, _check
    L = learner.lib
    E, N = d["agent_attr"].shape[:2]
    ws = torch.empty(int(L.fl_policy_workspace_bytes_grad_f32(E * N)), dtype=torch.uint8, device=learner.device)
    grads = [torch.full_like(p, float("nan")) for p in learner.parameters()]
    logits = torch.empty((E, N, 5), dtype=torch.float32, device=learner.device)
    value = torch.empty((E,), dtype=torch.float32, device=learner.device)
    stats = torch.empty(8, dtype=torch.float32, device=learner.device)
    prm = FlPpoParams(0.2, 0.5, 0.01)
    name = "fl_policy_ppo_grad_%s%s" % ("shard_" if gcounts is not None else "", {"fp32": "f32", "bf16": "bf16"}[learner.precision])
    extra = [] if gcounts is None else [gcounts.data_ptr()]
    ptrs = lambda ts: (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    _check(getattr(L, name)(ptrs([p.detach() for p in learner.parameters()]), ws.data_ptr(), ws.numel(), E, N,
                            *(d[k].data_ptr() for k, _, _ in MB_KEYS), *(d[k].data_ptr() for k in ROW_KEYS), *extra,
                            C.byref(prm), ptrs(grads), logits.data_ptr(), value.data_ptr(), stats.data_ptr(),
                            C.c_void_p(torch.cuda.current_stream(learner.device).cuda_stream)), name)
    torch.cuda.synchronize()
    return stats, logits, value, grads


def same_bytes(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def degenerate_live_rows(config, E, seed, T=None):
    obs = live_rows(config, E, 30, seed=seed, T=T)
    obs["valid_actions"][1, :3] = 0                                   # agents with no valid action
    obs["valid_actions"][E - 2] = 0                                   # a row with none
    return obs


def test_shard_call_with_own_counts_is_the_unsharded_call(learner, golden):
    cases = [("golden Test_03", golden_rows(golden, "t03_l0_random", (0, 46, 89, 133)), [1, 1, 0, 1]),
             ("live Test_02", degenerate_live_rows("Test_02", 6, 4, T=25), [1, 0, 1, 1, 0, 1])]
    for what, obs, acted in cases:
        d = device_mb(learner, obs, make_minibatch(learner, obs, seed=3, acted=acted))
        ref = call(learner, d)
        cnt = counts_of(learner, d)
        assert cnt.tolist() == [int(ref[0][5]), int(ref[0][6])], what
        got = call(learner, d, cnt)
        for a, b in zip(ref[:3], got[:3]):
            assert same_bytes(a, b), what
        for (name, _), a, b in zip(learner.named_parameters(), ref[3], got[3]):
            assert same_bytes(a, b), "%s: %s" % (what, name)
        print("%s %s: shard call with its own counts %s is byte-identical" % (learner.precision, what, cnt.tolist()))


@pytest.mark.parametrize("config,E,T", [("Test_02", 24, 25), ("Test_03", 16, None)])
def test_split_minibatch_sums_to_the_full_call(learner, config, E, T):
    obs = degenerate_live_rows(config, E, seed=6, T=T)
    acted = np.ones(E, np.uint8)
    acted[[0, 3, E - 1]] = 0                                          # reset rows
    d = device_mb(learner, obs, make_minibatch(learner, obs, seed=9, acted=acted))
    full = call(learner, d)
    full_cnt = counts_of(learner, d)
    for n_shards in (2, 3, 8):
        bounds = np.linspace(0, E, n_shards + 1).astype(int)
        cnt = sum(counts_of(learner, rows(d, lo, hi)) for lo, hi in zip(bounds[:-1], bounds[1:]))
        assert torch.equal(cnt, full_cnt) and cnt.tolist() == [int(full[0][5]), int(full[0][6])]
        parts = [call(learner, rows(d, lo, hi), cnt) for lo, hi in zip(bounds[:-1], bounds[1:])]
        assert same_bytes(torch.cat([p[1] for p in parts]), full[1]) and same_bytes(torch.cat([p[2] for p in parts]), full[2])
        stats = sum(p[0].double() for p in parts)
        assert stats[5] == full[0][5] and stats[6] == full[0][6]
        np.testing.assert_allclose(stats.cpu().numpy(), full[0].double().cpu().numpy(), rtol=1e-5, atol=1e-6)
        worst = 0.0
        for i, (name, _) in enumerate(learner.named_parameters()):
            g = sum(p[3][i].double() for p in parts)
            ref = full[3][i].double()
            err = float(torch.linalg.vector_norm(g - ref))
            scale = float(torch.linalg.vector_norm(ref)) + sum(float(torch.linalg.vector_norm(p[3][i].double())) for p in parts)
            assert torch.isfinite(g).all() and err <= REL * scale, "%s: %d shards, %s: %.3e > %.1e x %.3e" % (
                config, n_shards, name, err, REL, scale)
            worst = max(worst, err / scale if scale > 0 else 0.0)
        print("%s %s, %d rows in %d shards: worst per-tensor ||sum - full|| / (||full|| + sum ||shard||) = %.2e" % (
            learner.precision, config, E, n_shards, worst))


# ---- several GPUs ------------------------------------------------------------------------------------------------------
N_GPUS = torch.cuda.device_count() if torch.cuda.is_available() else 0
multi_gpu = pytest.mark.skipif(N_GPUS < 2, reason="needs two or more GPUs")


def _worker(rank, world, store_path, out_dir, precision, backend):
    import torch.distributed as dist
    import flatland_marl_b200 as fb
    from test_fork import short_worlds
    nccl = backend == "nccl"
    dev = torch.device("cuda", rank if nccl else 0)
    torch.cuda.set_device(dev)
    store = dist.FileStore(store_path, world)
    dist.init_process_group(backend, store=store, rank=rank, world_size=world, **(dict(device_id=dev) if nccl else {}))
    try:
        res = {}
        # a different seed per rank: the construction's broadcast makes every rank start from rank 0's parameters
        lg = fb.PolicyLearner(None, device=dev, seed=rank, precision=precision, group=dist.group.WORLD)
        ref = fb.PolicyLearner(fb.PolicyLearner(None, device=dev, seed=0).state_dict(), device=dev, precision=precision)
        res["params_equal_seed0"] = all(same_bytes(a.detach(), b.detach()) for a, b in zip(lg.parameters(), ref.parameters()))
        obs = degenerate_live_rows("Test_02", 10, seed=6, T=25)
        acted = np.ones(10, np.uint8)
        acted[[0, 3, 9]] = 0
        d = device_mb(ref, obs, make_minibatch(ref, obs, seed=9, acted=acted))
        full = call(ref, d)
        lo, hi = fb.shard_range(10, rank, world)
        share = rows(d, lo, hi)
        runs = []
        for _ in range(2):
            st = lg.ppo_grad(share).clone()
            runs.append((st, [p.grad.clone() for p in lg.parameters()]))
        torch.cuda.synchronize()
        res["two_calls_same"] = same_bytes(runs[0][0], runs[1][0]) and all(same_bytes(a, b) for a, b in zip(runs[0][1], runs[1][1]))
        res["grads_are_views"] = all(p.grad.data_ptr() == v.data_ptr() for p, v in zip(lg.parameters(), lg._grad_views))
        res["stats"], res["grads"] = runs[0][0].cpu(), [g.cpu() for g in runs[0][1]]
        res["full_stats"], res["full_grads"] = full[0].cpu(), [g.cpu() for g in full[3]]
        # an empty share: world - 1 rows, so one rank has none; and set_to_none grads are reattached
        for p in lg.parameters():
            p.grad = None
        k = world - 1
        lo, hi = fb.shard_range(k, rank, world)
        res["empty_share_rows"] = hi - lo
        st = lg.ppo_grad(rows(d, lo, hi)).clone()
        small = call(ref, rows(d, 0, k))
        res["empty_stats"], res["empty_grads"] = st.cpu(), [p.grad.cpu().clone() for p in lg.parameters()]
        res["small_stats"], res["small_grads"] = small[0].cpu(), [g.cpu() for g in small[3]]
        # a sharded Rollout + Adam loop: the same number of minibatches on every rank, no torch-side host sync inside
        E_tot, T = 6, 8
        lo, hi = fb.shard_range(E_tot, rank, world)
        batch = fb.BatchedRailEnv(short_worlds("Test_02", E_tot, T=20)[lo:hi], auto_reset=True, device=dev)
        batch.reset()
        ro = fb.Rollout(batch, lg.actor(), T=T, seed=3, env_offset=lo)
        opt = torch.optim.Adam(lg.parameters(), lr=1e-4)
        gen = torch.Generator(device=dev).manual_seed(100 + rank)
        for _ in range(3):
            ro.collect()
            ro.advantages()
            perm = torch.randperm(ro.T * batch.E, device=dev, generator=gen)
            torch.cuda.synchronize()
            torch.cuda.set_sync_debug_mode("error" if nccl else "default")
            try:
                for ids in torch.tensor_split(perm, 4):
                    stats = lg.ppo_grad(ro.minibatch(ids))
                    torch.nn.utils.clip_grad_norm_(lg.parameters(), 1.0)
                    opt.step()
            finally:
                torch.cuda.set_sync_debug_mode("default")
            ro.actor = lg.actor()
        res["loop_stats_finite"] = bool(torch.isfinite(stats).all())
        res["loop_params"] = [p.detach().cpu().clone() for p in lg.parameters()]
        torch.save(res, os.path.join(out_dir, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


def _run_ranks(world, tmp_path, precision, backend):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_worker, args=(r, world, str(tmp_path / "store"), str(tmp_path), precision, backend))
             for r in range(world)]
    for p in procs:
        p.start()
    try:
        for p in procs:
            p.join(timeout=600)
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(timeout=30)
            if p.is_alive():
                p.kill()
                p.join(timeout=30)
    assert [p.exitcode for p in procs] == [0] * world
    return [torch.load(str(tmp_path / ("rank%d.pt" % r))) for r in range(world)]


def _assert_close_sum(what, grads, ref_grads, names):
    worst = 0.0
    for name, g, ref in zip(names, grads, ref_grads):
        err = float(torch.linalg.vector_norm(g.double() - ref.double()))
        scale = float(torch.linalg.vector_norm(ref.double())) + float(torch.linalg.vector_norm(g.double()))
        assert err <= REL * scale, "%s %s: %.3e > %.1e x %.3e" % (what, name, err, REL, scale)
        worst = max(worst, err / scale if scale > 0 else 0.0)
    return worst


def _check_ranks(res, world, precision, backend):
    import flatland_marl_b200.policy_weights as pw
    names = [n for n, _, _ in pw.weight_spec()]
    r0 = res[0]
    for r in res:
        assert r["params_equal_seed0"] and r["two_calls_same"] and r["grads_are_views"]
        assert same_bytes(r["stats"], r0["stats"]) and all(same_bytes(a, b) for a, b in zip(r["grads"], r0["grads"]))
        assert same_bytes(r["empty_stats"], r0["empty_stats"]) and all(same_bytes(a, b) for a, b in zip(r["empty_grads"], r0["empty_grads"]))
        assert r["loop_stats_finite"]
        assert all(same_bytes(a, b) for a, b in zip(r["loop_params"], r0["loop_params"]))
        assert all(torch.isfinite(p).all() for p in r["loop_params"])
    assert sorted(r["empty_share_rows"] for r in res)[:2] == [0, 1]
    w1 = _assert_close_sum("union", r0["grads"], r0["full_grads"], names)
    w2 = _assert_close_sum("empty share", r0["empty_grads"], r0["small_grads"], names)
    for st, ref in ((r0["stats"], r0["full_stats"]), (r0["empty_stats"], r0["small_stats"])):
        assert st[5] == ref[5] and st[6] == ref[6]
        np.testing.assert_allclose(st.double().numpy(), ref.double().numpy(), rtol=1e-5, atol=1e-6)
    print("%s, %d ranks (%s): worst per-tensor difference to the single-GPU call %.2e (union), %.2e (empty share)" % (
        precision, world, backend, w1, w2))


@multi_gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_data_parallel_learner_over_gpus(tmp_path, precision):
    world = min(N_GPUS, 4)
    _check_ranks(_run_ranks(world, tmp_path, precision, "nccl"), world, precision, "nccl")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_data_parallel_learner_two_ranks_on_one_gpu(tmp_path, precision):
    _check_ranks(_run_ranks(2, tmp_path, precision, "gloo"), 2, precision, "gloo")
