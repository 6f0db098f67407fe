"""PolicyLearner — the PPO loss and its gradients for the reference network, computed on the device.

Holds the fp32 master parameters of the reference `Network` (solution/nn/net_tree.py:33-72) as torch Parameters and fills
their `.grad` with fl_policy_ppo_grad_f32 (include/flatland_policy_b200.h): a training forward in the fp32 path's arithmetic,
the clipped-surrogate PPO loss and a deterministic backward pass, all CUDA kernels of the library.  The optimiser is the
caller's: `torch.optim` and `torch.nn.utils.clip_grad_norm_` work on `parameters()` as on any module.

precision="bf16" computes the same loss through the same graph with the dense products of the 20 large weight matrices on
the tensor cores (fl_policy_ppo_grad_bf16: bf16 operands, fp32 accumulation, fp32 master weights and gradients); see
DESIGN.md §4.8 for what the two learners trade.

group= (a torch.distributed process group, NCCL on GPUs) makes the learner data-parallel: every rank passes its own share of
one minibatch, and ppo_grad leaves on every rank the gradient and the statistics of the whole minibatch (DESIGN.md §4.9,
INTEGRATION.md §7b).

ppo_grad's vf_clip and norm_adv are the clipped value loss and the advantage normalisation of common PPO implementations,
computed inside the same call (fl_policy_ppo_grad_ex_*; with a group, over the whole minibatch).
"""
import ctypes as C
import math
from collections import OrderedDict

import torch
import torch.distributed as dist

from . import policy_weights as pw
from ._lib import FlatlandB200Error
from .policy import BatchedActor, FlPpoOptions, FlPpoParams, _check, lib, weights_dict

OBS_KEYS = (("agent_attr", torch.float32, (83,)), ("forest", torch.float32, (31, 12)), ("adjacency", torch.int32, (30, 3)),
            ("node_order", torch.int32, (31,)))
MB_KEYS = OBS_KEYS + (("valid_actions", torch.uint8, (5,)), ("actions", torch.uint8, ()), ("log_probs", torch.float32, ()))
ROW_KEYS = (("advantages", torch.float32), ("returns", torch.float32), ("acted", torch.uint8))


class PolicyLearner:
    """The reference network's parameters, keyed by its state_dict names in weight_spec() order, as fp32 torch Parameters
    on `device`.

    weights: as BatchedActor — a reference checkpoint path (.pt state_dict or .npz), a state_dict-like dict, or None for
    `init_weights(seed)`.

    One update:
        stats = learner.ppo_grad(rollout.minibatch(ids))   # writes every parameter's .grad
        optimizer.step()                                   # e.g. torch.optim.Adam(learner.parameters())
        rollout.actor = learner.actor()                    # acting with the new parameters

    group: None, or a torch.distributed process group over which each minibatch is split by rows.  Construction is then a
    collective: the parameters are broadcast from the group's first rank, so every rank starts from the same bytes.  The 46
    .grad tensors and the statistics are views of one flat fp32 buffer, so that ppo_grad ends in a single all-reduce; views
    dropped by the caller (zero_grad(set_to_none=True)) are reattached by the next call.  Every rank must make the same
    sequence of ppo_grad calls, a rank with no rows in a minibatch included (pass it the empty minibatch).
    """

    def __init__(self, weights=None, device="cuda:0", seed=0, precision="fp32", group=None):
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        if not torch.cuda.is_available():
            raise FlatlandB200Error("PolicyLearner needs a CUDA device (no CPU fallback on the policy path)")
        self.lib = lib()
        self.precision = precision
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        w = pw.check_weights(weights_dict(weights, seed))
        self._params = OrderedDict((name, torch.nn.Parameter(torch.from_numpy(w[name].copy()).to(self.device)))
                                   for name, _, _ in pw.weight_spec())
        self._ws = None
        self._out = None
        self._stats = torch.zeros(8, dtype=torch.float32, device=self.device)
        self.group = group
        if group is not None:
            self._init_group()

    def _init_group(self):
        """The flat buffer [all parameters' gradients in weight_spec order | 8 statistics], its views, the int64 counts, and
        the parameters broadcast from the group's first rank."""
        ps = list(self._params.values())
        n = sum(p.numel() for p in ps)
        self._flat = torch.zeros(n + 8, dtype=torch.float32, device=self.device)
        self._grad_views, off = [], 0
        for p in ps:
            self._grad_views.append(self._flat[off:off + p.numel()].view(p.shape))
            off += p.numel()
        self._stats = self._flat[n:]
        self._counts = torch.zeros(2, dtype=torch.int64, device=self.device)
        self._moments = torch.zeros(2, dtype=torch.float64, device=self.device)
        with torch.no_grad():
            w = torch.cat([p.detach().reshape(-1) for p in ps])
            dist.broadcast(w, src=dist.get_global_rank(self.group, 0), group=self.group)
            off = 0
            for p in ps:
                p.copy_(w[off:off + p.numel()].view(p.shape))
                off += p.numel()

    def parameters(self):
        return iter(self._params.values())

    def named_parameters(self):
        return iter(self._params.items())

    def state_dict(self):
        """The parameters as CPU tensors under the reference's state_dict names (loadable by the reference `Network`)."""
        return OrderedDict((k, v.detach().cpu().clone()) for k, v in self._params.items())

    def actor(self, precision="bf16"):
        """A BatchedActor with the current parameters.  It copies them to the host once and, for bf16, packs and casts them
        there (pack_weights): a cost per update, not per minibatch."""
        return BatchedActor(self.state_dict(), device=self.device, precision=precision)

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _ptrs(self, tensors):
        return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])

    def _weights(self):
        ps = list(self._params.values())
        for p in ps:
            if p.device != self.device or p.dtype != torch.float32 or not p.is_contiguous():
                raise ValueError("parameters must stay contiguous float32 tensors on %s" % self.device)
        return self._ptrs([p.detach() for p in ps])

    def _check_obs(self, d, keys):
        a = d["agent_attr"]
        if a.dim() != 3:
            raise ValueError("agent_attr must be [E,N,83]")
        E, N = int(a.shape[0]), int(a.shape[1])
        for name, dt, tail in keys:
            if name not in d:
                raise KeyError("missing %s" % name)
            t = d[name]
            if t.device != self.device or t.dtype != dt or not t.is_contiguous():
                raise ValueError("%s must be a contiguous %s tensor on %s" % (name, dt, self.device))
            if tuple(t.shape) != (E, N) + tail:
                raise ValueError("%s must have shape %s, got %s" % (name, (E, N) + tail, tuple(t.shape)))
        return E, N

    def _outputs(self, E, N):
        if self._out is None or self._out[0].shape[:2] != (E, N):
            self._out = (torch.empty((E, N, 5), dtype=torch.float32, device=self.device),
                         torch.empty((E,), dtype=torch.float32, device=self.device))
        return self._out

    def forward(self, obs):
        """Logits [E,N,5] and values [E] of the current parameters: fl_policy_forward_f32 (fl_policy_forward_train_bf16 for
        precision="bf16"), whose bytes are those of the training forward inside ppo_grad.  Device tensors, valid until the next
        call."""
        E, N = self._check_obs(obs, OBS_KEYS)
        bf16 = self.precision == "bf16"
        need = int(self.lib.fl_policy_workspace_bytes_grad_bf16(E * N) if bf16 else self.lib.fl_policy_workspace_bytes_f32(E * N))
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        logits, value = self._outputs(E, N)
        fn, name = (self.lib.fl_policy_forward_train_bf16, "fl_policy_forward_train_bf16") if bf16 else \
            (self.lib.fl_policy_forward_f32, "fl_policy_forward_f32")
        _check(fn(self._weights(), self._ws.data_ptr(), self._ws.numel(), E, N, *(obs[k].data_ptr() for k, _, _ in OBS_KEYS),
                  logits.data_ptr(), value.data_ptr(), self._stream()), name)
        return logits, value

    def ppo_grad(self, mb, clip_eps=0.2, vf_coef=0.5, ent_coef=0.01, vf_clip=0.0, norm_adv=False, adv_eps=1e-8):
        """PPO loss of a minibatch (Rollout.minibatch's dict: the observation tensors, valid_actions, actions, log_probs
        [E,N,...], advantages, returns, acted [E], and values [E] when vf_clip > 0) and its gradient, written into every
        parameter's .grad (allocated when missing, overwritten otherwise).  The loss is stated in include/flatland_policy_b200.h
        (fl_policy_ppo_grad_f32, and FlPpoOptions for the options).

        vf_clip > 0: the clipped value loss vf_coef mean(max((V - R)^2, (V_clip - R)^2)), V_clip = V_old + clip(V - V_old,
        -vf_clip, vf_clip), with V_old = mb["values"], the behaviour critic's values.  norm_adv: the advantages normalised
        over the agents the policy term averages over, (A - mean) / (std + adv_eps), with the mean and the unbiased standard
        deviation of the whole minibatch (of every rank's share, with a group).  With the defaults (both off) the call writes
        the bytes it wrote before the options existed.

        Returns the statistics as a float32 [8] device tensor (policy loss, value loss, entropy, approximate KL, clip
        fraction, |S|, acted rows, total loss), reused by the next call.  The one host synchronisation is the fp32 path's
        (per-level node counts), in both precisions.

        With a group, mb is this rank's share of the minibatch (it may have no rows), and all of this is enqueued on the
        current stream with no torch-side host synchronisation: fl_policy_ppo_counts of the share, all_reduce of the counts;
        with norm_adv, fl_policy_ppo_moments of the share and all_reduce of those float64 sums; fl_policy_ppo_grad_ex_* with
        the minibatch's counts (and moments), all_reduce of the flat gradient and statistics buffer.  Every rank then holds the
        gradient and the statistics of the whole minibatch, byte-identical across ranks.  Every rank must pass the same
        norm_adv: it decides how many collectives the call makes."""
        E, N = self._check_obs(mb, MB_KEYS)
        for name, dt in ROW_KEYS:
            t = mb[name]
            if t.device != self.device or t.dtype != dt or not t.is_contiguous() or tuple(t.shape) != (E,):
                raise ValueError("%s must be a contiguous %s tensor of shape (%d,) on %s" % (name, dt, E, self.device))
        if not clip_eps > 0:
            raise ValueError("clip_eps must be positive")
        opts = self._options(mb, E, vf_clip, norm_adv, adv_eps)
        if self.group is not None:
            return self._ppo_grad_shard(mb, E, N, clip_eps, vf_coef, ent_coef, opts)
        self._workspace(E, N)
        grads = []
        for p in self._params.values():
            if p.grad is None or p.grad.shape != p.shape or p.grad.dtype != torch.float32 or p.grad.device != self.device \
                    or not p.grad.is_contiguous():
                p.grad = torch.empty_like(p, memory_format=torch.contiguous_format)
            grads.append(p.grad)
        logits, value = self._outputs(E, N)
        params = FlPpoParams(float(clip_eps), float(vf_coef), float(ent_coef))
        name = "fl_policy_ppo_grad_ex_bf16" if self.precision == "bf16" else "fl_policy_ppo_grad_ex_f32"
        _check(getattr(self.lib, name)(self._weights(), self._ws.data_ptr(), self._ws.numel(), E, N,
                                       *(mb[k].data_ptr() for k, _, _ in MB_KEYS), *(mb[k].data_ptr() for k, _ in ROW_KEYS),
                                       None, C.byref(params), self._ptrs(grads), logits.data_ptr(), value.data_ptr(),
                                       self._stats.data_ptr(), self._stream(), opts[1], None, C.byref(opts[0])), name)
        return self._stats

    def _options(self, mb, E, vf_clip, norm_adv, adv_eps):
        """(FlPpoOptions, pointer to the behaviour values or None), checked as the library checks them."""
        vf_clip, adv_eps = float(vf_clip), float(adv_eps)
        if not vf_clip >= 0:
            raise ValueError("vf_clip must be >= 0 (0: no value clipping)")
        if not (adv_eps >= 0 and math.isfinite(adv_eps)):
            raise ValueError("adv_eps must be finite and >= 0")
        if norm_adv not in (True, False, 0, 1):
            raise ValueError("norm_adv must be a bool")
        old = None
        if vf_clip > 0:
            if "values" not in mb:
                raise KeyError("vf_clip > 0 needs mb['values'], the behaviour critic's values (Rollout.minibatch)")
            t = mb["values"]
            if t.device != self.device or t.dtype != torch.float32 or not t.is_contiguous() or tuple(t.shape) != (E,):
                raise ValueError("values must be a contiguous float32 tensor of shape (%d,) on %s" % (E, self.device))
            old = t.data_ptr()
        return FlPpoOptions(vf_clip, int(bool(norm_adv)), adv_eps), old

    def _workspace(self, E, N):
        bf16 = self.precision == "bf16"
        need = int(self.lib.fl_policy_workspace_bytes_grad_bf16(E * N) if bf16 else self.lib.fl_policy_workspace_bytes_grad_f32(E * N))
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)

    def _ppo_grad_shard(self, mb, E, N, clip_eps, vf_coef, ent_coef, opts):
        """ppo_grad of one rank's share: this rank's contribution computed with the minibatch's counts (and, with norm_adv,
        its advantage moments), then summed over the group.  A share with no rows contributes zero counts, moments, gradients
        and statistics and joins the same collectives."""
        for p, v in zip(self._params.values(), self._grad_views):
            if p.grad is None or p.grad.data_ptr() != v.data_ptr() or p.grad.shape != v.shape or p.grad.stride() != v.stride():
                p.grad = v
        stream = self._stream()
        if E > 0:
            _check(self.lib.fl_policy_ppo_counts(E, N, mb["valid_actions"].data_ptr(), mb["acted"].data_ptr(),
                                                 self._counts.data_ptr(), stream), "fl_policy_ppo_counts")
        else:
            self._counts.zero_()
        dist.all_reduce(self._counts, group=self.group)
        norm = opts[0].norm_adv == 1
        if norm:
            if E > 0:
                _check(self.lib.fl_policy_ppo_moments(E, N, mb["valid_actions"].data_ptr(), mb["acted"].data_ptr(),
                                                      mb["advantages"].data_ptr(), self._moments.data_ptr(), stream),
                       "fl_policy_ppo_moments")
            else:
                self._moments.zero_()
            dist.all_reduce(self._moments, group=self.group)
        logits, value = self._outputs(E, N)
        if E > 0:
            self._workspace(E, N)
            params = FlPpoParams(float(clip_eps), float(vf_coef), float(ent_coef))
            name = "fl_policy_ppo_grad_ex_bf16" if self.precision == "bf16" else "fl_policy_ppo_grad_ex_f32"
            _check(getattr(self.lib, name)(self._weights(), self._ws.data_ptr(), self._ws.numel(), E, N,
                                           *(mb[k].data_ptr() for k, _, _ in MB_KEYS), *(mb[k].data_ptr() for k, _ in ROW_KEYS),
                                           self._counts.data_ptr(), C.byref(params), self._ptrs(self._grad_views),
                                           logits.data_ptr(), value.data_ptr(), self._stats.data_ptr(), stream, opts[1],
                                           self._moments.data_ptr() if norm else None, C.byref(opts[0])), name)
        else:
            self._flat.zero_()
        dist.all_reduce(self._flat, group=self.group)
        return self._stats

    def last_outputs(self):
        """(logits [E,N,5], values [E]) of the last ppo_grad or forward call, device tensors."""
        return self._out
