"""Rollout — PPO experience collected on the device, up to the learner's boundary.

T lock-step steps of observation -> policy forward -> seeded sampling (fl_policy_sample_actions) -> step, with every row the
batch returns copied into a trajectory buffer by one fl_copy_envs launch, GAE advantages over that buffer (fl_policy_gae),
and minibatches of its rows for the learner (PolicyLearner.ppo_grad, learner.py).
"""
import ctypes as C

import torch

from . import _lib
from .batch import BatchedRailEnv, _obs_buffers, _output_tensors
from .policy import _check
from .reset_pipeline import ResetPipeline


class Rollout:
    """Collects T steps of a whole batch with `actor` (a BatchedActor) exploring.

    env: a BatchedRailEnv built with auto_reset (an environment whose episode ended restarts in place in the next step, whose
    action is ignored) or a ResetPipeline around one (finished environments get new worlds).  Reset it before the first
    collect(); each collect() starts from the batch's current rows and leaves the batch T steps further.

    buffer (collect's result), device tensors allocated once and overwritten by every collect():
      row k = 0..T is what the batch held after step k of the collection (row 0: its rows when collect() began):
        the 7 observation tensors [T+1, E, N, ...], rewards [T+1, E, N] i32, dones [T+1, E, N+1] u8 (column N: "__all__"),
        values [T+1, E] f32 (the critic of row k; row T is the bootstrap value);
      per step k < T: actions [T, E, N] u8, log_probs [T, E, N] f32 (log pi_old of the action taken), acted [T, E] u8
        (0 where step k only reset an environment whose episode had ended: its action was ignored).

    Sampling uses seed, step = self.step + k and env_offset (the first global environment id of this batch in a sharded
    sweep: shard_range), so shards draw what one device would; self.step advances by T per collect(), and the random
    stream continues across calls.

    Host work: with a plain BatchedRailEnv and the bf16 actor the loop makes no host synchronisation and no host-to-device
    copy.  A ResetPipeline keeps its own one-step-late look at the dones flags (a synchronisation on an event recorded a
    step earlier) and replace_worlds' one synchronisation per batch of new worlds; the fp32 actor synchronises once per
    forward (per-level node counts)."""

    def __init__(self, env, actor, T, seed, env_offset=0, step=0):
        batch = env.batch if isinstance(env, ResetPipeline) else env
        if not isinstance(batch, BatchedRailEnv):
            raise TypeError("env must be a BatchedRailEnv or a ResetPipeline")
        if not batch.auto_reset:
            raise ValueError("Rollout needs a batch built with auto_reset: stepping a finished environment of a batch without "
                             "it only sets FL_ST_STEP_AFTER_DONE")
        if actor.device != batch.device:
            raise ValueError("actor and batch must be on the same device")
        if int(T) < 1:
            raise ValueError("T must be at least 1")
        self.env, self.batch, self.actor = env, batch, actor
        self.T, self.seed, self.env_offset, self.step = int(T), int(seed), int(env_offset), int(step)
        T, E, N, dev = self.T, batch.E, batch.N, batch.device
        # the buffer rows as one (T+1)*E-environment set of output rows, filled by fl_copy_envs (output rows only, parts = 0)
        obs, rewards, dones = _output_tensors((T + 1) * E, N, dev)
        self._outs = _obs_buffers(obs, rewards, dones)
        self._dst = _lib.FlBatch()
        self._dst.E, self._dst.N = (T + 1) * E, N
        self._src_ids = torch.arange(E, dtype=torch.int32, device=dev)
        self._dst_ids = torch.arange((T + 1) * E, dtype=torch.int32, device=dev).view(T + 1, E)
        rows = lambda t: t.view((T + 1, E) + tuple(t.shape[1:]))
        self.buffer = {k: rows(v) for k, v in obs.items()}
        self.buffer["rewards"], self.buffer["dones"] = rows(rewards), rows(dones)
        self.buffer["values"] = torch.zeros((T + 1, E), dtype=torch.float32, device=dev)
        self.buffer["actions"] = torch.zeros((T, E, N), dtype=torch.uint8, device=dev)
        self.buffer["log_probs"] = torch.zeros((T, E, N), dtype=torch.float32, device=dev)
        self.buffer["acted"] = torch.zeros((T, E), dtype=torch.uint8, device=dev)
        self._adv = torch.zeros((T, E), dtype=torch.float32, device=dev)
        self._ret = torch.zeros((T, E), dtype=torch.float32, device=dev)
        self._have_adv = False

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.batch.device).cuda_stream)

    def _copy_row(self, k):
        b = self.batch
        _lib.check(b.lib.fl_copy_envs(b._bp, C.byref(self._dst), self._src_ids.data_ptr(), self._dst_ids[k].data_ptr(), b.E, 0,
                                      C.byref(b._outs), C.byref(self._outs), self._stream()))

    def _forward(self, k):
        """Policy forward on the batch's current rows; the critic value goes to values[k]."""
        logits, value = self.actor.forward(self.batch.obs)
        self.buffer["values"][k].copy_(value)
        return logits

    def collect(self):
        """T steps from the batch's current rows; returns self.buffer (see the class documentation)."""
        b, buf = self.batch, self.buffer
        if not b._have_dist:
            raise ValueError("reset the batch before collecting")
        self._copy_row(0)
        for k in range(self.T):
            logits = self._forward(k)
            self.actor._sample_into(logits, b.obs["valid_actions"], self.seed, self.step + k, self.env_offset, buf["actions"][k],
                                    buf["log_probs"][k])
            torch.bitwise_xor(b.t["done_all"], 1, out=buf["acted"][k])      # done_all before the step: 1 = reset step
            self.env.step(buf["actions"][k])
            self._copy_row(k + 1)
        self._forward(self.T)
        self.step += self.T
        self._have_adv = False
        return buf

    def advantages(self, gamma=0.99, lam=0.95):
        """GAE over the last collect() (fl_policy_gae): (advantages, returns), float32 [T, E] device tensors reused by the next
        call.  Per environment, the reward of a row is the mean over its agents (the critic is a mean over agents); an episode
        end cuts the recurrence (time limits are terminal: no bootstrap); reset steps (acted == 0) are 0 in both."""
        buf, b = self.buffer, self.batch
        _check(self.actor.lib.fl_policy_gae(buf["rewards"].data_ptr(), buf["dones"].data_ptr(), buf["values"].data_ptr(),
                                            buf["acted"].data_ptr(), self.T, b.E, b.N, float(gamma), float(lam),
                                            self._adv.data_ptr(), self._ret.data_ptr(), self._stream()), "fl_policy_gae")
        self._have_adv = True
        return self._adv, self._ret

    MINIBATCH_KEYS = ("agent_attr", "forest", "adjacency", "node_order", "valid_actions", "actions", "log_probs")

    def minibatch(self, row_ids):
        """Rows k * E + e (step k < T, environment e) of the last collect(), gathered into the dict PolicyLearner.ppo_grad
        takes: the observation tensors, valid_actions, actions and log_probs [M, N, ...] of those rows, advantages and returns
        [M] of the last advantages() call, acted [M], and values [M] (the behaviour critic's value of each row, the V_old of
        ppo_grad's vf_clip).  row_ids: a sequence or tensor of ints; ids given on the host are
        range-checked there, a device tensor is used as it is (no host synchronisation).  Plain torch gathers."""
        if not self._have_adv:
            raise ValueError("call advantages() after collect() before taking minibatches")
        n = self.T * self.batch.E
        if isinstance(row_ids, torch.Tensor) and row_ids.is_cuda:
            ids = row_ids.to(device=self.batch.device, dtype=torch.int64)
        else:
            ids = torch.as_tensor(row_ids, dtype=torch.int64)
            if ids.dim() != 1 or ids.numel() == 0 or int(ids.min()) < 0 or int(ids.max()) >= n:
                raise ValueError("row_ids must be a non-empty list of ints in [0, T*E)")
            ids = ids.to(self.batch.device)
        buf = self.buffer
        rows = lambda t: t[: self.T].reshape((n,) + tuple(t.shape[2:])).index_select(0, ids)
        mb = {k: rows(buf[k]) for k in self.MINIBATCH_KEYS}
        mb["advantages"], mb["returns"], mb["acted"] = rows(self._adv), rows(self._ret), rows(buf["acted"])
        mb["values"] = rows(buf["values"])
        return mb
