"""VectorizedOnPolicyBuffer on device memory with the GAE / statistics done by libspo.

Drop-in for safepo/common/buffer.py:24-164 of the reference (constructor arguments,
``store`` / ``finish_path`` / ``get``, the 12 keys and the env-major order of ``get()``),
re-designed for the GPU:

* one contiguous ``[num_envs, size, ...]`` tensor per field instead of ``num_envs`` python
  dicts -- ``get()`` is a zero-copy reshape (flat index = env*size + t, the order the
  reference's ``torch.cat`` over envs produces, buffer.py:149-153);
* ``finish_path`` only records where a path ends and its bootstrap values; the dual GAE
  of *all* paths of *all* envs runs as one kernel inside ``get()`` (``spo_gae_dual``), then
  ``spo_adv_stats`` / ``spo_adv_apply`` standardise (buffer.py:154-160);
* the trainers bypass ``store`` entirely: ``ActorVCritic.step(..., store=(buf.struct, t))``
  writes the transition from inside the forward kernel and ``store_transition`` applies
  the segment rule of ppo_lag.py:199-234 for every env at once.
"""
from __future__ import annotations

import ctypes as C

import torch

from safepo import _lib as L

_SCALARS = ("reward", "cost", "done", "value_r", "value_c", "adv_r", "adv_c", "target_value_r", "target_value_c",
            "log_prob")


class VectorizedOnPolicyBuffer:
    def __init__(self, obs_space, act_space, size, gamma=0.99, lam=0.95, lam_c=0.95,
                 standardized_adv_r=True, standardized_adv_c=True, device="cpu", num_envs=1,
                 gae_mode="scan"):
        device = torch.device(device)
        if device.type != "cuda":
            raise L.SpoError("VectorizedOnPolicyBuffer lives in GPU memory: pass device='cuda:<id>' (no CPU path)")
        self.num_envs, self.size = int(num_envs), int(size)
        N, T = self.num_envs, self.size
        self._device = device
        self._gamma, self._lam, self._lam_c = gamma, lam, lam_c
        self._standardized_adv_r, self._standardized_adv_c = standardized_adv_r, standardized_adv_c
        self.gae_mode = {"scan": 0, "exact": 1}[gae_mode]
        f32 = dict(dtype=torch.float32, device=device)
        self.data = {"obs": torch.zeros((N, T, *obs_space.shape), **f32),
                     "act": torch.zeros((N, T, *act_space.shape), **f32)}
        for k in _SCALARS:
            self.data[k] = torch.zeros((N, T), **f32)
        self.seg_end = torch.zeros((N, T), dtype=torch.uint8, device=device)
        self.boot_r = torch.zeros((N, T), **f32)
        self.boot_c = torch.zeros((N, T), **f32)
        self.adv_mixed = torch.zeros(N * T, **f32)
        self.stats = torch.zeros(4, dtype=torch.float64, device=device)
        self.ptr_list = [0] * N
        self.path_start_idx_list = [0] * N
        d = self.data
        self.struct = L.Rollout(L.ptr(d["obs"]), L.ptr(d["act"]), L.ptr(d["reward"]), L.ptr(d["cost"]),
                                L.ptr(d["value_r"]), L.ptr(d["value_c"]), L.ptr(d["log_prob"]), L.ptr(self.seg_end),
                                L.ptr(self.boot_r), L.ptr(self.boot_c), N, T)

    # ---- reference-compatible API ---------------------------------------------------------
    @property
    def buffers(self):
        """Per-env views, shaped like the reference's list of dicts (buffer.py:53-73)."""
        return [{k: v[i] for k, v in self.data.items()} for i in range(self.num_envs)]

    def store(self, **data):
        """Append one transition per env (buffer.py:84-95): data[key][i] goes to env i."""
        t = self.ptr_list[0]
        assert t < self.size, "Buffer overflow"
        for key, value in data.items():
            self.data[key][:, t] = value.to(self._device)
        self.ptr_list = [t + 1] * self.num_envs

    def finish_path(self, last_value_r=None, last_value_c=None, idx=0):
        """Close the path of env ``idx`` at its current pointer (buffer.py:97-140); the GAE
        itself is deferred to get()."""
        end = self.ptr_list[idx] - 1
        if end < self.path_start_idx_list[idx]:
            return
        self.seg_end[idx, end] = 1
        self.boot_r[idx, end] = 0.0 if last_value_r is None else last_value_r.reshape(()).to(self._device)
        self.boot_c[idx, end] = 0.0 if last_value_c is None else last_value_c.reshape(()).to(self._device)
        self.path_start_idx_list[idx] = self.ptr_list[idx]

    def store_transition(self, t, reward, cost, terminated, truncated, epoch_end, next_v=None, final_v=None):
        """Vectorised slot-t bookkeeping of the rollout loop (ppo_lag.py:187-234): reward,
        cost [N] float32; terminated, truncated [N] uint8; next_v / final_v = (v_r, v_c)."""
        nr, nc = next_v if next_v is not None else (None, None)
        fr, fc = final_v if final_v is not None else (None, None)
        L.call("spo_store_transition", C.byref(self.struct), int(t), L.ptr(reward), L.ptr(cost), L.ptr(terminated),
               L.ptr(truncated), int(bool(epoch_end)), L.ptr(nr), L.ptr(nc), L.ptr(fr),
               L.ptr(fc), L.stream())
        self.ptr_list = [int(t) + 1] * self.num_envs

    def compute_gae(self):
        d = self.data
        L.call("spo_gae_dual", L.ptr(d["reward"]), L.ptr(d["cost"]), L.ptr(d["value_r"]), L.ptr(d["value_c"]),
               L.ptr(self.seg_end), L.ptr(self.boot_r), L.ptr(self.boot_c),
               float(self._gamma), float(self._gamma * self._lam), float(self._gamma * self._lam_c),
               L.ptr(d["adv_r"]), L.ptr(d["adv_c"]), L.ptr(d["target_value_r"]),
               L.ptr(d["target_value_c"]), self.num_envs, self.size, self.gae_mode, L.stream())

    def finalize(self, lagrangian_multiplier=0.0, all_reduce=None):
        """Statistics + standardisation (buffer.py:154-160) + Lagrange mix (ppo_lag.py:280-281).
        ``all_reduce(stats)``: optional hook summing the 4 fp64 statistics across ranks."""
        d = self.data
        S = self.num_envs * self.size
        L.call("spo_adv_stats", L.ptr(d["adv_r"]), L.ptr(d["adv_c"]), S, L.ptr(self.stats), L.stream())
        if all_reduce is not None:
            all_reduce(self.stats)
        lam = float(lagrangian_multiplier)
        L.call("spo_adv_apply", L.ptr(d["adv_r"]), L.ptr(d["adv_c"]), S, L.ptr(self.stats),
               int(self._standardized_adv_r), int(self._standardized_adv_c), lam, lam + 1,
               L.ptr(self.adv_mixed), L.stream())
        return self.adv_mixed

    def get(self, lagrangian_multiplier=0.0, all_reduce=None):
        """All collected data, env-major [S,...] views (buffer.py:142-164); resets pointers.
        ``data["adv"]`` additionally holds (adv_r - lam*adv_c)/(lam+1)."""
        self.compute_gae()
        mixed = self.finalize(lagrangian_multiplier, all_reduce)
        S = self.num_envs * self.size
        out = {k: v.reshape(S, *v.shape[2:]) for k, v in self.data.items()}
        out["adv"] = mixed
        self.ptr_list = [0] * self.num_envs
        self.path_start_idx_list = [0] * self.num_envs
        # the path boundaries / bootstrap values belong to the epoch just consumed (they are not part of the
        # returned dict): clear them so that a store()/finish_path()/get() loop never sees stale cuts
        self.reset_segments()
        return out

    def reset_segments(self):
        self.seg_end.zero_()
        self.boot_r.zero_()
        self.boot_c.zero_()


def masked_gae_returns(rewards, value_preds, masks, popart_mean, popart_sqrt_var, gamma, gae_lambda, out=None):
    """SeparatedReplayBuffer.compute_returns / compute_cost_returns of the multi-agent path
    (reference safepo/common/buffer.py:356-384) on the device: time-major ``rewards`` [T, N, 1], ``value_preds`` and
    ``masks`` [T+1, N, 1] (value_preds[-1] = the bootstrap), PopArt statistics as two floats.  Returns [T, N, 1]."""
    T, N = rewards.shape[0], rewards.shape[1]
    if value_preds.shape[0] != T + 1 or masks.shape[0] != T + 1:
        raise L.SpoError("value_preds / masks must have T+1 time steps")
    if out is None:
        out = torch.empty_like(rewards)
    L.call("spo_gae_masked", L.ptr(rewards), L.ptr(value_preds), L.ptr(masks), float(popart_mean), float(popart_sqrt_var),
           float(gamma), float(gamma) * float(gae_lambda), L.ptr(out), N, T, L.stream())
    return out


class SeparatedReplayBuffer:
    """The multi-agent buffer of one agent on the device (reference safepo/common/buffer.py:209-465; MLP policies: no
    recurrent states, continuous actions: no available_actions).  Time-major tensors [T+1, N, ...] / [T, N, ...] like the
    reference; ``compute_returns`` / ``compute_cost_returns`` run ``spo_gae_masked``; ``whole_batch_sample`` is
    ``feed_forward_generator`` with ``num_mini_batch = 1`` (the yaml's value): one sample holding every row in a random order."""

    def __init__(self, config, obs_dim, share_obs_dim, act_dim, device):
        self.episode_length, self.n_rollout_threads = int(config["episode_length"]), int(config["n_rollout_threads"])
        self.gamma, self.gae_lambda = float(config["gamma"]), float(config["gae_lambda"])
        self.device = torch.device(device)
        T, N = self.episode_length, self.n_rollout_threads

        def z(*shape):
            return torch.zeros(*shape, dtype=torch.float32, device=self.device)
        self.aver_episode_costs = z(T + 1, N, obs_dim)      # buffer.py:240 (observation-shaped until the first return_aver_insert)
        self.share_obs, self.obs = z(T + 1, N, share_obs_dim), z(T + 1, N, obs_dim)
        self.value_preds, self.returns = z(T + 1, N, 1), z(T + 1, N, 1)
        self.cost_preds, self.cost_returns = z(T + 1, N, 1), z(T + 1, N, 1)
        self.actions, self.action_log_probs = z(T, N, act_dim), z(T, N, act_dim)
        self.rewards, self.costs = z(T, N, 1), z(T, N, 1)
        self.masks, self.active_masks = z(T + 1, N, 1) + 1, z(T + 1, N, 1) + 1
        self.factor = z(T, N, 1) + 1
        self.step = 0

    def update_factor(self, factor):
        self.factor.copy_(factor)

    def return_aver_insert(self, aver_episode_costs):
        self.aver_episode_costs = torch.as_tensor(aver_episode_costs, dtype=torch.float32).to(self.device).clone()

    def insert(self, share_obs, obs, actions, action_log_probs, value_preds, rewards, masks, active_masks=None, costs=None, cost_preds=None):
        s = self.step
        self.share_obs[s + 1].copy_(share_obs)
        self.obs[s + 1].copy_(obs)
        self.actions[s].copy_(actions)
        self.action_log_probs[s].copy_(action_log_probs)
        self.value_preds[s].copy_(value_preds)
        self.rewards[s].copy_(rewards)
        self.masks[s + 1].copy_(masks)
        if active_masks is not None:
            self.active_masks[s + 1].copy_(active_masks)
        if costs is not None:
            self.costs[s].copy_(costs)
        if cost_preds is not None:
            self.cost_preds[s].copy_(cost_preds)
        self.step = (s + 1) % self.episode_length

    def after_update(self):
        for t in (self.share_obs, self.obs, self.masks, self.active_masks):
            t[0].copy_(t[-1])

    def compute_returns(self, next_value, popart_mean, popart_sqrt_var):
        """buffer.py:356-376 with the PopArt statistics as two floats (MultiAgentTrainer.popart_mean_sqrt_var)."""
        self.value_preds[-1].copy_(next_value)
        masked_gae_returns(self.rewards, self.value_preds, self.masks, popart_mean, popart_sqrt_var, self.gamma, self.gae_lambda,
                           out=self.returns[:-1])

    def compute_cost_returns(self, next_cost, popart_mean, popart_sqrt_var):
        self.cost_preds[-1].copy_(next_cost)
        masked_gae_returns(self.costs, self.cost_preds, self.masks, popart_mean, popart_sqrt_var, self.gamma, self.gae_lambda,
                           out=self.cost_returns[:-1])

    def whole_batch_sample(self, advantages, cost_adv, perm=None):
        T, N = self.episode_length, self.n_rollout_threads
        idx = torch.randperm(T * N, device=self.device) if perm is None else torch.as_tensor(perm).to(self.device)

        def flat(t):
            return t.reshape(-1, t.shape[-1])[idx].contiguous()
        return dict(share_obs=flat(self.share_obs[:-1]), obs=flat(self.obs[:-1]), actions=flat(self.actions),
                    value_preds=flat(self.value_preds[:-1]), returns=flat(self.returns[:-1]),
                    old_action_log_probs=flat(self.action_log_probs), adv_targ=flat(advantages), factor=flat(self.factor),
                    cost_preds=flat(self.cost_preds[:-1]), cost_returns=flat(self.cost_returns[:-1]), cost_adv_targ=flat(cost_adv),
                    aver_episode_costs=self.aver_episode_costs)
