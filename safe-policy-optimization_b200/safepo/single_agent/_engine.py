"""Shared machinery of the twelve single-agent trainers (ppo_lag, focops, cpo, trpo_lag and their siblings).

What the reference spells out four times as python loops
(safepo/single_agent/ppo_lag.py:159-349 and the byte-identical rollout blocks of
cpo/focops/trpo_lag) is expressed here once on top of the libspo kernels:

* ``Rollout``  -- the rollout / bootstrap control loop R0 (ppo_lag.py:159-235), vectorised:
  one fused step kernel per env step (forward + sample + log-prob + store), the segment
  rule applied to all envs by ``spo_store_transition``, episode accounting on the host in
  numpy exactly in the reference's env-index order (SURVEY Appendix A4).
* ``PolicyGradientUpdate`` -- ppo_lag.py:276-348 / focops.py:280-366: per pass one
  persistent ``spo_pg_update`` launch + one ``spo_actor_kl`` launch; early stop, logged
  losses and StopIter live in a device control block that is read once.
* ``TrustRegionUpdate`` -- cpo.py:351-571 / trpo_lag.py:358-494 on ``spo_surrogate_grad``,
  ``spo_conjugate_gradient``, ``spo_fvp``, ``spo_linesearch_eval``.

RNG modes (``args.rng``): ``host`` consumes torch's CPU generator draw-for-draw like the
reference on CPU (action noise, the discarded bootstrap samples of ppo_lag.py:206/211, the
two int64 draws per DataLoader pass) so a run is comparable number-for-number;
``device`` uses the in-kernel Philox stream and device-side permutations.
"""
from __future__ import annotations

import ctypes as C
import random
import time
from collections import deque

import numpy as np
import torch

from safepo import _lib as L
from safepo.common.buffer import VectorizedOnPolicyBuffer
from safepo.common.lagrange import Lagrange, PIDLagrangian
from safepo.common.logger import EpochLogger
from safepo.common.model import ActorVCritic

CUP_LAMBDA, CUP_NU = 0.95, 0.20       # cup.py:45-46


def _lagrange(upper_bound=None):
    return lambda args: Lagrange(args.cost_limit, args.lagrangian_multiplier_init, args.lagrangian_multiplier_lr,
                                 lagrangian_upper_bound=upper_bound)


# What sets the algorithms of a family apart.  Policy-gradient family (ppo_lag.py and its siblings, SURVEY 8f rank 2):
# algorithm -> (loss kind of spo_pg_update, multiplier factory or None).
PG_ALGOS = {
    "ppo_lag": (L.LOSS_PPO_CLIP, _lagrange()),
    "ppo": (L.LOSS_PPO_CLIP, None),
    "pg": (L.LOSS_PG, None),
    "cppo_pid": (L.LOSS_PPO_CLIP, lambda args: PIDLagrangian(args.cost_limit, args.lagrangian_multiplier_init)),
    "cup": (L.LOSS_PPO_CLIP, _lagrange(CUP_NU)),
    "focops": (L.LOSS_FOCOPS, _lagrange(2.0)),
}
# Trust-region family (cpo.py, trpo_lag.py and their siblings): algorithm -> (TrustRegionUpdate step: run_cpo with this
# variant, run_trpo or run_npg; multiplier factory or None; whether Misc/AcceptanceStep is logged).
TR_ALGOS = {
    "cpo": ("cpo", None, True),
    "pcpo": ("pcpo", None, True),
    "trpo_lag": ("trpo", _lagrange(), True),
    "trpo": ("trpo", None, True),
    "rcpo": ("npg", _lagrange(), False),
    "natural_pg": ("npg", None, False),
}


# ---------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------

def seed_all(seed):
    """ppo_lag.py:69-72."""
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)


def reference_order(S):
    """Sample order of one ``for batch in DataLoader(shuffle=True)`` pass of the reference
    (ppo_lag.py:283-294): the iterator draws a base seed, the RandomSampler a second one,
    both from the global CPU generator; the order is randperm(S) under the second."""
    torch.empty((), dtype=torch.int64).random_()
    s = int(torch.empty((), dtype=torch.int64).random_().item())
    g = torch.Generator()
    g.manual_seed(s)
    return torch.randperm(S, generator=g)


class LinearDecay:
    """LinearLR(start_factor=1, end_factor=0, total_iters=epochs) on one lr
    (ppo_lag.py:105-111), with torch's chained update so the float is identical."""

    def __init__(self, lr, epochs):
        self.lr, self.epochs, self.last = lr, epochs, 0

    def step(self):
        self.last += 1
        if self.last <= self.epochs:
            self.lr = self.lr * (1.0 + (0.0 - 1.0) / (self.epochs * 1.0 + (self.last - 1) * (0.0 - 1.0)))
        return self.lr


class AdamState:
    """Adam moments / step counters of the three nets, packed like the parameters."""

    def __init__(self, policy):
        dev = policy.flat.device
        self.m = torch.zeros_like(policy.flat)
        self.v = torch.zeros_like(policy.flat)
        self.t = torch.zeros(3, dtype=torch.int32, device=dev)


def _normalizer_state(roll):
    """What the reference checkpoints as "Normalizer" (ppo_lag.py:381-386: env.obs_rms): a host object with ``mean`` / ``var`` /
    ``count`` numpy fields and ``update()`` like gymnasium's RunningMeanStd -- evaluate.py:56-57 assigns the unpickled object
    straight to ``eval_env.obs_rms`` -- holding the device-side statistics when observations are normalised on the device, else
    whatever the env carries."""
    norm = getattr(roll, "obs_norm", None)
    if norm is not None:
        return norm.obs_rms.host_copy()
    return getattr(roll.env, "obs_rms", None)


def make_ctrl(device):
    return torch.zeros(L.CTRL_BYTES, dtype=torch.uint8, device=device)


def read_ctrl(ctrl):
    return ctrl.cpu().numpy().view(L.CTRL_DTYPE)[0]


# ---------------------------------------------------------------------------------------
# rollout
# ---------------------------------------------------------------------------------------

class Rollout:
    def __init__(self, env, policy, buffer, logger, args, device):
        self.env, self.policy, self.buffer, self.logger, self.args = env, policy, buffer, logger, args
        self.device = device
        N, D = args.num_envs, policy.obs_dim
        self.N, self.D, self.A = N, D, policy.act_dim
        self.host_rng = getattr(args, "rng", "device") == "host"
        self.ep_ret, self.ep_cost, self.ep_len = np.zeros(N), np.zeros(N), np.zeros(N)
        self.rew_deque, self.cost_deque, self.len_deque = deque(maxlen=50), deque(maxlen=50), deque(maxlen=50)
        # pinned staging: one H2D per env step carries next_obs | reward | cost | terminated | truncated
        self.stage_h = torch.empty(N * (D + 2) + N, dtype=torch.float32).pin_memory()
        self.stage_d = torch.empty_like(self.stage_h, device=device)
        self.flags_h = torch.empty(2 * N, dtype=torch.uint8).pin_memory()
        self.flags_d = torch.empty(2 * N, dtype=torch.uint8, device=device)
        self.final_h = torch.empty(N, D, dtype=torch.float32).pin_memory()
        self.final_d = torch.empty(N, D, dtype=torch.float32, device=device)
        self.act_h = torch.empty(N, self.A, dtype=torch.float32).pin_memory()
        self.obs_d = torch.empty(N, D, dtype=torch.float32, device=device)
        self.bytes_h2d = 0
        self.bytes_d2h = 0
        # SafeNormalizeObservation (env.py:66,77) on the device: statistics updated and observations
        # normalised right after the H2D of every env step (reset included, like gymnasium's wrapper)
        # A host env built by safepo.common.env.make_sa_mujoco_env is bare: it asks for both wrappers of the
        # reference's factory (env.py:62-66) through ``device_wrappers``.
        wants = getattr(env, "device_wrappers", ())
        self.obs_norm = None
        if getattr(args, "normalize_obs", False) or "normalize_obs" in wants:
            from safepo.common.normalizer import SafeNormalizeObservation
            self.obs_norm = SafeNormalizeObservation(D, device)
            if hasattr(env, "obs_rms"):
                env.obs_rms = self.obs_norm.obs_rms
        self.act_rescale = None
        if "rescale_action" in wants:
            from safepo.common.normalizer import SafeRescaleAction
            self.act_rescale = SafeRescaleAction(env.action_space.low, env.action_space.high, device)
            self.act_env_d = torch.empty(N, self.A, dtype=torch.float32, device=device)
        obs, _ = env.reset()
        self.obs_d.copy_(torch.as_tensor(np.asarray(obs), dtype=torch.float32))
        if self.obs_norm is not None:
            self.obs_norm.normalize(self.obs_d, out=self.obs_d)

    WINDOW = 50     # the reference's deque(maxlen=50) of finished episodes (ppo_lag.py:142-147)

    def _account_finished(self, finished):
        """Episode bookkeeping of ppo_lag.py:216-230 for the envs that finished in this step (ascending env index): every
        finished episode is appended to the three 50-episode deques and the running means of the deques are logged once
        per episode.  Vectorised: once the deques are full, the k running means of a step are the row means of a
        (k x 50) sliding window over [old deque | new values] -- np.mean along the contiguous last axis uses the same
        pairwise summation as np.mean of the deque, so the logged numbers are bit-identical to the reference's per-env
        loop; no Python iteration over envs (1024 of them finish in the same step at config 2).  While a deque is still
        filling (the first 50 episodes of a run) the windows have different lengths and the plain loop runs.
        The returns are accumulated on the host in float64 like the reference does with the env's float64 rewards
        (ep_ret += reward, ppo_lag.py:179-181): the device only ever sees their fp32 copies."""
        k = len(finished)
        if k == 0:
            return
        logger, W = self.logger, self.WINDOW
        if len(self.rew_deque) < W:
            for idx in finished:               # ascending env index, ppo_lag.py:199,216-230
                self.rew_deque.append(self.ep_ret[idx])
                self.cost_deque.append(self.ep_cost[idx])
                self.len_deque.append(self.ep_len[idx])
                logger.store(**{"Metrics/EpRet": np.mean(self.rew_deque), "Metrics/EpCost": np.mean(self.cost_deque),
                                "Metrics/EpLen": np.mean(self.len_deque)})
        else:
            means = []
            for dq, vals in ((self.rew_deque, self.ep_ret), (self.cost_deque, self.ep_cost), (self.len_deque, self.ep_len)):
                seq = np.concatenate([np.fromiter(dq, dtype=np.float64, count=W), vals[finished]])
                means.append(np.lib.stride_tricks.sliding_window_view(seq, W)[1:].mean(axis=1))
                dq.extend(seq[-min(k, W):])
            ed = logger.epoch_dict
            ed.setdefault("Metrics/EpRet", []).extend(means[0])
            ed.setdefault("Metrics/EpCost", []).extend(means[1])
            ed.setdefault("Metrics/EpLen", []).extend(means[2])
        self.ep_ret[finished] = 0.0
        self.ep_cost[finished] = 0.0
        self.ep_len[finished] = 0.0
        logger.logged = False

    def _burn_bootstrap_draws(self, terminated, truncated, epoch_end):
        """The reference obtains bootstrap values with policy.step(..., deterministic=False)
        (ppo_lag.py:204-213): every such call discards one [A] normal draw."""
        for idx in range(self.N):
            if (epoch_end or terminated[idx] or truncated[idx]) and not terminated[idx]:
                if epoch_end:
                    torch.empty(self.A).normal_()
                if truncated[idx]:
                    torch.empty(self.A).normal_()

    def run(self, T):
        """One epoch of rollout (T steps of all envs).  Returns wall-clock seconds."""
        t0 = time.time()
        N, D, A = self.N, self.D, self.A
        pol, buf, env, logger = self.policy, self.buffer, self.env, self.logger
        stage_h, stage_d = self.stage_h, self.stage_d
        obs_view = stage_d[: N * D].view(N, D)
        rew_view = stage_d[N * D: N * D + N]
        cost_view = stage_d[N * D + N: N * D + 2 * N]
        for t in range(T):
            eps = torch.empty(N, A).normal_().to(self.device, non_blocking=True) if self.host_rng else None
            act, _, _, _ = pol.step(self.obs_d, eps=eps, store=(buf.struct, t))
            if self.act_rescale is not None:     # the buffer keeps the policy's action; the env gets the rescaled one
                act = self.act_rescale.action(act, out=self.act_env_d)
            self.act_h.copy_(act, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            self.bytes_d2h += N * A * 4
            action = self.act_h.numpy()
            next_obs, reward, cost, terminated, truncated, info = env.step(action.squeeze() if N == 1 else action)
            self.ep_ret += reward
            self.ep_cost += cost
            self.ep_len += 1
            terminated = np.asarray(terminated, dtype=bool)
            truncated = np.asarray(truncated, dtype=bool)
            sh = stage_h.numpy()
            sh[: N * D] = np.asarray(next_obs, dtype=np.float32).reshape(-1)
            sh[N * D: N * D + N] = reward
            sh[N * D + N: N * D + 2 * N] = cost
            fh = self.flags_h.numpy()
            fh[:N] = terminated
            fh[N:] = truncated
            stage_d.copy_(stage_h, non_blocking=True)
            self.flags_d.copy_(self.flags_h, non_blocking=True)
            self.bytes_h2d += stage_h.numel() * 4 + 2 * N
            if self.obs_norm is not None:
                self.obs_norm.normalize(obs_view, out=obs_view)   # in place; final_observation stays raw (SURVEY A5)
            epoch_end = t >= T - 1
            any_trunc = bool(truncated.any())
            final_v = None
            if any_trunc:
                fin = info.get("final_observation_dense")
                if fin is None:  # gymnasium convention: object array of per-env arrays / None
                    fin = np.stack([a if a is not None else np.zeros(D) for a in info["final_observation"]])
                self.final_h.numpy()[:] = np.asarray(fin, dtype=np.float32)
                self.final_d.copy_(self.final_h, non_blocking=True)
                self.bytes_h2d += N * D * 4
                final_v = pol.values(self.final_d)     # raw final observation, ppo_lag.py:209-213
            next_v = pol.values(obs_view) if epoch_end else None
            buf.store_transition(t, rew_view, cost_view, self.flags_d[:N], self.flags_d[N:], epoch_end, next_v, final_v)
            self.obs_d.copy_(obs_view)
            if self.host_rng and (epoch_end or terminated.any() or any_trunc):
                self._burn_bootstrap_draws(terminated, truncated, epoch_end)
            self._account_finished(np.nonzero(terminated | truncated)[0])
        torch.cuda.current_stream().synchronize()
        return time.time() - t0


class DeviceTapeRollout(Rollout):
    """Rollout whose environment stream is already resident in HBM: the frame pools of a
    SyntheticVecEnv are copied to the device once, every step reads its frame there, and
    nothing crosses PCIe inside the loop (no action read-back either: the synthetic stream
    does not depend on the action).  Episode accounting still runs on the host from the
    env's own pools, so Jc / logging are identical to the host-env path."""

    def __init__(self, env, policy, buffer, logger, args, device):
        super().__init__(env, policy, buffer, logger, args, device)
        f32 = dict(dtype=torch.float32, device=device)
        self.obs_pool = torch.as_tensor(env._obs, **f32)
        self.final_pool = torch.as_tensor(env._final, **f32)
        self.rew_pool = torch.as_tensor(env._rew, **f32)
        self.cost_pool = torch.as_tensor(env._cost, **f32)
        self.zeros8 = torch.zeros(self.N, dtype=torch.uint8, device=device)
        self.ones8 = torch.ones(self.N, dtype=torch.uint8, device=device)
        self.k = 0  # frame index of the current observation

    def _flags(self, arr):
        if not arr.any():
            return self.zeros8
        if arr.all():
            return self.ones8
        return torch.as_tensor(arr.astype(np.uint8)).to(self.device, non_blocking=True)

    def run(self, T):
        t0 = time.time()
        N, A = self.N, self.A
        pol, buf, env, logger = self.policy, self.buffer, self.env, self.logger
        for t in range(T):
            eps = torch.empty(N, A).normal_().to(self.device, non_blocking=True) if self.host_rng else None
            pol.step(self.obs_pool[self.k], eps=eps, store=(buf.struct, t), outputs=False)
            _, reward, cost, terminated, truncated, info = env.step(None)
            k = env._k % env._pool
            self.ep_ret += reward
            self.ep_cost += cost
            self.ep_len += 1
            epoch_end = t >= T - 1
            any_trunc = bool(truncated.any())
            final_v = pol.values(self.final_pool[k]) if any_trunc else None
            next_v = pol.values(self.obs_pool[k]) if epoch_end else None
            buf.store_transition(t, self.rew_pool[k], self.cost_pool[k], self._flags(terminated), self._flags(truncated),
                                 epoch_end, next_v, final_v)
            self.k = k
            if self.host_rng and (epoch_end or terminated.any() or any_trunc):
                self._burn_bootstrap_draws(terminated, truncated, epoch_end)
            self._account_finished(np.nonzero(terminated | truncated)[0])
        return time.time() - t0


# ---------------------------------------------------------------------------------------
# minibatch updates: PPO-Lag / FOCOPS actor + critics, CPO / TRPO-Lag critics
# ---------------------------------------------------------------------------------------

def _old_dist(policy, obs, old_mean, old_log_std):
    """The old distribution of ppo_lag.py:277 / cpo.py:365: the actor's mean on ``obs`` into ``old_mean`` (reallocated when
    the batch size changed) and its log_std into ``old_log_std``.  Returns old_mean."""
    S = obs.shape[0]
    if old_mean is None or old_mean.shape[0] != S:
        old_mean = torch.empty(S, policy.act_dim, dtype=torch.float32, device=old_log_std.device)
    L.call("spo_actor_forward", C.byref(policy.dims), L.ptr(policy.flat), L.ptr(obs), S, L.ptr(old_mean), L.stream())
    old_log_std.copy_(policy.flat[: policy.act_dim])
    return old_mean


class _MinibatchUpdate:
    """What PolicyGradientUpdate and CriticRegression share: Adam state, control block and hyper-parameters of
    ``spo_pg_update``, and one pass of it over a shuffled batch."""

    def __init__(self, policy, cfg, host_rng, device, dp, lr_actor, lr_critic, focops_lam, focops_kl):
        self.policy, self.cfg, self.host_rng, self.device = policy, cfg, host_rng, device
        self.dp = dp          # safepo.common.dist.DataParallel or None
        self.adam = AdamState(policy)
        self.ctrl = make_ctrl(device)
        self.hp = L.HParams(lr_actor, lr_critic, lr_critic, 0.9, 0.999, 1e-8, cfg["max_grad_norm"],
                            0.001 if cfg.get("use_critic_norm", True) else 0.0, 0.8, 1.2, focops_lam, focops_kl,
                            2.0 if cfg.get("use_value_coefficient", False) else 1.0)

    def _pass(self, it, batch, kind, perms):
        """Pass ``it`` over ``batch`` in one persistent launch, in the order perms[it] if given, else the reference's
        DataLoader order (host RNG) or a device permutation."""
        S, B = batch.count, self.cfg["batch_size"]
        if perms is not None:
            perm = perms[it].to(self.device)
        elif self.host_rng:
            perm = reference_order(S).to(self.device)
        else:
            perm = torch.randperm(S, device=self.device)
        pol, adam = self.policy, self.adam
        args = (C.byref(pol.dims), L.ptr(pol.flat), L.ptr(adam.m), L.ptr(adam.v), L.ptr(adam.t), C.byref(batch), L.ptr(perm),
                perm.numel(), B, kind, C.byref(self.hp), L.ptr(self.ctrl))
        if self.dp is None:
            L.call("spo_pg_update", *args, L.stream())
        else:
            # ranks hold equal-sized shards; gradients are summed inside the kernel over NVLink
            comm = self.dp.comm_struct()
            L.call("spo_pg_update_dp", *args, C.byref(comm), L.stream())
            self.dp.advance((perm.numel() + B - 1) // B)


class PolicyGradientUpdate(_MinibatchUpdate):
    def __init__(self, policy, cfg, kind, epochs, host_rng, device, focops_lam=1.5, dp=None):
        if dp is not None:
            dp.broadcast(policy.flat)
            dp.setup_peer_buffers(policy.dims, device)
        super().__init__(policy, cfg, host_rng, device, dp, 3e-4, 3e-4, focops_lam, cfg["target_kl"])
        self.kind = kind
        self.sched = LinearDecay(3e-4, epochs)
        self.old_mean = None
        self.old_log_std = torch.zeros(policy.act_dim, dtype=torch.float32, device=device)

    def run(self, data, perms=None, refresh_old=True, kind=None, cup_coef=None, step_sched=True):
        """data: dict from buffer.get(lam).  Returns dict(stop_iter, kl, losses(3)).
        refresh_old=False keeps the old distribution of the previous call (tests drive the
        loop one minibatch at a time).  kind / cup_coef: run this call with another loss kind on the same
        optimizer state (CUP's projection stage, cup.py:355-404); step_sched=False leaves the actor's
        LinearLR alone (it steps once per epoch, after both stages)."""
        pol, cfg = self.policy, self.cfg
        kind = self.kind if kind is None else kind
        focops_lam_saved = self.hp.focops_lam
        if kind == L.LOSS_CUP_PROJECTION:
            self.hp.focops_lam = float(cup_coef)
        S = data["obs"].shape[0]
        if refresh_old or self.old_mean is None or self.old_mean.shape[0] != S:
            self.old_mean = _old_dist(pol, data["obs"], self.old_mean, self.old_log_std)
        old_std = None
        if kind in (L.LOSS_FOCOPS, L.LOSS_CUP_PROJECTION):
            old_std = torch.exp(self.old_log_std).expand(S, pol.act_dim).contiguous()
        batch = L.Batch(L.ptr(data["obs"]), L.ptr(data["act"]), L.ptr(data["log_prob"]), L.ptr(data["target_value_r"]),
                        L.ptr(data["target_value_c"]), L.ptr(data["adv"]), L.ptr(self.old_mean), L.ptr(old_std), S)
        self.hp.lr_actor = self.sched.lr
        self.ctrl.zero_()
        for it in range(cfg["learning_iters"]):
            self._pass(it, batch, kind, perms)
            if self.dp is None:
                L.call("spo_actor_kl", C.byref(pol.dims), L.ptr(pol.flat), L.ptr(data["obs"]), L.ptr(self.old_mean),
                       L.ptr(self.old_log_std), S, 0, cfg["target_kl"], L.ptr(self.ctrl), L.stream())
            else:
                L.call("spo_actor_kl_accumulate", C.byref(pol.dims), L.ptr(pol.flat), L.ptr(data["obs"]), L.ptr(self.old_mean),
                       L.ptr(self.old_log_std), S, L.ptr(self.ctrl), L.stream())
                kl_sum = self.ctrl.view(torch.float64)[L.CTRL_KL_SUM_F64_INDEX:L.CTRL_KL_SUM_F64_INDEX + 1]
                self.dp.all_reduce_sum(kl_sum)
                L.call("spo_kl_finalize", L.ptr(self.ctrl), float(S * self.dp.world), cfg["target_kl"], L.stream())
            if self.host_rng or perms is not None:
                # the reference stops drawing permutations once KL trips: stay in lock-step with its RNG
                if int(read_ctrl(self.ctrl)["stop"]):
                    break
        c = read_ctrl(self.ctrl)
        steps = max(int(c["steps"]), 1)
        self.hp.focops_lam = focops_lam_saved
        if step_sched:
            self.sched.step()
        return {"stop_iter": int(c["passes"]), "kl": float(c["final_kl"]),
                "loss_r": c["loss_sum"][0] / steps, "loss_c": c["loss_sum"][1] / steps, "loss_pi": c["loss_sum"][2] / steps,
                "steps": int(c["steps"])}


class CriticRegression(_MinibatchUpdate):
    """cpo.py:534-571 / trpo_lag.py:457-494: minibatch regression of the two critics
    (batch 128, lr 1e-3, 10 passes).  The joint clip (cpo.py:562) runs over policy.parameters(), but
    every fvp() call starts with policy.actor.zero_grad() (cpo.py:137, trpo_lag.py:139), which sets the
    actor's .grad to None, and nothing calls backward() on the actor afterwards: only the two critics'
    gradients enter the norm.  ``stale_actor_grad_sumsq`` stays as an explicit knob (default 0) for a
    caller whose actor does hold a gradient at this point."""

    def __init__(self, policy, cfg, host_rng, device, lr=1e-3, dp=None):
        if dp is not None and dp._peer is None:
            dp.setup_peer_buffers(policy.dims, device)
        super().__init__(policy, cfg, host_rng, device, dp, 0.0, lr, 1.5, 0.0)

    def run(self, data, stale_actor_grad_sumsq=0.0, perms=None):
        S = data["obs"].shape[0]
        batch = L.Batch(L.ptr(data["obs"]), None, None, L.ptr(data["target_value_r"]), L.ptr(data["target_value_c"]),
                        None, None, None, S)
        self.ctrl.zero_()
        self.ctrl.view(torch.float32)[L.CTRL_EXTRA_SUMSQ_F32_INDEX] = stale_actor_grad_sumsq
        for it in range(self.cfg["learning_iters"]):
            self._pass(it, batch, L.LOSS_CRITIC_ONLY, perms)
        c = read_ctrl(self.ctrl)
        steps = max(int(c["steps"]), 1)
        return {"loss_r": c["loss_sum"][0] / steps, "loss_c": c["loss_sum"][1] / steps, "steps": int(c["steps"])}


# ---------------------------------------------------------------------------------------
# CPO / TRPO-Lag actor update
# ---------------------------------------------------------------------------------------

class TrustRegionUpdate:
    """Actor step of cpo.py:351-519 / trpo_lag.py:358-442 on the libspo kernels.  The flat
    vectors (g, b, x, p, step) stay on the device; only the handful of scalars the case
    analysis needs are read back."""

    CG_ITERS, SEARCH_STEPS, STEP_FRACTION, DAMPING = 15, 15, 0.8, 0.1

    def __init__(self, policy, cfg, device, logger=None, dp=None):
        """``dp``: safepo.common.dist.DataParallel -- ranks hold disjoint env shards and identical weights; the flat
        gradients g / b, every Fisher-vector product and the line-search means are averaged over the ranks (SURVEY 8e
        exchange 3'), everything derived from them (CG vectors, the case analysis, the accepted step) is then replicated."""
        self.policy, self.cfg, self.device, self.logger, self.dp = policy, cfg, device, logger, dp
        if dp is not None:
            dp.broadcast(policy.flat)
        P = policy.n_actor
        f32 = dict(dtype=torch.float32, device=device)
        self.g, self.b, self.x, self.p, self.Fx = (torch.zeros(P, **f32) for _ in range(5))
        self.work = torch.zeros(4 * P + 8, **f32)
        self.loss = torch.zeros(1, **f32)
        self.out3 = torch.zeros(3, **f32)
        self.old_mean = None
        self.old_log_std = torch.zeros(policy.act_dim, **f32)

    def _log(self, msg, color="green"):
        if self.logger is not None:
            self.logger.log(msg, color)

    # -- kernels --
    def _grad(self, data, adv, out):
        pol = self.policy
        S = data["obs"].shape[0]
        L.call("spo_surrogate_grad", C.byref(pol.dims), L.ptr(pol.flat), L.ptr(data["obs"]), L.ptr(data["act"]),
               L.ptr(data["log_prob"]), L.ptr(adv), S, L.ptr(self.loss), L.ptr(out), L.stream())
        if self.dp is not None:
            self.dp.all_reduce_mean(out)
            self.dp.all_reduce_mean(self.loss)
        return self.loss.clone()

    def _cg(self, data, rhs, out):
        pol = self.policy
        S = data["obs"].shape[0]
        if self.dp is not None:
            # the solver split at the FVP: p = work[P:2P] -> z = work[2P:3P], averaged over the ranks, then one CG step
            P = pol.n_actor
            L.call("spo_cg_begin", C.byref(pol.dims), L.ptr(rhs), L.ptr(out), L.ptr(self.work), L.stream())
            p_vec, z_vec = self.work[P:2 * P], self.work[2 * P:3 * P]
            for _ in range(self.CG_ITERS):
                L.call("spo_fvp", C.byref(pol.dims), L.ptr(pol.flat), L.ptr(data["obs"]), S, L.ptr(p_vec), self.DAMPING,
                       L.ptr(z_vec), L.stream())
                self.dp.all_reduce_mean(z_vec)
                L.call("spo_cg_update", C.byref(pol.dims), L.ptr(out), L.ptr(self.work), 1e-10, 1e-6, L.stream())
            L.LAUNCHES["n"] += self.CG_ITERS + 1
            return
        L.call("spo_conjugate_gradient", C.byref(pol.dims), L.ptr(pol.flat), L.ptr(data["obs"]), S, L.ptr(rhs),
               self.CG_ITERS, self.DAMPING, 1e-10, 1e-6, L.ptr(out), L.ptr(self.work), L.stream())
        L.LAUNCHES["n"] += 2 * self.CG_ITERS + 1

    def _fvp(self, data, v, out):
        pol = self.policy
        S = data["obs"].shape[0]
        L.call("spo_fvp", C.byref(pol.dims), L.ptr(pol.flat), L.ptr(data["obs"]), S, L.ptr(v), self.DAMPING, L.ptr(out),
               L.stream())
        if self.dp is not None:
            self.dp.all_reduce_mean(out)

    def _eval(self, data, adv_a, adv_b):
        pol = self.policy
        S = data["obs"].shape[0]
        L.call("spo_linesearch_eval", C.byref(pol.dims), L.ptr(pol.flat), L.ptr(data["obs"]), L.ptr(data["act"]),
               L.ptr(data["log_prob"]), L.ptr(adv_a), L.ptr(adv_b), L.ptr(self.old_mean), L.ptr(self.old_log_std), S,
               L.ptr(self.out3), L.stream())
        if self.dp is not None:
            self.dp.all_reduce_mean(self.out3)
        return self.out3.cpu()

    def _old_dist(self, data):
        self.old_mean = _old_dist(self.policy, data["obs"], self.old_mean, self.old_log_std)

    # -- the steps shared by CPO, TRPO and NPG --
    def _direction(self, data, adv):
        """theta_old, g = grad mean(ratio * adv), the old distribution, x = (F + damping I)^-1 g by conjugate gradient
        and F x (cpo.py:353-372, trpo_lag.py:363-380).  Returns theta_old and the surrogate loss (device)."""
        theta_old = self.policy.actor_flat().clone()
        loss = self._grad(data, adv, self.g)
        self._old_dist(data)
        self._cg(data, self.g, self.x)
        self._fvp(data, self.x, self.Fx)
        return theta_old, loss

    def _scalars(self, loss, *extra):
        """The one device->host read of the update: [xHx, loss, |g|^2, |x|^2, *extra].  Returns them with the step
        length alpha = sqrt(2 target_kl / xHx)."""
        sc = torch.stack([torch.dot(self.x, self.Fx), loss[0], torch.dot(self.g, self.g), torch.dot(self.x, self.x),
                          *extra]).cpu()
        assert torch.isfinite(self.x).all(), "x is not finite"
        assert sc[0].item() >= 0, "xHx is negative"
        return sc, torch.sqrt(2 * self.cfg["target_kl"] / (sc[0] + 1e-8))

    def _misc(self, sc, alpha, step):
        return {"Misc/Alpha": alpha.item(), "Misc/FinalStepNorm": float(torch.norm(step)), "Misc/xHx": sc[0].item(),
                "Misc/gradient_norm": float(sc[2].sqrt()), "Misc/H_inv_g": float(sc[3].sqrt())}

    def _finish(self, theta_old, step, step_frac, acceptance, sc, alpha):
        """End of a line search: apply step_frac * step, or return to theta_old if no step was accepted (acceptance 0)."""
        if not acceptance:
            self._log("INFO: no suitable step found...")
            step = torch.zeros_like(step)
        self.policy.actor_flat().copy_(theta_old + step_frac * step)
        return {**self._misc(sc, alpha, step), "Misc/AcceptanceStep": acceptance}

    # -- CPO --
    def run_cpo(self, data, ep_costs, variant="cpo"):
        """cpo.py:351-519.  ep_costs = Jc - cost_limit (python float).
        variant="pcpo" (pcpo.py:371,392-401): projection step instead of the case analysis, optim_case 0,
        up to 200 line-search steps (pcpo.py:44)."""
        pol, kl_target = self.policy, self.cfg["target_kl"]
        theta_old, loss_r = self._direction(data, data["adv_r"])   # g = -grad(loss_pi_r) = grad mean(ratio*adv_r)
        loss_c = self._grad(data, data["adv_c"], self.b)            # b = grad mean(ratio*adv_c)
        self._cg(data, self.b, self.p)
        sc, alpha = self._scalars(loss_r, torch.dot(self.g, self.p), torch.dot(self.b, self.p), torch.dot(self.b, self.b),
                                  loss_c[0])
        xHx, r, s, bb = sc[0], sc[4], sc[5], sc[6]
        loss_reward_before, loss_cost_before = -float(sc[1]), float(sc[7])
        q = xHx
        search_steps = self.SEARCH_STEPS
        if variant == "pcpo":
            # sqrt(2 delta / (q + 1e-8)) * F x  -  max(0, (sqrt(2 delta / q) r + c) / s) * p   (F x: the reference's fvp(x))
            case, search_steps = 0, 200
            c_g = torch.sqrt(2 * kl_target / (q + 1e-8)).item()
            c_p = torch.clamp_min((torch.sqrt(2 * kl_target / q) * r + ep_costs) / s, torch.tensor(0.0)).item()
            step = c_g * self.Fx - c_p * self.p
        elif bb <= 1e-6 and ep_costs < 0:
            A_, B_, case = torch.zeros(1), torch.zeros(1), 4
        else:
            assert torch.isfinite(r).all() and torch.isfinite(s).all(), "r/s not finite"
            A_ = q - r ** 2 / (s + 1e-8)
            B_ = 2 * kl_target - ep_costs ** 2 / (s + 1e-8)
            if ep_costs < 0 and B_ < 0:
                case = 3
            elif ep_costs < 0 <= B_:
                case = 2
            elif ep_costs >= 0 and B_ >= 0:
                case = 1
                self._log("Alert! Attempting feasible recovery!", "yellow")
            else:
                case = 0
                self._log("Alert! Attempting infeasible recovery!", "red")
        if variant == "pcpo":
            pass
        elif case in (3, 4):
            nu_star, lambda_star = torch.zeros(1), 1 / (alpha + 1e-8)
            step = alpha.item() * self.x
        elif case in (1, 2):
            lambda_a, lambda_b = torch.sqrt(A_ / B_), torch.sqrt(q / (2 * kl_target))
            r_num, eps_cost = r.item(), ep_costs + 1e-8
            zero, inf = torch.as_tensor(0.0), torch.as_tensor(torch.inf)
            if ep_costs < 0:
                la, lb = torch.clamp(lambda_a, zero, r_num / eps_cost), torch.clamp(lambda_b, r_num / eps_cost, inf)
            else:
                la, lb = torch.clamp(lambda_a, r_num / eps_cost, inf), torch.clamp(lambda_b, zero, r_num / eps_cost)
            f_a = -0.5 * (A_ / (la + 1e-8) + B_ * la) - r * ep_costs / (s + 1e-8)
            f_b = -0.5 * (q / (lb + 1e-8) + 2 * kl_target * lb)
            lambda_star = la if f_a >= f_b else lb
            nu_star = torch.clamp(lambda_star * ep_costs - r, min=0) / (s + 1e-8)
            step = (1.0 / (lambda_star + 1e-8)).item() * (self.x - nu_star.item() * self.p)
        else:
            lambda_star, nu_star = torch.zeros(1), torch.sqrt(2 * kl_target / (s + 1e-8))
            step = -nu_star.item() * self.p
        step_frac, acceptance, kl = 1.0, 0, 0.0
        expected = float(torch.dot(self.g, step))
        for i in range(search_steps):
            pol.actor_flat().copy_(theta_old + step_frac * step)
            o = self._eval(data, data["adv_r"], data["adv_c"])
            loss_reward, loss_cost, kl = -float(o[0]), float(o[1]), float(o[2])
            improve, cost_diff = loss_reward_before - loss_reward, loss_cost - loss_cost_before
            self._log(f"Expected Improvement: {expected} Actual: {improve}")
            if not np.isfinite(kl):
                self._log("WARNING: KL not finite")
                continue
            if (improve < 0) if case > 1 else False:
                self._log("INFO: did not improve improve <0")
            elif cost_diff > max(-ep_costs, 0):
                self._log(f"INFO: no improve {cost_diff} > {max(-ep_costs, 0)}")
            elif kl > kl_target:
                self._log(f"INFO: violated KL constraint {kl} at step {i + 1}.")
            else:
                self._log(f"Accept step at i={i + 1}")
                acceptance = i + 1
                break
            step_frac *= self.STEP_FRACTION
        return {**self._finish(theta_old, step, step_frac, acceptance, sc, alpha),
                "Loss/Loss_actor": loss_reward_before + loss_cost_before, "Train/KL": kl, "case": case, "step_frac": step_frac}

    # -- TRPO-Lag --
    def run_trpo(self, data, advantage):
        """trpo_lag.py:363-442."""
        pol, kl_target = self.policy, self.cfg["target_kl"]
        theta_old, loss0 = self._direction(data, advantage)
        sc, alpha = self._scalars(loss0)
        loss_before = -float(sc[1])
        step = self.x * alpha.item()
        expected = float(torch.dot(self.g, step))
        step_frac, final_kl, acceptance, loss_pi = 1.0, 0.0, 0, loss_before
        for i in range(self.SEARCH_STEPS):
            pol.actor_flat().copy_(theta_old + step_frac * step)
            o = self._eval(data, advantage, None)
            loss_pi, kl = -float(o[0]), float(o[2])
            improve = loss_before - loss_pi
            self._log(f"Expected Improvement: {expected} Actual: {improve}")
            if not np.isfinite(loss_pi):
                self._log("WARNING: loss_pi not finite")
            elif improve < 0:
                self._log("INFO: did not improve improve <0")
            elif kl > kl_target:
                self._log("INFO: violated KL constraint.")
            else:
                acceptance, final_kl = i + 1, kl
                self._log(f"Accept step at i={acceptance}")
                break
            step_frac *= 0.8
        return {**self._finish(theta_old, step, step_frac, acceptance, sc, alpha),
                "Loss/Loss_actor": loss_pi, "Train/KL": final_kl, "step_frac": step_frac}

    def run_npg(self, data, advantage):
        """natural_pg.py:355-387 / rcpo.py: the TRPO direction at full length, no line search."""
        theta_old, loss0 = self._direction(data, advantage)
        sc, alpha = self._scalars(loss0)
        step = self.x * alpha.item()
        self.policy.actor_flat().copy_(theta_old + step)
        o = self._eval(data, advantage, None)           # KL(old || new).mean() at the new parameters
        return {**self._misc(sc, alpha, step), "Loss/Loss_actor": -float(sc[1]), "Train/KL": float(o[2])}


# ---------------------------------------------------------------------------------------
# main() of the two families
# ---------------------------------------------------------------------------------------

def make_env(args):
    if getattr(args, "env", "synthetic") == "mujoco":
        from safepo.common.env import make_sa_mujoco_env  # needs safety_gymnasium on the host
        return make_sa_mujoco_env(num_envs=args.num_envs, env_id=args.task, seed=args.seed)
    from safepo.common.synthetic_env import make_synthetic_env
    return make_synthetic_env(args.num_envs, args.task, args.seed, episode_len=getattr(args, "episode_len", 1000))


def _setup(args, config, env, quiet):
    """Seeding, device, env, policy, buffer, logger and rollout loop of every main() (ppo_lag.py:69-147).
    Returns (device, policy, buffer, logger, rollout); the rollout holds the env."""
    seed_all(args.seed)
    if args.device != "cuda":
        raise L.SpoError("this build has no CPU path: run with --device cuda")
    device = torch.device(f"cuda:{args.device_id}")
    torch.cuda.set_device(device)
    if env is None:
        env, obs_space, act_space = make_env(args)
    else:
        obs_space, act_space = env.observation_space, env.action_space
    policy = ActorVCritic(obs_space.shape[0], act_space.shape[0], config["hidden_sizes"]).to(device)
    buffer = VectorizedOnPolicyBuffer(obs_space, act_space, size=args.steps_per_epoch // args.num_envs, device=device,
                                      num_envs=args.num_envs, gamma=config["gamma"], gae_mode=getattr(args, "gae", "scan"))
    logger = EpochLogger(args.log_dir, seed=str(args.seed), verbose=not quiet, use_tensorboard=not quiet)
    logger.save_config({**vars(args), **config})
    logger.setup_torch_saver(policy.actor)
    logger.log("Start with training.")
    roll_cls = DeviceTapeRollout if getattr(args, "resident_env", False) else Rollout
    return device, policy, buffer, logger, roll_cls(env, policy, buffer, logger, args, device)


def _mean_episode_cost(logger, dp, device):
    return logger.get_stats("Metrics/EpCost") if dp is None else dp.mean_episode_cost(logger, device=device)


def _log_epoch(logger, roll, args, epoch, train, t_roll, t_upd, data, misc=()):
    """One row of progress.csv once an episode has finished since the last row: the episode metrics, Train/Epoch,
    Train/TotalSteps, the family's ``train`` columns (value None: the mean of the stored values), the losses, timings and
    mean advantages, then the ``misc`` columns.  Checkpoints the actor and the observation statistics at the first epoch
    and every 100th."""
    if logger.logged:
        return
    for k in ("Metrics/EpRet", "Metrics/EpCost", "Metrics/EpLen"):
        logger.log_tabular(k)
    logger.log_tabular("Train/Epoch", epoch + 1)
    logger.log_tabular("Train/TotalSteps", (epoch + 1) * args.steps_per_epoch)
    for k, v in train.items():
        logger.log_tabular(k, v)
    for k in ("Loss/Loss_reward_critic", "Loss/Loss_cost_critic", "Loss/Loss_actor"):
        logger.log_tabular(k)
    logger.log_tabular("Time/Rollout", t_roll)
    logger.log_tabular("Time/Update", t_upd)
    logger.log_tabular("Time/Total", t_roll + t_upd)
    logger.log_tabular("Value/RewardAdv", data["adv_r"].mean().item())
    logger.log_tabular("Value/CostAdv", data["adv_c"].mean().item())
    for k in misc:
        logger.log_tabular(k)
    logger.dump_tabular()
    if (epoch + 1) % 100 == 0 or epoch == 0:
        logger.torch_save(itr=epoch)
        logger.save_state({"Normalizer": _normalizer_state(roll)}, itr=epoch)


def _multiplier_columns(lagrange):
    return {} if lagrange is None else {"Train/LagragianMultiplier": lagrange.lagrangian_multiplier}


def run_trust_region(args, config, algo, env=None, max_epochs=None, quiet=False, dp=None):
    """main() of cpo.py / trpo_lag.py and their siblings (TR_ALGOS).
    ``dp``: a safepo.common.dist.DataParallel when launched one process per GPU (envs sharded; g, b, every FVP result and
    the line-search means averaged over the ranks; the critics' gradients summed inside the update kernel)."""
    method, multiplier, logs_acceptance = TR_ALGOS[algo]
    device, policy, buffer, logger, roll = _setup(args, config, env, quiet)
    lagrange = None if multiplier is None else multiplier(args)
    trust = TrustRegionUpdate(policy, config, device, logger=None if quiet else logger, dp=dp)
    critics = CriticRegression(policy, config, roll.host_rng, device, dp=dp)
    red = None if dp is None else dp.all_reduce_sum
    misc = ("Misc/Alpha", "Misc/FinalStepNorm", "Misc/xHx", "Misc/gradient_norm", "Misc/H_inv_g") + \
        (("Misc/AcceptanceStep",) if logs_acceptance else ())
    timings = []
    epochs = args.total_steps // args.steps_per_epoch
    for epoch in range(epochs if max_epochs is None else min(epochs, max_epochs)):
        t_roll = roll.run(buffer.size)
        t1 = time.time()
        if lagrange is not None:
            lagrange.update_lagrange_multiplier(_mean_episode_cost(logger, dp, device))
        # without a multiplier the advantage is adv_r itself (trpo.py:361): (adv_r - 0 * adv_c) / 1, exactly
        data = buffer.get(0.0 if lagrange is None else lagrange.lagrangian_multiplier, all_reduce=red)
        if method == "trpo":
            res = trust.run_trpo(data, data["adv"])
        elif method == "npg":
            res = trust.run_npg(data, data["adv"])
        else:
            res = trust.run_cpo(data, _mean_episode_cost(logger, dp, device) - args.cost_limit, variant=method)
        cres = critics.run(data)
        torch.cuda.synchronize()
        t_upd = time.time() - t1
        timings.append({"rollout": t_roll, "update": t_upd, "steps": cres["steps"], "acceptance": res.get("Misc/AcceptanceStep")})
        logger.store(**{k: v for k, v in res.items() if k.startswith(("Misc/", "Loss/", "Train/"))})
        logger.store(**{"Loss/Loss_reward_critic": cres["loss_r"], "Loss/Loss_cost_critic": cres["loss_c"]})
        _log_epoch(logger, roll, args, epoch, {**_multiplier_columns(lagrange), "Train/KL": None}, t_roll, t_upd, data, misc)
    logger.close()
    return policy, logger, timings, {"rollout": roll, "trust": trust, "critics": critics, "lagrange": lagrange, "buffer": buffer}


def run_policy_gradient(args, config, algo, env=None, max_epochs=None, quiet=False, dp=None):
    """main() of ppo_lag.py / focops.py and their siblings (PG_ALGOS).  Returns (policy, logger, per-epoch timing list, parts).
    ``dp``: a safepo.common.dist.DataParallel when launched one process per GPU."""
    kind, multiplier = PG_ALGOS[algo]
    device, policy, buffer, logger, roll = _setup(args, config, env, quiet)
    lagrange = None if multiplier is None else multiplier(args)
    epochs = args.total_steps // args.steps_per_epoch
    upd = PolicyGradientUpdate(policy, config, kind, epochs, roll.host_rng, device, dp=dp)
    red = None if dp is None else dp.all_reduce_sum
    timings = []
    for epoch in range(epochs if max_epochs is None else min(epochs, max_epochs)):
        t_roll = roll.run(buffer.size)
        t1 = time.time()
        ep_costs = _mean_episode_cost(logger, dp, device)
        if lagrange is not None:
            lagrange.update_lagrange_multiplier(ep_costs)
        # without a multiplier the advantage is adv_r itself (ppo.py:272): (adv_r - 0 * adv_c) / 1, exactly
        lam = lagrange.lagrangian_multiplier if lagrange is not None else 0.0
        if algo == "cup":
            # cup.py:284: the first stage is plain PPO on adv_r; the multiplier enters the projection stage only
            data = buffer.get(0.0, all_reduce=red)
            res = upd.run(data, step_sched=False)
            coef = (1 - config["gamma"] * CUP_LAMBDA) / (1 - config["gamma"])
            res2 = upd.run({**data, "adv": data["adv_c"].reshape(-1)}, kind=L.LOSS_CUP_PROJECTION, cup_coef=lam * coef)
            stop_iters = {"Train/StopIter": res["stop_iter"], "Train/SeconStageStopIter": res2["stop_iter"]}
            res["kl"], res["steps"] = res2["kl"], res["steps"] + res2["steps"]
        else:
            data = buffer.get(lam, all_reduce=red)
            res = upd.run(data)
            stop_iters = {"Train/StopIter": res["stop_iter"]}
        torch.cuda.synchronize()
        t_upd = time.time() - t1
        timings.append({"rollout": t_roll, "update": t_upd, "stop_iter": res["stop_iter"], "steps": res["steps"]})
        logger.store(**{"Loss/Loss_reward_critic": res["loss_r"], "Loss/Loss_cost_critic": res["loss_c"],
                        "Loss/Loss_actor": res["loss_pi"]})
        train = {**stop_iters, "Train/KL": res["kl"], **_multiplier_columns(lagrange), "Train/LR": upd.sched.lr}
        _log_epoch(logger, roll, args, epoch, train, t_roll, t_upd, data)
    logger.close()
    return policy, logger, timings, {"rollout": roll, "update": upd, "lagrange": lagrange, "buffer": buffer}
