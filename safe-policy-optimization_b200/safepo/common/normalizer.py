"""On-device counterparts of the two env wrappers that sit between ``env.step`` and
``policy.step`` in the reference (safepo/common/env.py:58-80):

* :class:`SafeNormalizeObservation` -- safepo/common/wrappers.py:42-49 (gymnasium's
  ``NormalizeObservation``): running mean / variance of the observations (``obs_rms``, the object
  the reference checkpoints as "Normalizer", ppo_lag.py:381-386), float64 statistics, fp32 output.
* :class:`SafeRescaleAction` -- ``SafeRescaleAction(env, -1.0, 1.0)`` (env.py:62,76).

Both call libspo kernels (csrc/spo_envio.cu); there is no CPU path."""
import torch

from .. import _lib as L


class RunningMeanStd:
    """gymnasium.wrappers.normalize.RunningMeanStd: ``mean``, ``var`` (device float64), ``count``."""

    def __init__(self, shape, device, epsilon=1e-4):
        self.mean = torch.zeros(shape, dtype=torch.float64, device=device)
        self.var = torch.ones(shape, dtype=torch.float64, device=device)
        self.count = float(epsilon)

    def host_copy(self):
        """Picklable host object with gymnasium's RunningMeanStd surface (numpy ``mean`` / ``var``, float ``count``,
        ``update(x)``): what the trainers store as the checkpoint's "Normalizer" (ppo_lag.py:381-386)."""
        h = HostRunningMeanStd(tuple(self.mean.shape))
        h.mean, h.var, h.count = self.mean.cpu().numpy().copy(), self.var.cpu().numpy().copy(), float(self.count)
        return h

    def state_dict(self):
        return {"mean": self.mean.cpu().numpy(), "var": self.var.cpu().numpy(), "count": self.count}

    def load_state_dict(self, state):
        self.mean.copy_(torch.as_tensor(state["mean"], dtype=torch.float64))
        self.var.copy_(torch.as_tensor(state["var"], dtype=torch.float64))
        self.count = float(state["count"])


class HostRunningMeanStd:
    """Host-side (numpy) running statistics with the attribute / method names of
    gymnasium.wrappers.normalize.RunningMeanStd, which the reference pickles into its checkpoints and
    evaluate.py:56-57 re-attaches to an env whose wrapper then reads ``.mean`` / ``.var`` and calls
    ``.update(obs)``.  The merge is the parallel-variance formula gymnasium publishes (restated in oracle/envio.py)."""

    def __init__(self, shape=(), epsilon=1e-4):
        import numpy as np
        self.mean = np.zeros(shape, "float64")
        self.var = np.ones(shape, "float64")
        self.count = float(epsilon)

    def update(self, x):
        import numpy as np
        x = np.asarray(x, dtype=np.float64)
        b_mean, b_var, b_n = x.mean(axis=0), x.var(axis=0), x.shape[0]
        delta = b_mean - self.mean
        tot = self.count + b_n
        new_mean = self.mean + delta * b_n / tot
        m2 = self.var * self.count + b_var * b_n + np.square(delta) * self.count * b_n / tot
        self.mean, self.var, self.count = new_mean, m2 / tot, tot


class SafeNormalizeObservation:
    """``normalize(obs)`` = the wrapper's ``normalize``: update ``obs_rms`` with the batch of
    observations (one row per env), return ``(obs - mean) / sqrt(var + epsilon)`` as fp32."""

    def __init__(self, obs_dim, device, epsilon=1e-8):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.SpoError("SafeNormalizeObservation runs on a CUDA device only (no CPU fallback)")
        self.obs_dim = int(obs_dim)
        self.epsilon = float(epsilon)
        self.obs_rms = RunningMeanStd((self.obs_dim,), self.device)

    def normalize(self, obs, update=True, out=None):
        if obs.dim() != 2 or obs.shape[1] != self.obs_dim or obs.dtype != torch.float32:
            raise L.SpoError(f"obs must be fp32 [n, {self.obs_dim}], got {tuple(obs.shape)} {obs.dtype}")
        n = obs.shape[0]
        if out is None:
            out = torch.empty_like(obs)
        L.call("spo_obs_normalize", L.ptr(obs), n, self.obs_dim, L.ptr(self.obs_rms.mean), L.ptr(self.obs_rms.var),
               self.obs_rms.count, None, 1 if update else 0, self.epsilon, L.ptr(out), L.stream())
        if update:
            self.obs_rms.count += n
        return out


class SafeRescaleAction:
    """Policy actions in [min_action, max_action] -> the env's [low, high] box, clipped."""

    def __init__(self, low, high, device, min_action=-1.0, max_action=1.0):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.SpoError("SafeRescaleAction runs on a CUDA device only (no CPU fallback)")
        self.low = torch.as_tensor(low, dtype=torch.float32).reshape(-1).to(self.device).contiguous()
        self.high = torch.as_tensor(high, dtype=torch.float32).reshape(-1).to(self.device).contiguous()
        self.min_action, self.max_action = float(min_action), float(max_action)

    def action(self, act, out=None):
        A = self.low.numel()
        if act.dim() != 2 or act.shape[1] != A or act.dtype != torch.float32:
            raise L.SpoError(f"act must be fp32 [n, {A}], got {tuple(act.shape)} {act.dtype}")
        if out is None:
            out = torch.empty_like(act)
        L.call("spo_action_rescale", L.ptr(act), act.shape[0], A, L.ptr(self.low), L.ptr(self.high), self.min_action,
               self.max_action, L.ptr(out), L.stream())
        return out
