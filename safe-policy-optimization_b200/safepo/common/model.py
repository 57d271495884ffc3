"""ActorVCritic on a packed device buffer, evaluated by libspo kernels.

Drop-in for the classes of the reference's safepo/common/model.py:30-170 (same class,
attribute and state_dict names, same construction-time RNG consumption), but the three
MLPs are not evaluated by torch: ``step`` is one fused CUDA launch
(``spo_policy_step``: three MLP forwards + Gaussian sample + log-prob [+ the write into
the rollout buffer]) and the parameters of all three nets are views into ONE flat fp32
device buffer laid out as include/spo.h describes (actor first, log_std first inside the
actor -- the flat vector CPO/TRPO work on, cpo.py:70-78).

No autograd: gradients are produced by the fused update kernels (spo_pg_update,
spo_surrogate_grad), which is how the shipped trainers use these classes.
"""
from __future__ import annotations

import ctypes as C
import math

import torch
import torch.nn as nn
from torch.distributions import Normal

from safepo import _lib as L

_NETS = ("actor", "reward_critic", "cost_critic")  # packed order (include/spo.h)


def build_mlp_network(sizes):
    """tanh MLP with identity output (reference model.py:30-48).  Draw order per layer:
    nn.Linear's default init, then a second kaiming-uniform(a=sqrt 5) over the weight --
    kept so that a seed produces the reference's initial weights."""
    mods = []
    last = len(sizes) - 2
    for j, (fan_in, fan_out) in enumerate(zip(sizes[:-1], sizes[1:])):
        lin = nn.Linear(fan_in, fan_out)
        nn.init.kaiming_uniform_(lin.weight, a=math.sqrt(5))
        mods.extend((lin, nn.Tanh() if j < last else nn.Identity()))
    return nn.Sequential(*mods)


class _PackedNet(nn.Module):
    """Common part of Actor / VCritic: knows where it lives in the packed buffer."""

    def __init__(self):
        super().__init__()
        self._owner = None  # ActorVCritic (set by the owner; plain attribute, not a submodule)

    def _bind(self, owner):
        object.__setattr__(self, "_owner", owner)

    def _require_owner(self):
        if self._owner is None or self._owner.flat is None:
            raise L.SpoError("this network is not attached to a packed ActorVCritic on a CUDA device "
                             "(construct ActorVCritic(...).to('cuda'); there is no CPU path)")
        return self._owner


class Actor(_PackedNet):
    """Gaussian policy head: ``mean`` MLP + state-independent ``log_std`` (model.py:51-81)."""

    def __init__(self, obs_dim, act_dim, hidden_sizes=[64, 64]):
        super().__init__()
        self.mean = build_mlp_network([obs_dim] + list(hidden_sizes) + [act_dim])
        self.log_std = nn.Parameter(torch.zeros(act_dim), requires_grad=True)

    def forward(self, obs):
        own = self._require_owner()
        mean = own.actor_mean(obs)
        return Normal(mean, torch.exp(self.log_std.detach()))


class VCritic(_PackedNet):
    """State-value head (model.py:84-108)."""

    def __init__(self, obs_dim, hidden_sizes=[64, 64]):
        super().__init__()
        self.critic = build_mlp_network([obs_dim] + list(hidden_sizes) + [1])
        self._which = None

    def forward(self, obs):
        own = self._require_owner()
        v_r, v_c = own.values(obs)
        return v_r if self._which == "reward_critic" else v_c


class ActorVCritic(nn.Module):
    """Actor + reward critic + cost critic (model.py:111-170) over one packed buffer."""

    def __init__(self, obs_dim, act_dim, hidden_sizes=[64, 64]):
        super().__init__()
        hidden_sizes = list(hidden_sizes)
        if hidden_sizes != [64, 64]:
            raise L.SpoError(f"hidden_sizes={hidden_sizes}: libspo implements the reference's MuJoCo default [64, 64] only")
        self.obs_dim, self.act_dim = int(obs_dim), int(act_dim)
        # registration / construction order of the reference (model.py:133-135) => same RNG stream
        self.reward_critic = VCritic(obs_dim, hidden_sizes)
        self.cost_critic = VCritic(obs_dim, hidden_sizes)
        self.actor = Actor(obs_dim, act_dim, hidden_sizes)
        self.reward_critic._which, self.cost_critic._which = "reward_critic", "cost_critic"
        for m in (self.reward_critic, self.cost_critic, self.actor):
            m._bind(self)
        self.flat = None           # packed fp32 parameters on the device
        self.dims = L.dims(obs_dim, act_dim, 64)
        self.n_actor, self.n_critic, self.n_total = 0, 0, 0
        self._philox_seed, self._philox_offset = None, 0

    # ---- packing -------------------------------------------------------------------------
    def _named(self, net):
        mod = getattr(self, net)
        # named_parameters order: actor -> log_std, mean.0.weight, mean.0.bias, ...
        return list(mod.named_parameters())

    def _pack(self, device):
        if device.type != "cuda":
            self.flat = None
            return
        self.n_actor, self.n_critic, self.n_total = L.param_count(self.dims)
        flat = torch.empty(self.n_total, dtype=torch.float32, device=device)
        off = 0
        with torch.no_grad():
            for net in _NETS:
                for _, prm in self._named(net):
                    n = prm.numel()
                    view = flat[off:off + n].view(prm.shape)
                    view.copy_(prm.data)
                    prm.data = view
                    off += n
        assert off == self.n_total, (off, self.n_total)
        o = L.param_offsets(self.dims, 0)
        assert o["log_std"] == 0 and o["w1"] == self.act_dim
        self.flat = flat

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        dev = next(self.parameters()).device
        self._pack(dev)
        return out

    def actor_flat(self):
        """View of the actor slice == get_flat_params_from(policy.actor) (cpo.py:70-78)."""
        return self.flat[: self.n_actor]

    # ---- evaluation ------------------------------------------------------------------------
    def _check(self, obs):
        if self.flat is None:
            raise L.SpoError("ActorVCritic is not on a CUDA device: call .to('cuda') (no CPU path)")
        if obs.dtype != torch.float32 or not obs.is_cuda:
            raise L.SpoError("obs must be a float32 CUDA tensor")
        single = obs.dim() == 1
        o2 = obs.reshape(1, -1) if single else obs
        if o2.shape[-1] != self.obs_dim:
            raise L.SpoError(f"obs has {o2.shape[-1]} features, expected {self.obs_dim}")
        return o2.contiguous(), single

    def step(self, obs, deterministic=False, eps=None, store=None, outputs=True):
        """(action, log_prob, value_r, value_c) for ``obs`` of shape [N,D] or [D]
        (model.py:149-170).  ``eps`` [N,A]: standard-normal draws to use instead of the
        in-kernel Philox stream (parity with a host generator).  ``store=(rollout_struct, t)``
        additionally writes the transition into slot t of a VectorizedOnPolicyBuffer;
        ``outputs=False`` (only with ``store``) skips the separate output tensors."""
        o2, single = self._check(obs)
        n = o2.shape[0]
        dev = o2.device
        if outputs or store is None:
            act = torch.empty(n, self.act_dim, dtype=torch.float32, device=dev)
            logp = torch.empty(n, dtype=torch.float32, device=dev)
            v_r = torch.empty(n, dtype=torch.float32, device=dev)
            v_c = torch.empty(n, dtype=torch.float32, device=dev)
        else:
            act = logp = v_r = v_c = None
        if eps is not None:
            eps = eps.reshape(n, self.act_dim).to(device=dev, dtype=torch.float32).contiguous()
        if self._philox_seed is None:
            self._philox_seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
        self._philox_offset += 1
        st, t = (C.byref(store[0]), int(store[1])) if store is not None else (None, 0)
        L.call("spo_policy_step", C.byref(self.dims), L.ptr(self.flat), L.ptr(o2), L.ptr(eps),
               self._philox_seed, self._philox_offset, int(bool(deterministic)), n,
               L.ptr(act), L.ptr(logp), L.ptr(v_r), L.ptr(v_c), st, t, L.stream())
        if act is None:
            return None
        if single:
            return act[0], logp[0], v_r[0], v_c[0]
        return act, logp, v_r, v_c

    def values(self, obs):
        o2, single = self._check(obs)
        n = o2.shape[0]
        v_r = torch.empty(n, dtype=torch.float32, device=o2.device)
        v_c = torch.empty(n, dtype=torch.float32, device=o2.device)
        L.call("spo_critic_values", C.byref(self.dims), L.ptr(self.flat), L.ptr(o2), n, L.ptr(v_r), L.ptr(v_c),
               L.stream())
        return (v_r[0], v_c[0]) if single else (v_r, v_c)

    def actor_mean(self, obs):
        o2, single = self._check(obs)
        n = o2.shape[0]
        mean = torch.empty(n, self.act_dim, dtype=torch.float32, device=o2.device)
        L.call("spo_actor_forward", C.byref(self.dims), L.ptr(self.flat), L.ptr(o2), n, L.ptr(mean), L.stream())
        return mean[0] if single else mean

    def forward(self, obs):
        return self.step(obs)
