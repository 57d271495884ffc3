"""MAPPO-Lag on the device: the per-iteration part of the reference's ``Runner`` (safepo/multi_agent/mappolag.py:402-504,
583-597: ``collect`` / ``insert`` / ``compute`` / ``train``) around ``MultiAgentNets`` / ``MultiAgentTrainer``
(safepo/common/ma_model.py) and ``SeparatedReplayBuffer`` (safepo/common/buffer.py).  One runner holds all agents of one
GPU's environments; the environments themselves (Isaac Gym / multi-agent MuJoCo in the reference) are the caller's: it
feeds ``insert`` with what ``envs.step`` returned.  Random draws can be injected (``eps`` in ``collect``, ``agent_order`` and
``perms`` in ``train``) so that a run can be replayed against the oracle; by default they come from the device generator.
There is no CPU path."""
from __future__ import annotations

import argparse
import os
import time

import torch

from safepo.common.buffer import SeparatedReplayBuffer
from safepo.common.ma_model import MultiAgentNets, MultiAgentTrainer


class Runner:
    trainer_cls = MultiAgentTrainer          # the per-agent trainer (macpo.Runner swaps in MACPOTrainer)

    def __init__(self, nets, config, obs_dim, share_obs_dim, act_dim):
        """``nets``: one MultiAgentNets per agent (all on the same device)."""
        self.config, self.num_agents = dict(config), len(nets)
        self.nets = list(nets)
        self.device = nets[0].device
        self.trainer = [self.trainer_cls(n, self.config) for n in self.nets]
        self.buffer = [SeparatedReplayBuffer(self.config, obs_dim, share_obs_dim, act_dim, self.device) for _ in self.nets]
        self.T, self.N = int(config["episode_length"]), int(config["n_rollout_threads"])

    def _dev(self, x):
        return torch.as_tensor(x).to(self.device)

    def warmup(self, obs, share_obs):
        """obs [N, agents, D], share_obs [N, agents, DS] of the reset (mappolag.py:396-405)."""
        obs, share_obs = self._dev(obs), self._dev(share_obs)
        for a, b in enumerate(self.buffer):
            b.share_obs[0].copy_(share_obs[:, a])
            b.obs[0].copy_(obs[:, a])

    @torch.no_grad()
    def collect(self, step, eps=None):
        """get_actions of every agent on its buffer's step-th observations (mappolag.py:408-445): values [N, agents, 1], the
        per-agent lists of actions / per-dimension log-probs, cost predictions [N, agents, 1]."""
        values, actions, logps, cost_preds = [], [], [], []
        for a, nets in enumerate(self.nets):
            b = self.buffer[a]
            e = None if eps is None else self._dev(eps[a]).contiguous()
            v, act, lp, cp = nets.get_actions(b.share_obs[step], b.obs[step], eps=e)
            values.append(v), actions.append(act), logps.append(lp), cost_preds.append(cp)
        return torch.stack(values, dim=1), actions, logps, torch.stack(cost_preds, dim=1)

    @torch.no_grad()
    def insert(self, obs, share_obs, rewards, costs, dones, values, actions, action_log_probs, cost_preds):
        """One environment step into every agent's buffer (mappolag.py:447-487): an environment whose agents are all done
        gets mask 0 (and active mask 1); an agent done alone gets active mask 0."""
        obs, share_obs, rewards, costs = self._dev(obs), self._dev(share_obs), self._dev(rewards), self._dev(costs)
        dones = self._dev(dones).bool()
        dones_env = torch.all(dones, dim=1)
        masks = torch.ones(self.N, self.num_agents, 1, device=self.device)
        masks[dones_env] = 0.0
        active_masks = torch.ones(self.N, self.num_agents, 1, device=self.device)
        active_masks[dones] = 0.0
        active_masks[dones_env] = 1.0
        for a, b in enumerate(self.buffer):
            b.insert(share_obs[:, a], obs[:, a], actions[a], action_log_probs[a], values[:, a], rewards[:, a], masks[:, a],
                     active_masks[:, a], costs=costs[:, a], cost_preds=cost_preds[:, a])

    @torch.no_grad()
    def compute(self):
        """Bootstrap values of the last observations and the masked GAE returns of both critics (mappolag.py:583-597)."""
        for nets, b, tr in zip(self.nets, self.buffer, self.trainer):
            mean, sd = tr.popart_mean_sqrt_var()
            b.compute_returns(nets._value(nets.critic, b.share_obs[-1]), mean, sd)
            b.compute_cost_returns(nets._value(nets.cost_critic, b.share_obs[-1]), mean, sd)

    def train(self, agent_order=None, perms=None, collect_outputs=False):
        """Sequential update of the agents in a random order; every updated agent multiplies the importance ratio of its new
        against its old policy into the factor the following agents see (mappolag.py:489-519)."""
        T, N = self.T, self.N
        factor = torch.ones(T, N, 1, device=self.device)
        order = torch.randperm(self.num_agents).tolist() if agent_order is None else [int(a) for a in agent_order]
        outs = {}
        for a in order:
            b, tr, nets = self.buffer[a], self.trainer[a], self.nets[a]
            A = b.actions.shape[-1]
            b.update_factor(factor)
            flat_obs, flat_act = b.obs[:-1].reshape(-1, b.obs.shape[-1]), b.actions.reshape(-1, A)
            with torch.no_grad():
                old_lp = nets.evaluate_actions(flat_obs, flat_act)
            outs[a] = tr.train(b, perms=None if perms is None else perms[a])
            with torch.no_grad():
                new_lp = nets.evaluate_actions(flat_obs, flat_act)
                factor = factor * torch.prod(torch.exp(new_lp - old_lp).reshape(T, N, A), dim=-1, keepdim=True)
            b.after_update()
        return outs if collect_outputs else order

    def _agent_log(self, a, out):
        """The logged values of agent a's last update (mappolag.py:362-373)."""
        value_loss, critic_norm, policy_loss, entropy, actor_norm, imp, cost_loss, cost_norm = out
        return {f"Loss/Loss_reward_critic/agent{a}": float(value_loss), f"Loss/Loss_cost_critic/agent{a}": float(cost_loss),
                f"Loss/Loss_actor/agent{a}": float(policy_loss), f"Misc/Entropy/agent{a}": float(entropy),
                f"Misc/Ratio/agent{a}": float(imp.mean()), f"Misc/Lagrange/agent{a}": float(self.trainer[a].lamda_lagr)}

    def return_aver_cost(self, aver_episode_costs):
        for b in self.buffer:
            b.return_aver_insert(aver_episode_costs)

    def run(self, envs, iterations, logger=None):
        """The training loop of the reference's Runner.run (mappolag.py:300-373) for ``iterations`` iterations of ``episode_length``
        steps: ``envs.reset() -> (obs [N, agents, D], share_obs [N, agents, DS], _)``, ``envs.step(actions) -> (obs, share_obs,
        rewards [N, agents, 1], costs [N, agents, 1], dones [N, agents], infos, _)`` with device tensors; the per-environment
        episode sums live on the device, nothing is read back inside an iteration except the PopArt statistics in compute()/train()
        and the logged scalars at its end.  Returns the list of per-iteration log rows."""
        obs, share_obs, _ = envs.reset()
        self.warmup(obs, share_obs)
        ep_rew = torch.zeros(self.N, device=self.device)
        ep_cost = torch.zeros(self.N, device=self.device)
        rows, start = [], time.time()
        for it in range(int(iterations)):
            done_rew, done_cost = [], []
            for step in range(self.T):
                values, actions, logps, cost_preds = self.collect(step)
                obs, share_obs, rewards, costs, dones, _infos, _ = envs.step(actions)
                dones_env = torch.all(self._dev(dones).bool(), dim=1)
                ep_rew += torch.mean(self._dev(rewards), dim=1).flatten()
                ep_cost += torch.mean(self._dev(costs), dim=1).flatten()
                done_rew.append(ep_rew[dones_env].clone())
                done_cost.append(ep_cost[dones_env].clone())
                ep_rew[dones_env] = 0
                ep_cost[dones_env] = 0
                self.insert(obs, share_obs, rewards, costs, dones, values, actions, logps, cost_preds)
            self.compute()
            outs = self.train(collect_outputs=True)
            row = {"Train/Epoch": it, "Train/TotalSteps": (it + 1) * self.T * self.N}
            finished_rew, finished_cost = torch.cat(done_rew), torch.cat(done_cost)
            if finished_rew.numel():
                row["Metrics/EpRet"] = float(finished_rew.mean())
                row["Metrics/EpCost"] = float(finished_cost.mean())
                self.return_aver_cost(finished_cost.mean())          # mappolag.py:349-351
            for a, out in outs.items():                              # the reference logs the last update of every agent's train()
                row.update(self._agent_log(a, out))
            row["Time/Total"] = time.time() - start
            row["Time/FPS"] = int(row["Train/TotalSteps"] / max(row["Time/Total"], 1e-9))
            rows.append(row)
            if logger is not None:
                for k, v in row.items():
                    logger.log_tabular(k, v)
                logger.dump_tabular()
        return rows


def init_state(in_dim, hidden_size, layer_N, head, act_dim=0, std_x_coef=1.0, actor_gain=0.01, generator=None):
    """Random weights of one MultiAgentActor / MultiAgentCritic in the reference's layout and initialisation (mlp.py:27-38: orthogonal
    with the ReLU gain, zero biases; distributions.py:21-36: fc_mean orthogonal with gain 0.01, log_std = std_x_coef; model.py:336-339:
    v_out orthogonal) -- there is no checkpoint to load offline."""
    import torch.nn as nn

    def ortho(rows, cols, gain):
        w = torch.empty(rows, cols)
        nn.init.orthogonal_(w, gain=gain, generator=generator)
        return w
    relu_gain = nn.init.calculate_gain("relu")
    st = {"base.feature_norm.weight": torch.ones(in_dim), "base.feature_norm.bias": torch.zeros(in_dim)}
    dims = [in_dim] + [hidden_size] * (1 + layer_N)
    for li, name in enumerate(["fc1"] + [f"fc2.{i}" for i in range(layer_N)]):
        st[f"base.mlp.{name}.0.weight"] = ortho(hidden_size, dims[li], relu_gain)
        st[f"base.mlp.{name}.0.bias"] = torch.zeros(hidden_size)
        st[f"base.mlp.{name}.2.weight"] = torch.ones(hidden_size)
        st[f"base.mlp.{name}.2.bias"] = torch.zeros(hidden_size)
    if head == "actor":
        st["act.action_out.log_std"] = torch.ones(act_dim) * std_x_coef
        st["act.action_out.fc_mean.weight"] = ortho(act_dim, hidden_size, actor_gain)
        st["act.action_out.fc_mean.bias"] = torch.zeros(act_dim)
    else:
        st["v_out.weight"] = ortho(1, hidden_size, 1.0)
        st["v_out.bias"] = torch.zeros(1)
    return st


# the yaml's values (safepo/multi_agent/marl_cfg/mappolag/config.yaml) that this path reads
DEFAULT_CONFIG = dict(episode_length=8, n_rollout_threads=1024, hidden_size=512, layer_N=2, gamma=0.96, gae_lambda=0.95, learning_iters=5,
                      num_mini_batch=1, actor_lr=9e-5, critic_lr=5e-3, opti_eps=1e-5, weight_decay=0.0, clip_param=0.2, huber_delta=10.0,
                      entropy_coef=0.0, max_grad_norm=10.0, cost_limit=25.0, lagrangian_coef_rate=1e-5, value_loss_coef=1.0, lamda_lagr=0.78,
                      std_x_coef=1.0, std_y_coef=0.5, actor_gain=0.01)


def main(argv=None):
    """`python -m safepo.multi_agent.mappolag --env synthetic`: MAPPO-Lag on a synthetic multi-agent stream of config 5's shape (the
    reference's Isaac-Gym / multi-agent MuJoCo environments are not installable offline)."""
    from safepo.common.logger import EpochLogger
    from safepo.common.synthetic_env import SyntheticMultiAgentEnv
    ap = argparse.ArgumentParser()
    ap.add_argument("--env", default="synthetic", choices=("synthetic",))
    ap.add_argument("--num-envs", type=int, default=1024)
    ap.add_argument("--num-agents", type=int, default=2)
    ap.add_argument("--obs-dim", type=int, default=398)
    ap.add_argument("--share-obs-dim", type=int, default=398)
    ap.add_argument("--act-dim", type=int, default=20)
    ap.add_argument("--hidden-size", type=int, default=512)
    ap.add_argument("--iterations", type=int, default=10)
    ap.add_argument("--episode-len", type=int, default=64, help="steps after which the synthetic environments finish an episode")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--device", default="cuda:0")
    ap.add_argument("--log-dir", default=os.path.join("runs", "synthetic", "mappolag", "seed0"))
    args = ap.parse_args(argv)
    cfg = dict(DEFAULT_CONFIG, n_rollout_threads=args.num_envs, hidden_size=args.hidden_size)
    g = torch.Generator().manual_seed(args.seed)
    nets = []
    for _ in range(args.num_agents):
        nets.append(MultiAgentNets(init_state(args.obs_dim, cfg["hidden_size"], cfg["layer_N"], "actor", args.act_dim, cfg["std_x_coef"], cfg["actor_gain"], g),
                                   init_state(args.share_obs_dim, cfg["hidden_size"], cfg["layer_N"], "critic", generator=g),
                                   init_state(args.share_obs_dim, cfg["hidden_size"], cfg["layer_N"], "critic", generator=g),
                                   args.device, layer_N=cfg["layer_N"], std_x_coef=cfg["std_x_coef"], std_y_coef=cfg["std_y_coef"]))
    runner = Runner(nets, cfg, args.obs_dim, args.share_obs_dim, args.act_dim)
    envs = SyntheticMultiAgentEnv(args.num_envs, args.num_agents, args.obs_dim, args.share_obs_dim, args.act_dim, args.episode_len, args.seed,
                                  runner.device)
    logger = EpochLogger(args.log_dir, seed=args.seed, use_tensorboard=False)
    rows = runner.run(envs, args.iterations, logger=logger)
    logger.close()
    return rows


__all__ = ["Runner", "MultiAgentNets", "MultiAgentTrainer", "SeparatedReplayBuffer", "init_state", "DEFAULT_CONFIG", "main"]


if __name__ == "__main__":
    main()
