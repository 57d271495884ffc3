"""MACPO on the device: the reference's multi-agent constrained trust-region method (safepo/multi_agent/macpo.py), the
multi-agent counterpart of CPO.  The runner is MAPPO-Lag's (collect / insert / compute / train with the cross-agent factor,
macpo.py:584-688 are the same methods) around ``MACPOTrainer`` (safepo/common/ma_model.py), which replaces the clipped
surrogate and the Lagrange multiplier by one constrained natural-gradient step per agent and iteration.  There is no CPU path."""
from __future__ import annotations

import argparse
import os

import torch

from safepo.common.ma_model import MACPOTrainer, MultiAgentNets
from safepo.multi_agent import mappolag
from safepo.multi_agent.mappolag import init_state


class Runner(mappolag.Runner):
    trainer_cls = MACPOTrainer

    def _agent_log(self, a, out):
        """macpo.py:402-414: what MACPO_Trainer.train stores per update (Loss/Loss_cost_critic is the cost surrogate there)."""
        return {f"Loss/Loss_reward_critic/agent{a}": float(out["value_loss"]), f"Loss/Loss_cost_critic/agent{a}": out["cost_loss"],
                f"Loss/Loss_actor_improve/agent{a}": out["loss_improve"], f"Loss/Loss_actor_expected_improve/agent{a}": out["expected_improve"],
                f"Misc/Reward_critic_norm/agent{a}": float(out["critic_grad_norm"]), f"Misc/Cost_critic_norm/agent{a}": float(out["cost_grad_norm"]),
                f"Misc/Entropy/agent{a}": out["dist_entropy"], f"Misc/Ratio/agent{a}": out["ratio"], f"Misc/KL/agent{a}": out["kl"]}


# the yaml's values (safepo/multi_agent/marl_cfg/macpo/config.yaml) that this path reads
DEFAULT_CONFIG = dict(episode_length=8, n_rollout_threads=1024, hidden_size=512, layer_N=2, gamma=0.96, gae_lambda=0.95, num_mini_batch=1,
                      critic_lr=5e-3, opti_eps=1e-5, weight_decay=0.0, clip_param=0.2, huber_delta=10.0, max_grad_norm=10.0, cost_limit=25.0,
                      value_loss_coef=1.0, target_kl=0.016, searching_steps=10, conjugate_gradient_iters=10, step_fraction=0.5,
                      fraction_coef=0.1, std_x_coef=1.0, std_y_coef=0.5, actor_gain=0.01)


def main(argv=None):
    """`python -m safepo.multi_agent.macpo --env synthetic`: MACPO on a synthetic multi-agent stream of config 5's shape (the
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
    ap.add_argument("--log-dir", default=os.path.join("runs", "synthetic", "macpo", "seed0"))
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


__all__ = ["Runner", "MACPOTrainer", "MultiAgentNets", "init_state", "DEFAULT_CONFIG", "main"]


if __name__ == "__main__":
    main()
