"""Generate tests/golden/macpo.pt from the REAL reference's MACPO (safepo/multi_agent/macpo.py), the fixture that pins
oracle/macpo_oracle.py (tests/test_macpo_cpu.py) and through it the device trainer.

Runs only where the reference is checked out (see make_golden.py, whose environment stubs it reuses):

    python tests/golden/make_golden_macpo.py          # writes tests/golden/macpo.pt

Stored, at small dimensions (obs 10, share_obs 14, act 3, hidden 32, the yaml's layer_N = 2) with one intra-op thread:
  * one fisher_vector_product on a random vector;
  * trpo_update calls from the same weights whose samples reach optim_case 0, 1, 2, 3 and 4, and one whose line search
    rejects every trial -- the case is steered with aver_episode_costs around cost_limit, a zero cost advantage (case 4) and a
    tiny target_kl with a huge fraction_coef (rejection); for each the returned scalars and the actor's state dict, the critics'
    and PopArt state once (they do not depend on the steering), and the parameter-sized intermediates of case 1;
  * two runner iterations of two agents through macpo.Runner's own collect / insert / compute / train on a stand-in self."""
from __future__ import annotations

import importlib
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as mg  # noqa: E402

RET = ("value_loss", "critic_grad_norm", "kl", "loss_improve", "expected_improve", "dist_entropy", "ratio", "cost_loss", "cost_grad_norm",
       "whether_recover_policy_value", "cost_preds_batch", "cost_returns_batch", "B_cost_loss_grad", "lam", "nu", "g_step_dir", "b_step_dir",
       "x", "action_mu", "action_std", "B_cost_loss_grad_dot")
KEEP = ("critic_lr", "opti_eps", "weight_decay", "clip_param", "huber_delta", "max_grad_norm", "cost_limit", "gamma", "gae_lambda",
        "value_loss_coef", "layer_N", "std_x_coef", "std_y_coef", "target_kl", "searching_steps", "conjugate_gradient_iters",
        "step_fraction", "fraction_coef", "episode_length", "n_rollout_threads")


class Sp:
    def __init__(self, d):
        self.shape = (d,)


class Log:
    def store(self, **kw):
        pass


def _cfg(**kw):
    import yaml
    cfg = yaml.safe_load(open(os.path.join(mg.REF, "safepo", "multi_agent", "marl_cfg", "macpo", "config.yaml")))
    cfg.update(device="cpu", algorithm_name="macpo", **kw)
    return cfg


def _perturb(pol):
    with torch.no_grad():       # move the LayerNorm affine parameters and biases off their trivial initial values
        for net in (pol.actor, pol.critic, pol.cost_critic):
            for k, v in net.state_dict().items():
                if k.endswith("bias") or ".2.weight" in k or "feature_norm" in k or k.endswith("log_std"):
                    v.add_(0.1 * torch.randn_like(v))


def _states(pol):
    return {n: {k: v.detach().clone() for k, v in getattr(pol, n).state_dict().items()} for n in ("actor", "critic", "cost_critic")}


def _instrument(tr):
    """Record the right-hand sides of the two CG solves and the actor loads of the line search (one per trial, plus one restore)."""
    rec = dict(rhs=[], loads=0)
    cg, upd = tr.conjugate_gradient, tr.update_model

    def conjugate_gradient(*a, **k):
        rec["rhs"].append(a[7].clone())
        return cg(*a, **k)

    def update_model(model, new_params):
        if model is tr.policy.actor:
            rec["loads"] += 1
        return upd(model, new_params)
    tr.conjugate_gradient, tr.update_model = conjugate_gradient, update_model
    return rec


def gen_macpo(out):
    m = importlib.import_module("safepo.multi_agent.macpo")
    threads = torch.get_num_threads()
    torch.set_num_threads(1)    # LayerNorm's backward reductions depend on the intra-op thread count (see make_golden.gen_ma_update)
    D, DS, A, N = 10, 14, 3, 24
    cfg = _cfg(n_rollout_threads=4, hidden_size=32)
    torch.manual_seed(31)
    pol = m.MACPO_Policy(cfg, Sp(D), Sp(DS), Sp(A))
    _perturb(pol)
    init = _states(pol)
    g = torch.Generator().manual_seed(32)
    obs, share = torch.randn(N, D, generator=g) * 2 + 0.5, torch.randn(N, DS, generator=g) * 3
    rnn, masks = np.zeros((N, 1, 32), dtype=np.float32), np.ones((N, 1), dtype=np.float32)
    with torch.no_grad():
        det = pol.get_actions(share, obs, rnn, rnn, masks, deterministic=True, rnn_states_cost=rnn)
        smp = pol.get_actions(share, obs, rnn, rnn, masks, deterministic=False, rnn_states_cost=rnn)
    base = dict(share_obs=share, obs=obs, actions=smp[1].clone(), value_preds=det[0].clone() + 0.1 * torch.randn(N, 1, generator=g),
                returns=torch.randn(N, 1, generator=g) * 4 + 1, old_action_log_probs=smp[2].clone() + 0.05 * torch.randn(N, A, generator=g),
                adv_targ=torch.randn(N, 1, generator=g), factor=torch.rand(N, 1, generator=g) + 0.5,
                cost_preds=det[5].clone() + 0.1 * torch.randn(N, 1, generator=g), cost_returns=torch.randn(N, 1, generator=g).abs() * 30,
                cost_adv_targ=torch.randn(N, 1, generator=g))

    # ---- one Fisher-vector product ----
    tr = m.MACPO_Trainer(cfg, pol)
    p = torch.randn(sum(v.numel() for v in pol.actor.parameters()), generator=g)
    fvp = tr.fisher_vector_product(pol.actor, obs, rnn, base["actions"], masks, None, masks, p.clone()).clone()

    # ---- trpo_update per case, every one from the initial weights ----
    cases = []
    for name, aver, overrides, zero_cost_adv in (("case0", 80.0, {}, False), ("case1", 25.5, {}, False), ("case2", 24.9, {}, False),
                                                 ("case3", 0.0, {}, False), ("case4", 10.0, {}, True),
                                                 ("rejected", 0.0, {"target_kl": 1e-6, "fraction_coef": 1e5}, False)):
        ccfg = dict(cfg, **overrides)
        for n_ in ("actor", "critic", "cost_critic"):
            getattr(pol, n_).load_state_dict(init[n_])
        pol.critic_optimizer = torch.optim.Adam(pol.critic.parameters(), lr=cfg["critic_lr"], eps=cfg["opti_eps"], weight_decay=cfg["weight_decay"])
        pol.cost_optimizer = torch.optim.Adam(pol.cost_critic.parameters(), lr=cfg["critic_lr"], eps=cfg["opti_eps"], weight_decay=cfg["weight_decay"])
        pol.config = ccfg
        tr = m.MACPO_Trainer(ccfg, pol)
        rec = _instrument(tr)
        sample = dict(base, aver_episode_costs=torch.full((N, 1), aver) + 0.01 * torch.randn(N, 1, generator=g))
        if zero_cost_adv:
            sample["cost_adv_targ"] = torch.zeros(N, 1)
        tup = (share.numpy(), obs.numpy(), rnn, rnn, sample["actions"].numpy(), sample["value_preds"], sample["returns"], masks, masks,
               sample["old_action_log_probs"], sample["adv_targ"], None, sample["factor"], sample["cost_preds"], sample["cost_returns"], rnn,
               sample["cost_adv_targ"], sample["aver_episode_costs"])
        r = tr.trpo_update(tup)
        res = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in zip(RET, r)}
        rescale = float((sample["aver_episode_costs"].mean() - cfg["cost_limit"]) * (1 - cfg["gamma"]))
        if res["b_step_dir"].dim() == 0:
            optim_case = 4
        else:
            w = float(res["whether_recover_policy_value"])
            optim_case = (3 if w < 0 else 2) if rescale < 0 else (1 if w >= 0 else 0)
        trials = rec["loads"]
        accepted = -1 if trials == ccfg["searching_steps"] + 1 else trials - 1
        vn = tr.value_normalizer
        print(name, "optim_case", optim_case, "accepted", accepted)
        for k in ("cost_preds_batch", "cost_returns_batch", "B_cost_loss_grad"):     # inputs, and b (= B_cost_loss_grad) once
            res.pop(k)
        vectors = dict(g=rec["rhs"][0], b=rec["rhs"][1], g_step_dir=res.pop("g_step_dir"), b_step_dir=res.pop("b_step_dir"), x=res.pop("x"))
        st = _states(pol)
        # the critics' updates do not depend on what steers the case: stored once, checked equal here
        critics = dict(critic=st["critic"], cost_critic=st["cost_critic"], popart=(vn.running_mean.clone(), vn.running_mean_sq.clone(), vn.debiasing_term.clone()))
        if cases:
            ref = cases[0]["critics"]
            assert all(torch.equal(ref[n_][k], critics[n_][k]) for n_ in ("critic", "cost_critic") for k in ref[n_])
            assert all(torch.equal(a, b) for a, b in zip(ref["popart"], critics["popart"]))
        cases.append(dict(name=name, cfg_overrides=overrides, sample=sample, out=res, optim_case=optim_case,
                          vectors=vectors if name == "case1" else None,    # the parameter-sized intermediates of one case (fixture size)
                          accepted=accepted, actor=st["actor"], critics=critics if not cases else None))
    torch.set_num_threads(threads)
    out["update"] = dict(cfg={k: cfg[k] for k in KEEP}, dims=(D, DS, A, N), init=init, fvp=dict(p=p, out=fvp), cases=cases)


def gen_macpo_epoch(out):
    """Two MACPO training iterations of two agents through macpo.Runner's collect / insert / compute / train (macpo.py:584-688)
    on a stand-in ``self`` (the Runner's constructor needs environments that are not installable here): T = 4 steps, 6 envs."""
    m = importlib.import_module("safepo.multi_agent.macpo")
    T, N, D, DS, A, H, NA = 4, 6, 10, 14, 3, 32, 2
    cfg = _cfg(n_rollout_threads=N, hidden_size=H, episode_length=T, env_name="synthetic")
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    torch.manual_seed(41)
    policy = [m.MACPO_Policy(cfg, Sp(D), Sp(DS), Sp(A)) for _ in range(NA)]
    for pol in policy:
        _perturb(pol)
    init = [_states(pol) for pol in policy]
    fake = types.SimpleNamespace(config=cfg, num_agents=NA, logger=Log(), policy=policy, trainer=[m.MACPO_Trainer(cfg, pol) for pol in policy],
                                 buffer=[m.SeparatedReplayBuffer(cfg, Sp(D), Sp(DS), Sp(A)) for _ in range(NA)])
    g = torch.Generator().manual_seed(42)
    obs0, share0 = torch.randn(N, NA, D, generator=g) * 2 + 0.5, torch.randn(N, NA, DS, generator=g) * 3
    for a in range(NA):
        fake.buffer[a].share_obs[0].copy_(share0[:, a])
        fake.buffer[a].obs[0].copy_(obs0[:, a])
    stream, iters = [], []
    seed = 87
    torch.manual_seed(seed)
    train_episode_costs = torch.zeros(1, N)
    for it in range(2):
        steps = []
        for step in range(T):
            values, actions, action_log_probs, rnn_states, rnn_states_critic, cost_preds, rnn_states_cost = m.Runner.collect(fake, step)
            obs, share_obs = torch.randn(N, NA, D, generator=g) * 2 + 0.5, torch.randn(N, NA, DS, generator=g) * 3
            rewards, costs = torch.randn(N, NA, 1, generator=g), (torch.rand(N, NA, 1, generator=g) < 0.3).float()
            dones = (torch.rand(N, generator=g) < 0.2)[:, None].expand(N, NA).clone()
            train_episode_costs += torch.mean(costs, dim=1).flatten()
            data = (obs, share_obs, rewards, costs, dones, None, values, actions, action_log_probs, rnn_states, rnn_states_critic,
                    cost_preds, rnn_states_cost, train_episode_costs.mean())
            m.Runner.insert(fake, data)
            steps.append(dict(obs=obs, share_obs=share_obs, rewards=rewards, costs=costs, dones=dones))
        m.Runner.compute(fake)
        m.Runner.train(fake)
        res = []
        for a in range(NA):
            vn = fake.trainer[a].value_normalizer
            st = _states(policy[a])          # the critics' states after the last iteration only (fixture size)
            res.append(dict(factor=fake.buffer[a].factor.clone(), popart=(vn.running_mean.clone(), vn.running_mean_sq.clone(), vn.debiasing_term.clone()),
                            returns=fake.buffer[a].returns.clone(), cost_returns=fake.buffer[a].cost_returns.clone(),
                            state=st if it == 1 else dict(actor=st["actor"])))
        stream.append(steps)
        iters.append(dict(agents=res))
        if it == 0:
            for a in range(NA):
                fake.buffer[a].return_aver_insert(torch.tensor(27.5))
    torch.set_num_threads(threads)
    out["epoch"] = dict(cfg={k: cfg[k] for k in KEEP}, dims=(T, N, D, DS, A, H, NA), init=init, obs0=obs0, share_obs0=share0, seed=seed,
                        stream=stream, iters=iters, aver_cost_after_first=27.5)


def main():
    sys.path.insert(0, mg.ROOT)
    mg.import_reference()
    out = {}
    gen_macpo(out)
    gen_macpo_epoch(out)
    path = os.path.join(HERE, "macpo.pt")
    torch.save(out, path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
