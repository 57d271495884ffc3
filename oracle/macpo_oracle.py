"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): CPU restatement of MACPO, the multi-agent constrained trust-region
trainer (safepo/multi_agent/macpo.py:98-420 and the Runner's train at :657-688), on the MAPPO-Lag networks, buffer and
runner of oracle/ma_oracle.py.  Same torch ops in the same order as the reference: flat_grad, the Fisher-vector product by
double backprop of the reference's ``kl_divergence``, conjugate_gradient, the five-way ``optim_case`` analysis with all of
its 1e-8 substitutions and the backtracking line search.  Pinned bit for bit against the reference's own classes by
tests/golden/make_golden_macpo.py (fixture macpo.pt) and tests/test_macpo_cpu.py.

Reference quirk kept: kl_divergence (macpo.py:153-166) computes log std_old - log std + (std_old^2 + dmu^2) / (1e-8 + 2 std^2)
- 1/2, the log term with the sign of KL(new || old)'s, so the line-search "KL" can be negative, and the log_std block of the
Fisher matrix it defines is not the Gaussian Fisher (see ``closed_form_fvp``)."""
import numpy as np
import torch

from oracle.ma_oracle import OracleMABuffer, OracleMARunner, OracleMATrainer, OraclePopArt, ma_actor_dist, ma_critic_value


def kl_divergence(mu, std, mu_old, std_old):
    """macpo.py:153-166 on already evaluated means / standard deviations, [n, 1]."""
    logstd = torch.log(std)
    mu_old = mu_old.detach()
    std_old = std_old.detach()
    logstd_old = torch.log(std_old)
    kl = logstd_old - logstd + (std_old.pow(2) + (mu_old - mu).pow(2)) / (1e-8 + 2.0 * std.pow(2)) - 0.5
    return kl.sum(1, keepdim=True)


def flat_grad(grads):
    return torch.cat([g.view(-1) for g in grads if g is not None])


def macpo_case(q_coef, r_coef, s_coef, bb, rescale_constraint_val, target_kl):
    """macpo.py:271-321: (optim_case, lam, nu, whether_recover_policy_value) with the reference's scalar
    types (0-d / [1] float32 tensors and Python floats) and every 1e-8 substitution."""
    if bb <= 1e-8 and rescale_constraint_val < 0:
        r_coef, s_coef = torch.tensor(0), torch.tensor(0)
        positive_Cauchy_value = torch.tensor(0)
        whether_recover_policy_value = torch.tensor(0)
        optim_case = 4
    else:
        if r_coef == 0:
            r_coef = 1e-8
        if s_coef == 0:
            s_coef = 1e-8
        positive_Cauchy_value = q_coef - (r_coef ** 2) / (1e-8 + s_coef)
        whether_recover_policy_value = 2 * target_kl - (rescale_constraint_val ** 2) / (1e-8 + s_coef)
        if rescale_constraint_val < 0 and whether_recover_policy_value < 0:
            optim_case = 3
        elif rescale_constraint_val < 0 and whether_recover_policy_value >= 0:
            optim_case = 2
        elif rescale_constraint_val >= 0 and whether_recover_policy_value >= 0:
            optim_case = 1
        else:
            optim_case = 0
    if whether_recover_policy_value == 0:
        whether_recover_policy_value = 1e-8
    if optim_case in [3, 4]:
        lam = torch.sqrt(q_coef / (2 * target_kl))
        nu = torch.tensor(0)
    elif optim_case in [1, 2]:
        LA, LB = [0, r_coef / rescale_constraint_val], [r_coef / rescale_constraint_val, np.inf]
        LA, LB = (LA, LB) if rescale_constraint_val < 0 else (LB, LA)
        proj = lambda x, L: max(L[0], min(L[1], x))          # noqa: E731
        lam_a = proj(torch.sqrt(positive_Cauchy_value / whether_recover_policy_value), LA)
        lam_b = proj(torch.sqrt(q_coef / (torch.tensor(2 * target_kl))), LB)
        f_a = lambda lam: -0.5 * (positive_Cauchy_value / (1e-8 + lam) + whether_recover_policy_value * lam) \
            - r_coef * rescale_constraint_val / (1e-8 + s_coef)                          # noqa: E731
        f_b = lambda lam: -0.5 * (q_coef / (1e-8 + lam) + 2 * target_kl * lam)          # noqa: E731
        lam = lam_a if f_a(lam_a) >= f_b(lam_b) else lam_b
        nu = max(0, lam * rescale_constraint_val - r_coef) / (1e-8 + s_coef)
    else:
        lam = torch.tensor(0)
        nu = torch.sqrt(torch.tensor(2 * target_kl) / (1e-8 + s_coef))
    return optim_case, lam, nu, whether_recover_policy_value


class OracleMACPOTrainer(OracleMATrainer):
    """MACPO_Trainer (macpo.py:96-414) around three OracleMANets: Adam for both critics, one PopArt shared by the reward and
    the cost value loss (4 updates of its statistics per trpo_update), the actor moved only by the trust-region step."""

    def __init__(self, actor, critic, cost_critic, cfg):
        self.actor, self.critic, self.cost_critic, self.cfg = actor, critic, cost_critic, cfg
        self.opt_c = torch.optim.Adam(critic.params(), lr=cfg["critic_lr"], eps=cfg["opti_eps"], weight_decay=cfg["weight_decay"])
        self.opt_k = torch.optim.Adam(cost_critic.params(), lr=cfg["critic_lr"], eps=cfg["opti_eps"], weight_decay=cfg["weight_decay"])
        self.popart = OraclePopArt(1)

    def _eval(self, obs, actions):
        dist = ma_actor_dist(self.actor, obs, self.cfg.get("std_x_coef", 1.0), self.cfg.get("std_y_coef", 0.5))
        return dist.log_prob(actions), dist.entropy().mean(), dist.mean, dist.stddev

    def _set_actor(self, flat):
        i = 0
        for p in self.actor.params():
            k = p.numel()
            p.data.copy_(flat[i:i + k].view(p.size()))
            i += k

    def _draw_like_actor_init(self):
        """The reference builds old_actor as a fresh Actor (macpo.py:331-335) and overwrites its weights: its initialisation draws
        from the global generator (nn.Linear's reset_parameters, then orthogonal_, per layer, model.py / mlp.py / distributions.py)
        and so moves the batch permutation of the agents trained after this one.  Same draws, results discarded."""
        p = self.actor.p
        shapes = [p["base.mlp.fc1.0.weight"].shape] + [p[f"base.mlp.fc2.{i}.0.weight"].shape for i in range(self.actor.layer_N)] + \
            [p["act.action_out.fc_mean.weight"].shape]
        for out_f, in_f in shapes:
            lin = torch.nn.Linear(in_f, out_f)
            torch.nn.init.orthogonal_(lin.weight)

    def fisher_vector_product(self, obs, actions, p):
        """macpo.py:187-198: Hessian of the mean quirky KL of the actor against a detached copy of itself, times p, + 0.1 p."""
        _, _, mu, std = self._eval(obs, actions)
        _, _, mu_old, std_old = self._eval(obs, actions)
        kl = kl_divergence(mu, std, mu_old, std_old).mean()
        kl_grad = flat_grad(torch.autograd.grad(kl, self.actor.params(), create_graph=True, allow_unused=True))
        kl_hessian_p = torch.autograd.grad((kl_grad * p).sum(), self.actor.params(), allow_unused=True)
        kl_hessian_p = torch.cat([h.contiguous().view(-1) for h in kl_hessian_p if h is not None]).data
        return kl_hessian_p + 0.1 * p

    def conjugate_gradient(self, obs, actions, b, nsteps, residual_tol=1e-10):
        """macpo.py:168-185."""
        x = torch.zeros(b.size(), dtype=b.dtype)
        r = b.clone()
        p = b.clone()
        rdotr = torch.dot(r, r)
        for _ in range(nsteps):
            _Avp = self.fisher_vector_product(obs, actions, p)
            alpha = rdotr / (torch.dot(p, _Avp) + 1e-8)
            x += alpha * p
            r -= alpha * _Avp
            new_rdotr = torch.dot(r, r)
            betta = new_rdotr / rdotr
            p = r + betta * p
            rdotr = new_rdotr
            if rdotr < residual_tol:
                break
        return x

    def trpo_update(self, s):
        """macpo.py:200-380 on a sample dict (the keys of OracleMABuffer.whole_batch_sample).  Returns a dict: the reference's
        returned values under their names plus the intermediates g, b, optim_case and ``accepted`` (index of the accepted
        line-search trial, -1 when every trial was rejected and the actor restored)."""
        c = self.cfg
        obs, actions = s["obs"], s["actions"]
        action_log_probs, dist_entropy, action_mu, action_std = self._eval(obs, actions)
        values = ma_critic_value(self.critic, s["share_obs"])
        cost_values = ma_critic_value(self.cost_critic, s["share_obs"])

        value_loss = self.cal_value_loss(values, s["value_preds"], s["returns"])
        self.opt_c.zero_grad()
        (value_loss * c["value_loss_coef"]).backward()
        critic_grad_norm = torch.nn.utils.clip_grad_norm_(self.critic.params(), c["max_grad_norm"])
        self.opt_c.step()
        cost_loss = self.cal_value_loss(cost_values, s["cost_preds"], s["cost_returns"])
        self.opt_k.zero_grad()
        (cost_loss * c["value_loss_coef"]).backward()
        cost_grad_norm = torch.nn.utils.clip_grad_norm_(self.cost_critic.params(), c["max_grad_norm"])
        self.opt_k.step()

        rescale_constraint_val = (s["aver_episode_costs"].mean() - c["cost_limit"]) * (1 - c["gamma"])
        if rescale_constraint_val == 0:
            rescale_constraint_val = 1e-8

        ratio = torch.exp(action_log_probs - s["old_action_log_probs"])
        ratio = torch.prod(ratio, dim=-1, keepdim=True)
        reward_loss = -torch.sum(ratio * s["factor"] * s["adv_targ"], dim=-1, keepdim=True).mean()
        reward_loss_grad = flat_grad(torch.autograd.grad(reward_loss, self.actor.params(), retain_graph=True, allow_unused=True))
        cost_loss = torch.sum(ratio * s["factor"] * s["cost_adv_targ"], dim=-1, keepdim=True).mean()
        cost_loss_grad = flat_grad(torch.autograd.grad(cost_loss, self.actor.params(), retain_graph=True, allow_unused=True))
        B_cost_loss_grad = flat_grad(cost_loss_grad.unsqueeze(0))

        g_step_dir = self.conjugate_gradient(obs, actions, reward_loss_grad.data, nsteps=c["conjugate_gradient_iters"])
        b_step_dir = self.conjugate_gradient(obs, actions, B_cost_loss_grad.data, nsteps=c["conjugate_gradient_iters"])

        q_coef = (reward_loss_grad * g_step_dir).sum(0, keepdim=True)
        r_coef = (reward_loss_grad * b_step_dir).sum(0, keepdim=True)
        s_coef = (cost_loss_grad * b_step_dir).sum(0, keepdim=True)
        fraction = c["step_fraction"]
        loss_improve = 0
        bb = torch.dot(B_cost_loss_grad, B_cost_loss_grad)
        optim_case, lam, nu, whether_recover_policy_value = macpo_case(q_coef, r_coef, s_coef, bb, rescale_constraint_val, c["target_kl"])
        if optim_case == 4:
            b_step_dir = torch.tensor(0)

        x_a = (1. / (lam + 1e-8)) * (g_step_dir + nu * b_step_dir)
        x_b = (nu * b_step_dir)
        x = x_a if optim_case > 0 else x_b

        reward_loss = reward_loss.detach()
        cost_loss = cost_loss.detach()
        params = torch.cat([p.data.view(-1) for p in self.actor.params()])
        old_params = params.clone()
        self._draw_like_actor_init()
        mu_old, std_old = action_mu.detach(), action_std.detach()

        expected_improve = -torch.dot(x, reward_loss_grad).sum(0, keepdim=True)
        expected_improve = expected_improve.detach()
        flag, accepted, kl, mu, std = False, -1, None, action_mu, action_std
        for i in range(c["searching_steps"]):
            x_norm = torch.norm(x)
            if x_norm > 0.5:
                x = x * 0.5 / x_norm
            new_params = params - c["fraction_coef"] * (fraction ** i) * x
            self._set_actor(new_params)
            with torch.no_grad():
                action_log_probs, dist_entropy, mu, std = self._eval(obs, actions)
            ratio = torch.exp(action_log_probs - s["old_action_log_probs"])
            ratio = torch.prod(ratio, dim=-1, keepdim=True)
            new_reward_loss = torch.sum(ratio * s["factor"] * s["adv_targ"], dim=-1, keepdim=True).mean()
            new_cost_loss = torch.sum(ratio * s["factor"] * s["cost_adv_targ"], dim=-1, keepdim=True).mean()
            new_reward_loss = -new_reward_loss
            loss_improve = new_reward_loss - reward_loss
            kl = kl_divergence(mu, std, mu_old, std_old).mean()
            if ((kl < c["target_kl"]) and (loss_improve < 0 if optim_case > 1 else True)
                    and (new_cost_loss.mean() - cost_loss.mean() <= max(-rescale_constraint_val, 0))):
                flag, accepted = True, i
                break
            expected_improve *= fraction
        if not flag:
            self._set_actor(old_params)
        return dict(value_loss=value_loss.detach(), critic_grad_norm=critic_grad_norm, kl=kl, loss_improve=torch.as_tensor(loss_improve),
                    expected_improve=expected_improve, dist_entropy=dist_entropy.detach(), ratio=ratio.detach(), cost_loss=cost_loss,
                    cost_grad_norm=cost_grad_norm, whether_recover_policy_value=torch.as_tensor(whether_recover_policy_value),
                    lam=torch.as_tensor(lam), nu=torch.as_tensor(nu), g=reward_loss_grad.detach(), b=B_cost_loss_grad.detach(),
                    g_step_dir=g_step_dir, b_step_dir=torch.as_tensor(b_step_dir), x=x, action_mu=mu, action_std=std, B_cost_loss_grad_dot=bb,
                    optim_case=optim_case, accepted=accepted)

    def train(self, buf, perm=None):
        """macpo.py:382-400: advantages standardised with +1e-5 and without masking, ONE trpo_update on the whole batch."""
        advantages = buf.returns[:-1] - self.popart.denormalize(buf.value_preds[:-1])
        advantages = (advantages - torch.mean(advantages.clone())) / (torch.std(advantages.clone()) + 1e-5)
        cost_adv = buf.cost_returns[:-1] - self.popart.denormalize(buf.cost_preds[:-1])
        cost_adv = (cost_adv - cost_adv.clone().mean()) / (cost_adv.clone().std() + 1e-5)
        return self.trpo_update(buf.whole_batch_sample(advantages, cost_adv, perm))


class OracleMACPORunner(OracleMARunner):
    """macpo.Runner's per-iteration part: collect / insert / compute are MAPPO-Lag's; train (macpo.py:657-688) runs one
    MACPO_Trainer.train per agent in a random order with the cross-agent factor."""

    def __init__(self, nets, cfg, T, N, obs_dim, share_obs_dim, act_dim):
        self.cfg, self.T, self.N, self.num_agents = cfg, T, N, len(nets)
        self.nets = nets
        self.buffer = [OracleMABuffer(T, N, obs_dim, share_obs_dim, act_dim, cfg["gamma"], cfg["gae_lambda"]) for _ in nets]
        self.trainer = [OracleMACPOTrainer(a, c, k, cfg) for a, c, k in nets]

    def train(self, agent_order=None, perms=None):
        factor = torch.ones(self.T, self.N, 1)
        outs = {}
        for agent_id in (torch.randperm(self.num_agents) if agent_order is None else agent_order):
            a = int(agent_id)
            b, tr, actor = self.buffer[a], self.trainer[a], self.nets[a][0]
            A = b.actions.shape[-1]
            b.factor.copy_(factor)
            flat_obs, flat_act = b.obs[:-1].reshape(-1, b.obs.shape[-1]), b.actions.reshape(-1, A)
            with torch.no_grad():
                old_lp = ma_actor_dist(actor, flat_obs).log_prob(flat_act)
            outs[a] = tr.train(b, None if perms is None else perms[a])
            with torch.no_grad():
                new_lp = ma_actor_dist(actor, flat_obs).log_prob(flat_act)
            factor = factor * torch.prod(torch.exp(new_lp - old_lp).reshape(self.T, self.N, A), dim=-1, keepdim=True)
            b.after_update()
        return outs


def closed_form_fvp(actor, obs, v, damping=0.1, std_x_coef=1.0, std_y_coef=0.5):
    """The Fisher-vector product of fisher_vector_product in the form the device computes it (float64 when the actor and v
    are): forward tangents block by block, the mean block J^T diag(2 / (1e-8 + 2 std^2)) J v / n by one backward pass, the
    quirky log_std block and the damping.  At coincidence (mu = mu_old, std = std_old) the KL's first derivative in mu is 0 and
    its mu-std cross term vanishes; in std its first derivative is f_s = -1/s - 4 s^3 / D^2 (D = 1e-8 + 2 s^2, ~ -2/s, not 0) and
    its second f_ss = 1/s^2 - 4 s^2 / D^2 + 32 s^4 / D^3 (~ 4/s^2), so the log_std block is f_ss s'^2 + f_s s'' per dimension."""
    import torch.nn.functional as F
    p = actor.p
    names = list(p.keys())
    t, i = {}, 0
    for k in names:
        t[k] = v[i:i + p[k].numel()].view(p[k].shape)
        i += p[k].numel()

    def ln_stats(x):
        m = x.mean(-1, keepdim=True)
        rstd = torch.rsqrt(((x - m) ** 2).mean(-1, keepdim=True) + 1e-5)
        return (x - m) * rstd, rstd
    with torch.no_grad():
        xh, _ = ln_stats(obs)
        x = xh * p["base.feature_norm.weight"] + p["base.feature_norm.bias"]
        dx = xh * t["base.feature_norm.weight"] + t["base.feature_norm.bias"]
        blocks = [("base.mlp.fc1.0", "base.mlp.fc1.2")] + [(f"base.mlp.fc2.{j}.0", f"base.mlp.fc2.{j}.2") for j in range(actor.layer_N)]
        for lin, ln in blocks:
            W, b = p[lin + ".weight"], p[lin + ".bias"]
            z = F.linear(x, W, b)
            dz = dx @ W.t() + x @ t[lin + ".weight"].t() + t[lin + ".bias"]
            pre = F.elu(z)
            dpre = dz * torch.where(pre > 0, torch.ones_like(pre), pre + 1)
            ph, rstd = ln_stats(pre)
            dph = rstd * (dpre - dpre.mean(-1, keepdim=True) - ph * (dpre * ph).mean(-1, keepdim=True))
            x = ph * p[ln + ".weight"] + p[ln + ".bias"]
            dx = dph * p[ln + ".weight"] + ph * t[ln + ".weight"] + t[ln + ".bias"]
        Wm = p["act.action_out.fc_mean.weight"]
        dmu = dx @ Wm.t() + x @ t["act.action_out.fc_mean.weight"].t() + t["act.action_out.fc_mean.bias"]
        sg = torch.sigmoid(p["act.action_out.log_std"] / std_x_coef)
        s = sg * std_y_coef
        D = 1e-8 + 2.0 * s ** 2
        dmean = dmu * (2.0 / D) / obs.shape[0]
    # J^T dmean: the backward pass of mean = features(obs) W_m^T + b_m
    mean = F.linear(actor.features(obs), Wm, p["act.action_out.fc_mean.bias"])
    grads = torch.autograd.grad((mean * dmean).sum(), [p[k] for k in names], allow_unused=True)
    out = []
    for k, g in zip(names, grads):
        if k == "act.action_out.log_std":
            ds = std_y_coef * sg * (1 - sg) / std_x_coef
            dds = std_y_coef * sg * (1 - sg) * (1 - 2 * sg) / std_x_coef ** 2
            f_s = -1.0 / s - 4.0 * s ** 3 / D ** 2
            f_ss = 1.0 / s ** 2 - 4.0 * s ** 2 / D ** 2 + 32.0 * s ** 4 / D ** 3
            g = (f_ss * ds ** 2 + f_s * dds) * t[k]
        out.append(g.detach().reshape(-1))
    return torch.cat(out) + damping * v
