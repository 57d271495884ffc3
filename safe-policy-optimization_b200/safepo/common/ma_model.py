"""Multi-agent (MAPPO-Lag) networks on the device (SURVEY section 8f rank 3).

``MultiAgentNets`` holds the weights of one agent's actor, reward critic and cost critic under the reference's own
``state_dict`` names (safepo/common/model.py:172-363: ``base.feature_norm``, ``base.mlp.fc1``, ``base.mlp.fc2.{i}``,
``act.action_out`` / ``v_out``) and evaluates ``MAPPO_L_Policy.get_actions`` (safepo/multi_agent/mappolag.py:69-82) with
libspo kernels: one ``spo_ma_mlp_layer`` launch per hidden layer and one ``spo_ma_head`` launch per net.

``MultiAgentTrainer`` is the device side of ``MAPPO_L_Trainer.ppo_update`` (mappolag.py:135-199) for one agent: training
forward with the activations kept, the clipped-surrogate / clipped-Huber loss heads, the backward pass layer by layer
(``spo_ma_ln_elu_bwd``, ``spo_ma_gemm_tn``, ``spo_ma_gemm_nn``), ``clip_grad_norm_`` + Adam on the packed parameters
(``spo_ma_clip_adam``), the PopArt value normaliser and the Lagrange-multiplier step -- no host synchronisation inside an
update, no CPU path.  Each net's parameters live in one packed fp32 buffer; ``net.p[name]`` are views into it."""
from __future__ import annotations

import torch

from safepo import _lib as L


class _Net:
    def __init__(self, state, device, layer_N):
        # one packed buffer per net (every tensor starts on a 16-byte boundary), parameters as views: the update kernels
        # run over the whole buffer, the layer kernels over the views
        offs, total = {}, 0
        for k, v in state.items():
            offs[k] = total
            total += (v.numel() + 3) // 4 * 4
        self.flat = torch.zeros(total, dtype=torch.float32, device=device)
        self.gflat = torch.zeros(total, dtype=torch.float32, device=device)      # gradients of the last update (before the clip)
        self.exp_avg = torch.zeros(total, dtype=torch.float32, device=device)
        self.exp_avg_sq = torch.zeros(total, dtype=torch.float32, device=device)
        self.p, self.g = {}, {}
        for k, v in state.items():
            sl = slice(offs[k], offs[k] + v.numel())
            self.p[k] = self.flat[sl].view(v.shape)
            self.g[k] = self.gflat[sl].view(v.shape)
            self.p[k].copy_(v.detach().to(device=device, dtype=torch.float32))
        self.layer_N = layer_N
        self.H = self.p["base.mlp.fc1.0.weight"].shape[0]
        self.D = self.p["base.mlp.fc1.0.weight"].shape[1]
        self.step = 0            # Adam step count
        # (weight, bias, ln weight, ln bias) names of the 1 + layer_N blocks
        self.blocks = [("base.mlp.fc1.0.weight", "base.mlp.fc1.0.bias", "base.mlp.fc1.2.weight", "base.mlp.fc1.2.bias")] + \
            [(f"base.mlp.fc2.{i}.0.weight", f"base.mlp.fc2.{i}.0.bias", f"base.mlp.fc2.{i}.2.weight", f"base.mlp.fc2.{i}.2.bias")
             for i in range(layer_N)]

    def state_dict(self):
        return {k: v.detach().clone() for k, v in self.p.items()}

    def features(self, x, work):
        """MLPBase.forward: feature_norm folded into the first layer's launch."""
        p, n = self.p, x.shape[0]
        a, b = work
        w, bb, lw, lb = self.blocks[0]
        L.call("spo_ma_mlp_layer", L.ptr(x), n, self.D, L.ptr(p[w]), L.ptr(p[bb]), L.ptr(p[lw]), L.ptr(p[lb]), self.H,
               L.ptr(p["base.feature_norm.weight"]), L.ptr(p["base.feature_norm.bias"]), L.ptr(a), L.stream())
        for w, bb, lw, lb in self.blocks[1:]:
            L.call("spo_ma_mlp_layer", L.ptr(a), n, self.H, L.ptr(p[w]), L.ptr(p[bb]), L.ptr(p[lw]), L.ptr(p[lb]), self.H, None, None,
                   L.ptr(b), L.stream())
            a, b = b, a
        return a


class MultiAgentNets:
    def __init__(self, actor_state, critic_state, cost_critic_state, device, layer_N=2, std_x_coef=1.0, std_y_coef=0.5):
        device = torch.device(device)
        self._require_cuda(device)
        self.device = device
        self.actor = _Net(actor_state, device, layer_N)
        self.critic = _Net(critic_state, device, layer_N)
        self.cost_critic = _Net(cost_critic_state, device, layer_N)
        self.act_dim = self.actor.p["act.action_out.fc_mean.weight"].shape[0]
        self.std_x_coef, self.std_y_coef = float(std_x_coef), float(std_y_coef)
        self._work = {}

    @staticmethod
    def _require_cuda(device):
        if device.type != "cuda":
            raise L.SpoError("MultiAgentNets runs on a CUDA device only (no CPU fallback)")

    def _buffers(self, n, H):
        key = (n, H)
        if key not in self._work:
            self._work[key] = (torch.empty(n, H, dtype=torch.float32, device=self.device), torch.empty(n, H, dtype=torch.float32, device=self.device))
        return self._work[key]

    def _value(self, net, cent_obs):
        n = cent_obs.shape[0]
        feat = net.features(cent_obs, self._buffers(n, net.H))
        out = torch.empty(n, 1, dtype=torch.float32, device=self.device)
        L.call("spo_ma_head", L.ptr(feat), n, net.H, L.ptr(net.p["v_out.weight"]), L.ptr(net.p["v_out.bias"]), 1, None, 1.0, 1.0, None,
               L.ptr(out), None, L.stream())
        return out

    def get_actions(self, cent_obs, obs, eps=None, deterministic=False):
        """(values [N,1], actions [N,A], action_log_probs [N,A], cost_preds [N,1]) like MAPPO_L_Policy.get_actions.
        ``eps`` [N,A]: the standard-normal draws to use (torch.randn on the device when omitted and not deterministic)."""
        for t in (cent_obs, obs):
            if not (t.device.type == self.device.type and t.dtype == torch.float32 and t.is_contiguous()):   # self.device is CUDA (constructor)
                raise L.SpoError("MultiAgentNets needs contiguous fp32 CUDA tensors")
        n, A, net = obs.shape[0], self.act_dim, self.actor
        feat = net.features(obs, self._buffers(n, net.H))
        if deterministic:
            eps = None
        elif eps is None:
            eps = torch.randn(n, A, dtype=torch.float32, device=self.device)
        actions = torch.empty(n, A, dtype=torch.float32, device=self.device)
        logp = torch.empty(n, A, dtype=torch.float32, device=self.device)
        L.call("spo_ma_head", L.ptr(feat), n, net.H, L.ptr(net.p["act.action_out.fc_mean.weight"]), L.ptr(net.p["act.action_out.fc_mean.bias"]),
               A, L.ptr(net.p["act.action_out.log_std"]), self.std_x_coef, self.std_y_coef, L.ptr(eps), L.ptr(actions),
               L.ptr(logp), L.stream())
        return self._value(self.critic, cent_obs), actions, logp, self._value(self.cost_critic, cent_obs)


    def evaluate_actions(self, obs, actions):
        """Per-dimension log-probabilities of given actions under the current actor (MultiAgentActor.evaluate_actions,
        model.py:270-296 -> act.py:62-77), as the runner needs them for the cross-agent factor (mappolag.py:474-497): the mean
        from the forward kernels, then Normal.log_prob's own formula element-wise on the device."""
        n, A, net = obs.shape[0], self.act_dim, self.actor
        feat = net.features(obs, self._buffers(n, net.H))
        mean = torch.empty(n, A, dtype=torch.float32, device=self.device)
        L.call("spo_ma_head", L.ptr(feat), n, net.H, L.ptr(net.p["act.action_out.fc_mean.weight"]), L.ptr(net.p["act.action_out.fc_mean.bias"]),
               A, L.ptr(net.p["act.action_out.log_std"]), self.std_x_coef, self.std_y_coef, None, L.ptr(mean), None, L.stream())
        std = torch.sigmoid(net.p["act.action_out.log_std"] / self.std_x_coef) * self.std_y_coef
        return -((actions - mean) ** 2) / (2 * std ** 2) - std.log() - _LOG_SQRT_2PI


_LOG_SQRT_2PI = 0.9189385332046727      # math.log(math.sqrt(2 * math.pi)), torch.distributions.Normal.log_prob

# the 18 positions of the sample tuple MAPPO_L_Trainer.ppo_update unpacks (mappolag.py:137-141)
_SAMPLE_KEYS = ("share_obs", "obs", "rnn_states", "rnn_states_critic", "actions", "value_preds", "returns", "masks", "active_masks",
                "old_action_log_probs", "adv_targ", "available_actions", "factor", "cost_preds", "cost_returns", "rnn_states_cost",
                "cost_adv_targ", "aver_episode_costs")


class MultiAgentTrainer:
    """``MAPPO_L_Trainer`` for one agent around ``MultiAgentNets`` (mappolag.py:115-199; MLP policy, no recurrence, no
    active masks, clipped + Huber value loss with the shared PopArt normaliser -- the yaml's defaults).  ``cfg`` carries the
    reference's keys: actor_lr, critic_lr, opti_eps, weight_decay, clip_param, huber_delta, entropy_coef, max_grad_norm,
    cost_limit, gamma, lagrangian_coef_rate, value_loss_coef, lamda_lagr."""

    def __init__(self, nets: MultiAgentNets, cfg):
        self.nets, self.cfg, self.device = nets, dict(cfg), nets.device
        dev = self.device
        self.lamda_lagr = torch.full((1,), float(cfg["lamda_lagr"]), dtype=torch.float32, device=dev)
        self.popart_state = torch.zeros(3, dtype=torch.float32, device=dev)     # running_mean, running_mean_sq, debiasing_term
        self.popart_beta, self.popart_eps = 0.99999, 1e-5                      # popart.py:48
        self._adam_work = torch.empty(1024, dtype=torch.float32, device=dev)
        self._bufs = {}

    # ---- workspace ----
    def _ws(self, n, net):
        key = (n, net.D, net.H, net.layer_N)
        if key not in self._bufs:
            dev, H, D, nl = self.device, net.H, net.D, 1 + net.layer_N
            A = self.nets.act_dim
            f = dict(dtype=torch.float32, device=dev)
            nb32, nb256 = (n + 31) // 32, (n + 255) // 256
            wmax = max(H * max(H, D), A * H)
            self._bufs[key] = dict(
                xn=torch.empty(n, D, **f), pre=[torch.empty(n, H, **f) for _ in range(nl)], out=[torch.empty(n, H, **f) for _ in range(nl)],
                dy=torch.empty(n, max(H, D), **f), dy2=torch.empty(n, max(H, D), **f), dz=torch.empty(n, H, **f),
                part=torch.empty(max(nb32 * 3 * H, nb32 * 2 * D, nb32 * 66, nb256 * 2, 32 * wmax), **f),
                dmean=torch.empty(n, A, **f), v=torch.empty(n, 1, **f), dv=torch.empty(n, **f), rn_c=torch.empty(n, **f), rn_o=torch.empty(n, **f))
        return self._bufs[key]

    # ---- pieces ----
    def _forward_train(self, net, x, ws):
        p, n = net.p, x.shape[0]
        w, bb, lw, lb = net.blocks[0]
        L.call("spo_ma_mlp_layer_train", L.ptr(x), n, net.D, L.ptr(p[w]), L.ptr(p[bb]), L.ptr(p[lw]), L.ptr(p[lb]), net.H,
               L.ptr(p["base.feature_norm.weight"]), L.ptr(p["base.feature_norm.bias"]), L.ptr(ws["out"][0]), L.ptr(ws["pre"][0]),
               L.ptr(ws["xn"]), L.stream())
        for i, (w, bb, lw, lb) in enumerate(net.blocks[1:], start=1):
            L.call("spo_ma_mlp_layer_train", L.ptr(ws["out"][i - 1]), n, net.H, L.ptr(p[w]), L.ptr(p[bb]), L.ptr(p[lw]), L.ptr(p[lb]), net.H,
                   None, None, L.ptr(ws["out"][i]), L.ptr(ws["pre"][i]), None, L.stream())
        return ws["out"][-1]

    def _gemm_tn(self, A_, B_, out, R, M, N, ws):
        """out[M][N] = A_[R][M]^T B_[R][N] (sum over the R rows in slices, partials reduced in order)."""
        tiles = ((M + 127) // 128) * ((N + 63) // 64)            # 128 x 64 output tiles, >= 2 CTAs per SM wanted
        slices = max(1, min(32, (296 + tiles - 1) // tiles, R // 256))
        while slices > 1 and (slices - 1) * (((R + slices - 1) // slices + 31) // 32 * 32) >= R:   # no empty slice (32-row chunks)
            slices -= 1
        L.call("spo_ma_gemm_tn", L.ptr(A_), L.ptr(B_), L.ptr(ws["part"]), R, M, N, slices, L.stream())
        L.call("spo_ma_partial_reduce", L.ptr(ws["part"]), slices, M * N, 1, M * N, L.ptr(out), None, None, 1.0, L.stream())

    def _backward(self, net, x, ws, dfeat):
        """Gradients of every block and of the input LayerNorm from dfeat = d loss / d features (in ws['dy'])."""
        p, g, n, H = net.p, net.g, x.shape[0], net.H
        nb32 = (n + 31) // 32
        dy, dy2 = dfeat, (ws["dy2"] if dfeat is ws["dy"] else ws["dy"])
        for i in reversed(range(len(net.blocks))):
            w, bb, lw, lb = net.blocks[i]
            L.call("spo_ma_ln_elu_bwd", L.ptr(dy), L.ptr(ws["pre"][i]), L.ptr(p[lw]), n, H, L.ptr(ws["dz"]), L.ptr(ws["part"]), L.stream())
            L.call("spo_ma_partial_reduce", L.ptr(ws["part"]), nb32, 3 * H, 3, H, L.ptr(g[lw]), L.ptr(g[lb]), L.ptr(g[bb]), 1.0, L.stream())
            inp, K = (ws["out"][i - 1], H) if i > 0 else (ws["xn"], net.D)
            self._gemm_tn(ws["dz"], inp, g[w], n, H, K, ws)
            L.call("spo_ma_gemm_nn", L.ptr(ws["dz"]), L.ptr(p[w]), L.ptr(dy2), n, K, H, L.stream())
            dy, dy2 = dy2, dy
        L.call("spo_ma_ln_in_bwd", L.ptr(dy), L.ptr(x), n, net.D, L.ptr(ws["part"]), L.stream())
        L.call("spo_ma_partial_reduce", L.ptr(ws["part"]), nb32, 2 * net.D, 2, net.D, L.ptr(g["base.feature_norm.weight"]),
               L.ptr(g["base.feature_norm.bias"]), None, 1.0, L.stream())

    def _clip_adam(self, net, lr):
        c = self.cfg
        net.step += 1
        norm = torch.empty(2, dtype=torch.float32, device=self.device)
        L.call("spo_ma_clip_adam", L.ptr(net.flat), L.ptr(net.gflat), L.ptr(net.exp_avg), L.ptr(net.exp_avg_sq), net.flat.numel(),
               float(c["max_grad_norm"]), float(lr), 0.9, 0.999, float(c["opti_eps"]), float(c["weight_decay"]), net.step,
               L.ptr(self._adam_work), L.ptr(norm), L.stream())
        return norm[0]

    def _critic_update(self, net, share_obs, value_preds, returns, ws):
        """cal_value_loss (mappolag.py:121-133) + the critic's optimiser step (:174-186); returns (loss, grad norm)."""
        c, n, H = self.cfg, share_obs.shape[0], net.H
        feat = self._forward_train(net, share_obs, ws)
        L.call("spo_ma_head", L.ptr(feat), n, H, L.ptr(net.p["v_out.weight"]), L.ptr(net.p["v_out.bias"]), 1, None, 1.0, 1.0, None,
               L.ptr(ws["v"]), None, L.stream())
        # the reference normalises the returns twice, UPDATING the shared statistics both times: first for the clipped error
        for dst in (ws["rn_c"], ws["rn_o"]):
            L.call("spo_ma_popart_normalize", L.ptr(returns), n, L.ptr(self.popart_state), self.popart_beta, self.popart_eps, L.ptr(dst), L.stream())
        nb256 = (n + 255) // 256
        L.call("spo_ma_value_loss", L.ptr(ws["v"]), L.ptr(value_preds), L.ptr(ws["rn_c"]), L.ptr(ws["rn_o"]), n, float(c["clip_param"]),
               float(c["huber_delta"]), float(c["value_loss_coef"]) / n, L.ptr(ws["dv"]), L.ptr(ws["part"]), L.stream())
        loss = torch.empty(1, dtype=torch.float32, device=self.device)
        L.call("spo_ma_partial_reduce", L.ptr(ws["part"]), nb256, 2, 1, 1, L.ptr(loss), None, None, 1.0 / n, L.stream())
        L.call("spo_ma_partial_reduce", L.ptr(ws["part"]), nb256, 2, 2, 1, None, L.ptr(net.g["v_out.bias"]), None, 1.0, L.stream())
        self._gemm_tn(ws["dv"], feat, net.g["v_out.weight"], n, 1, H, ws)
        L.call("spo_ma_gemm_nn", L.ptr(ws["dv"]), L.ptr(net.p["v_out.weight"]), L.ptr(ws["dy"]), n, H, 1, L.stream())
        self._backward(net, share_obs, ws, ws["dy"])
        return loss[0], self._clip_adam(net, c["critic_lr"])

    # ---- the update ----
    def ppo_update(self, sample):
        """One update on the whole sample (a dict with the oracle's keys, or the reference's 18-tuple).  Returns
        (value_loss, critic_grad_norm, policy_loss, dist_entropy, actor_grad_norm, imp_weights, cost_loss, cost_grad_norm) as device
        tensors, like mappolag.py:199."""
        if not isinstance(sample, dict):
            sample = {k: v for k, v in zip(_SAMPLE_KEYS, sample)}
        dev, c, nets = self.device, self.cfg, self.nets

        def dv_(x, cols=None):
            t = torch.as_tensor(x, dtype=torch.float32).to(dev).contiguous()
            return t.reshape(t.shape[0], -1) if cols is None else t.reshape(-1)
        obs, share_obs, actions, old_logp = dv_(sample["obs"]), dv_(sample["share_obs"]), dv_(sample["actions"]), dv_(sample["old_action_log_probs"])
        value_preds, returns, adv, factor = dv_(sample["value_preds"], 1), dv_(sample["returns"], 1), dv_(sample["adv_targ"], 1), dv_(sample["factor"], 1)
        cost_preds, cost_returns, cost_adv = dv_(sample["cost_preds"], 1), dv_(sample["cost_returns"], 1), dv_(sample["cost_adv_targ"], 1)
        aver_costs = dv_(sample["aver_episode_costs"], 1)
        n, A = obs.shape[0], nets.act_dim
        if aver_costs.numel() != n:      # the reference only uses aver_episode_costs.mean() (mappolag.py:170); its buffer field is not [n]
            aver_costs = aver_costs.mean().expand(n).contiguous()

        # ---- actor: surrogate on the product of the per-dimension ratios, Lagrangian-mixed advantage ----
        net = nets.actor
        ws = self._ws(n, net)
        feat = self._forward_train(net, obs, ws)
        nb32 = (n + 31) // 32
        imp = torch.empty(n, 1, dtype=torch.float32, device=dev)
        wm, bm, ls = net.p["act.action_out.fc_mean.weight"], net.p["act.action_out.fc_mean.bias"], net.p["act.action_out.log_std"]
        L.call("spo_ma_actor_loss", L.ptr(feat), n, net.H, L.ptr(wm), L.ptr(bm), L.ptr(ls), A, L.ptr(actions), L.ptr(old_logp), L.ptr(adv),
               L.ptr(cost_adv), L.ptr(factor), L.ptr(self.lamda_lagr), 1.0 - float(c["clip_param"]), 1.0 + float(c["clip_param"]),
               nets.std_x_coef, nets.std_y_coef, L.ptr(ws["dmean"]), L.ptr(imp), L.ptr(ws["part"]), L.stream())
        scal = torch.empty(2, dtype=torch.float32, device=dev)
        L.call("spo_ma_actor_finalize", L.ptr(ws["part"]), nb32, n, L.ptr(ls), A, nets.std_x_coef, nets.std_y_coef, float(c["entropy_coef"]),
               L.ptr(net.g["act.action_out.fc_mean.bias"]), L.ptr(net.g["act.action_out.log_std"]), L.ptr(scal), L.stream())
        self._gemm_tn(ws["dmean"], feat, net.g["act.action_out.fc_mean.weight"], n, A, net.H, ws)
        L.call("spo_ma_gemm_nn", L.ptr(ws["dmean"]), L.ptr(wm), L.ptr(ws["dy"]), n, net.H, A, L.stream())
        self._backward(net, obs, ws, ws["dy"])
        actor_grad_norm = self._clip_adam(net, c["actor_lr"])
        # ---- Lagrange multiplier (uses the importance weights of THIS update, mappolag.py:169-172) ----
        L.call("spo_ma_lagrange_step", L.ptr(imp), L.ptr(cost_adv), L.ptr(aver_costs), n, float(c["cost_limit"]), float(c["gamma"]),
               float(c["lagrangian_coef_rate"]), L.ptr(self.lamda_lagr), L.stream())
        # ---- critics ----
        value_loss, critic_grad_norm = self._critic_update(nets.critic, share_obs, value_preds, returns, self._ws(n, nets.critic))
        cost_loss, cost_grad_norm = self._critic_update(nets.cost_critic, share_obs, cost_preds, cost_returns, self._ws(n, nets.cost_critic))
        return value_loss, critic_grad_norm, scal[0], scal[1], actor_grad_norm, imp, cost_loss, cost_grad_norm


    # ---- MAPPO_L_Trainer.train (mappolag.py:200-234) ----
    def popart_mean_sqrt_var(self):
        """(mean, sqrt(var)) of the PopArt normaliser as host floats (popart.py:64-74): one device -> host copy of 3 floats."""
        st = self.popart_state.cpu()
        den = st[2].clamp(min=self.popart_eps)
        mean, mean_sq = st[0] / den, st[1] / den
        var = (mean_sq - mean ** 2).clamp(min=1e-2)
        return float(mean), float(torch.sqrt(var))

    def train(self, buf, perms=None):
        """learning_iters whole-batch updates on a SeparatedReplayBuffer: advantages = returns - denormalised predictions,
        standardised by the mean / unbiased std over the entries (the reference writes NaN into inactive entries and then
        takes torch.mean, so a buffer with any inactive entry yields NaN advantages there too -- reproduced).  ``perms``: the row
        orders to use (one per iteration; torch.randperm on the device when omitted)."""
        mean, sd = self.popart_mean_sqrt_var()

        def standardise(ret, pred):
            adv = ret[:-1] - (pred[:-1] * sd + mean)
            copy = adv.clone()
            copy[buf.active_masks[:-1] == 0.0] = float("nan")
            return (adv - torch.mean(copy)) / (torch.std(copy) + 1e-8)
        advantages = standardise(buf.returns, buf.value_preds)
        cost_adv = standardise(buf.cost_returns, buf.cost_preds)
        out = None
        for it in range(int(self.cfg["learning_iters"])):
            perm = None if perms is None else perms[it]
            out = self.ppo_update(buf.whole_batch_sample(advantages, cost_adv, perm))
        return out

