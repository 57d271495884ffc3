"""Generate the golden fixtures under tests/golden/ from the REAL reference.

Runs only in the build container (needs /root/reference, read-only).  It imports the
reference's own modules -- with the environment packages that are not installable
offline stubbed in sys.modules and ``LinearLR(verbose=...)`` shimmed (torch 2.11 dropped
that kwarg) -- feeds them seeded inputs and stores inputs + outputs.  The fixtures are
what pins ``oracle/`` (tests/test_oracle_golden.py) and, through it, the CUDA path.

    python tests/golden/make_golden.py            # rewrites tests/golden/*.pt
"""
from __future__ import annotations

import csv
import importlib
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"


class _Anything(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return type(name, (), {"__init__": lambda self, *a, **k: None})


def import_reference():
    """Stub gymnasium / safety_gymnasium (absent offline) and import safepo from REF."""
    names = ["gymnasium", "gymnasium.vector", "gymnasium.vector.vector_env", "gymnasium.spaces", "gymnasium.wrappers",
             "gymnasium.wrappers.normalize", "safety_gymnasium", "safety_gymnasium.wrappers",
             "safety_gymnasium.vector", "safety_gymnasium.vector.async_vector_env", "safety_gymnasium.vector.utils",
             "safety_gymnasium.vector.utils.tile_images", "safety_gymnasium.tasks",
             "safety_gymnasium.tasks.safe_multi_agent", "safety_gymnasium.tasks.safe_multi_agent.safe_mujoco_multi"]
    for n in names:
        if n not in sys.modules:
            m = _Anything(n)
            m.__path__ = []
            sys.modules[n] = m
    if REF not in sys.path:
        sys.path.insert(0, REF)
    mods = {}
    for algo in ("ppo_lag", "focops", "cpo", "trpo_lag", "ppo", "pg", "cppo_pid", "trpo", "natural_pg", "rcpo", "pcpo", "cup"):
        m = importlib.import_module(f"safepo.single_agent.{algo}")
        if hasattr(m, "LinearLR"):
            real = m.LinearLR
            m.LinearLR = (lambda real: (lambda opt, **kw: real(opt, **{k: v for k, v in kw.items() if k != "verbose"})))(real)
        mods[algo] = m
    mods["buffer"] = importlib.import_module("safepo.common.buffer")
    mods["model"] = importlib.import_module("safepo.common.model")
    mods["lagrange"] = importlib.import_module("safepo.common.lagrange")
    return mods


def state_of(policy):
    return {n: {k: v.detach().clone() for k, v in getattr(policy, n).state_dict().items()}
            for n in ("reward_critic", "cost_critic", "actor")}


def gen_forward(ref, out):
    cases = []
    for (D, A, n, seed) in ((60, 2, 7, 0), (88, 2, 33, 1), (27, 8, 5, 2)):
        torch.manual_seed(seed)
        pol = ref["model"].ActorVCritic(D, A, [64, 64])
        with torch.no_grad():
            pol.actor.log_std.copy_(torch.linspace(-0.5, 0.3, A))
        obs = torch.randn(n, D)
        g = torch.Generator().manual_seed(100 + seed)
        eps = torch.randn(n, A, generator=g)
        # rsample draws from the global generator: replay eps by seeding then re-drawing
        torch.manual_seed(999)
        with torch.no_grad():
            act, logp, vr, vc = pol.step(obs)
        torch.manual_seed(999)
        eps_used = torch.empty(n, A).normal_()
        with torch.no_grad():
            dact, dlogp, _, _ = pol.step(obs, deterministic=True)
            a1, l1, r1, c1 = pol.step(obs[0])  # single-row form, ppo_lag.py:206
        cases.append(dict(D=D, A=A, state=state_of(pol), obs=obs, eps=eps_used, act=act, logp=logp, v_r=vr, v_c=vc,
                          det_act=dact, det_logp=dlogp, row_shapes=[tuple(a1.shape), tuple(l1.shape), tuple(r1.shape)]))
    out["forward"] = cases


def gen_gae(ref, out):
    B = ref["buffer"]
    # Appendix B.1
    adv, tgt = B.calculate_adv_and_value_targets(torch.tensor([0.5, 0.4, 0.3, 0.2]), torch.tensor([1.0, 0.0, 2.0, 0.2]),
                                                 lam=0.95, gamma=0.99)
    out["gae_kat"] = dict(adv=adv, tgt=tgt)
    # Appendix B.2: buffer layout / two segments
    class Sp:  # noqa
        def __init__(s, d): s.shape = (d,)
    buf = B.VectorizedOnPolicyBuffer(Sp(1), Sp(1), size=4, num_envs=2)
    for t in range(4):
        z = torch.tensor([float(t), 10.0 + t])
        buf.store(obs=torch.tensor([[t + 0.0], [t + 100.0]]), act=torch.zeros(2, 1), reward=z, cost=z / 2,
                  value_r=z / 10, value_c=z / 5, log_prob=torch.zeros(2))
        if t == 1:
            buf.finish_path(idx=0)
        if t == 3:
            buf.finish_path(torch.tensor([0.7]), torch.tensor([0.3]), idx=0)
            buf.finish_path(torch.tensor([1.1]), torch.tensor([0.9]), idx=1)
    out["buffer_kat"] = {k: v.clone() for k, v in buf.get().items()}
    # random segmentations through the reference buffer
    cases = []
    for (N, T, seed, p_end) in ((3, 17, 0, 0.2), (5, 64, 1, 0.05), (2, 133, 2, 0.02), (4, 1, 3, 0.5)):
        g = torch.Generator().manual_seed(seed)
        rew, cost = torch.randn(N, T, generator=g), (torch.rand(N, T, generator=g) < 0.3).float()
        v_r, v_c = torch.randn(N, T, generator=g), torch.randn(N, T, generator=g).abs()
        seg = (torch.rand(N, T, generator=g) < p_end)
        seg[:, -1] = True
        boot_r, boot_c = torch.randn(N, T, generator=g) * seg, torch.randn(N, T, generator=g) * seg
        term = (torch.rand(N, T, generator=g) < 0.3) & seg  # terminated => zero bootstrap
        boot_r, boot_c = boot_r * (~term), boot_c * (~term)
        buf = B.VectorizedOnPolicyBuffer(Sp(1), Sp(1), size=T, num_envs=N, gamma=0.99, lam=0.95, lam_c=0.9)
        for t in range(T):
            buf.store(obs=torch.zeros(N, 1), act=torch.zeros(N, 1), reward=rew[:, t], cost=cost[:, t],
                      value_r=v_r[:, t], value_c=v_c[:, t], log_prob=torch.zeros(N))
            for n in range(N):
                if seg[n, t]:
                    buf.finish_path(boot_r[n, t].reshape(1), boot_c[n, t].reshape(1), idx=n)
        raw = {k: torch.stack([b[k] for b in buf.buffers]).clone() for k in ("adv_r", "adv_c", "target_value_r", "target_value_c")}
        data = buf.get()
        cases.append(dict(rew=rew, cost=cost, v_r=v_r, v_c=v_c, seg_end=seg.to(torch.uint8), boot_r=boot_r, boot_c=boot_c,
                          lam=0.95, lam_c=0.9, gamma=0.99, raw=raw,
                          get={k: data[k].clone() for k in ("adv_r", "adv_c", "target_value_r", "target_value_c")}))
    out["gae_cases"] = cases


def gen_lagrange(ref, out):
    L = ref["lagrange"].Lagrange(25.0, 0.001, 0.035)
    seq = []
    for jc in (0.0, 50.0, 50.0, 10.0, 31.5, 2.0):
        L.update_lagrange_multiplier(jc)
        seq.append(L.lagrangian_multiplier)
    L2 = ref["lagrange"].Lagrange(25.0, 0.001, 0.035, lagrangian_upper_bound=2.0)
    seq2 = []
    for jc in (500.0,) * 80:
        L2.update_lagrange_multiplier(jc)
        seq2.append(L2.lagrangian_multiplier)
    out["lagrange"] = dict(jc=[0.0, 50.0, 50.0, 10.0, 31.5, 2.0], lam=seq, capped=seq2)


def _make_data(pol, S, D, A, seed):
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(S, D, generator=g)
    with torch.no_grad():
        dist = pol.actor(obs)
        act = dist.mean + dist.stddev * torch.randn(S, A, generator=g)
        logp = dist.log_prob(act).sum(-1)
        vr, vc = pol.reward_critic(obs), pol.cost_critic(obs)
    return dict(obs=obs, act=act, log_prob=logp, target_value_r=vr + torch.randn(S, generator=g),
                target_value_c=vc + torch.randn(S, generator=g).abs(), adv_r=torch.randn(S, generator=g),
                adv_c=torch.randn(S, generator=g))


def gen_update_chain(ref, out):
    """N consecutive minibatch steps of ppo_lag.py:298-336 and focops.py:309-357 driven
    with explicit index lists (DataLoader order checked separately)."""
    from torch.nn.utils.clip_grad import clip_grad_norm_
    from torch.distributions import Normal
    res = {}
    for kind in ("ppo", "focops"):
        D, A, S, B = 60, 2, 1000, 64
        torch.manual_seed(5)
        pol = ref["model"].ActorVCritic(D, A, [64, 64])
        with torch.no_grad():
            pol.actor.log_std.copy_(torch.tensor([-0.2, 0.1]))
        init = state_of(pol)
        data = _make_data(pol, S, D, A, 77)
        lam = 0.37
        adv = (data["adv_r"] - lam * data["adv_c"]) / (lam + 1)
        with torch.no_grad():
            od = pol.actor(data["obs"])
            old_mean, old_std = od.mean.clone(), od.stddev.clone()
        opt_a = torch.optim.Adam(pol.actor.parameters(), lr=3e-4)
        opt_r = torch.optim.Adam(pol.reward_critic.parameters(), lr=3e-4)
        opt_c = torch.optim.Adam(pol.cost_critic.parameters(), lr=3e-4)
        g = torch.Generator().manual_seed(3)
        perms = [torch.randperm(S, generator=g) for _ in range(8)]
        losses, kls = [], []
        for perm in perms:
            for s in range(0, S, B):
                idx = perm[s:s + B]
                obs_b, act_b, lp_b = data["obs"][idx], data["act"][idx], data["log_prob"][idx]
                opt_r.zero_grad()
                loss_r = torch.nn.functional.mse_loss(pol.reward_critic(obs_b), data["target_value_r"][idx])
                opt_c.zero_grad()
                loss_c = torch.nn.functional.mse_loss(pol.cost_critic(obs_b), data["target_value_c"][idx])
                for p in pol.reward_critic.parameters():
                    loss_r += p.pow(2).sum() * 0.001
                for p in pol.cost_critic.parameters():
                    loss_c += p.pow(2).sum() * 0.001
                dist = pol.actor(obs_b)
                log_prob = dist.log_prob(act_b).sum(dim=-1)
                ratio = torch.exp(log_prob - lp_b)
                if kind == "ppo":
                    loss_pi = -torch.min(ratio * adv[idx], torch.clamp(ratio, 0.8, 1.2) * adv[idx]).mean()
                else:
                    old_b = Normal(loc=old_mean[idx], scale=old_std[idx])
                    temp_kl = torch.distributions.kl_divergence(dist, old_b).sum(-1, keepdim=True)
                    loss_pi = ((temp_kl - (1 / 1.5) * ratio * adv[idx]) * (temp_kl.detach() <= 0.02).type(torch.float32)).mean()
                opt_a.zero_grad()
                (loss_pi + loss_r + loss_c).backward()
                clip_grad_norm_(pol.parameters(), 40.0)
                opt_r.step(); opt_c.step(); opt_a.step()
                losses.append((loss_r.item(), loss_c.item(), loss_pi.item()))
            with torch.no_grad():
                nd = pol.actor(data["obs"])
                kls.append(torch.distributions.kl.kl_divergence(od, nd).sum(-1, keepdim=True).mean().item())
        res[kind] = dict(D=D, A=A, init=init, data=data, lam=lam, perms=perms, losses=torch.tensor(losses),
                         kls=torch.tensor(kls), final=state_of(pol), batch=B)
    # both kinds start from the same seeded weights, data and minibatch orders: the file keeps one copy of them
    for key in ("init", "data", "perms"):
        torch.testing.assert_close(res["focops"][key], res["ppo"][key], rtol=0, atol=0)
        res["focops"][key] = res["ppo"][key]
    out["update_chain"] = res


def gen_dataloader(ref, out):
    from torch.utils.data import DataLoader, TensorDataset
    torch.manual_seed(11)
    S = 257
    dl = DataLoader(TensorDataset(torch.arange(S)), batch_size=64, shuffle=True)
    orders = []
    for _ in range(3):
        orders.append(torch.cat([b[0] for b in dl]))
    out["dataloader"] = dict(seed=11, S=S, orders=orders)


def gen_trust(ref, out):
    cpo = ref["cpo"]
    D, A, S = 88, 2, 512
    torch.manual_seed(9)
    pol = ref["model"].ActorVCritic(D, A, [64, 64])
    with torch.no_grad():
        pol.actor.log_std.copy_(torch.tensor([-0.3, 0.2]))
    data = _make_data(pol, S, D, A, 21)
    g = torch.Generator().manual_seed(4)
    P = sum(p.numel() for p in pol.actor.parameters())
    v = torch.randn(P, generator=g)
    Fv = cpo.fvp(v, pol, data["obs"]).detach().clone()
    rhs = torch.randn(P, generator=g)
    x = cpo.conjugate_gradients(cpo.fvp, pol, data["obs"], rhs, 15).detach().clone()
    pol.actor.zero_grad()
    dist = pol.actor(data["obs"])
    ratio = torch.exp(dist.log_prob(data["act"]).sum(-1) - data["log_prob"])
    loss = (ratio * data["adv_r"]).mean()
    loss.backward()
    grad = cpo.get_flat_gradients_from(pol.actor).clone()
    theta = cpo.get_flat_params_from(pol.actor).clone()
    names = [n for n, _ in pol.actor.named_parameters()]
    out["trust"] = dict(D=D, A=A, state=state_of(pol), data=data, v=v, Fv=Fv, rhs=rhs, cg_x=x, surr=loss.detach(),
                        surr_grad=grad, theta=theta, names=names, P=P)


def run_reference_main(ref, algo, args_kw, env_kw):
    """Drive the reference's own main() with the synthetic vector env injected."""
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "spo_synthetic_env", os.path.join(ROOT, "safe-policy-optimization_b200", "safepo", "common", "synthetic_env.py"))
    senv = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(senv)
    SyntheticVecEnv, TASK_DIMS = senv.SyntheticVecEnv, senv.TASK_DIMS
    from oracle.trainers import default_args
    mod = ref[algo]
    tmp = tempfile.mkdtemp()
    args = default_args(**args_kw)
    args.log_dir = os.path.join(tmp, "exp", args.task, algo, "run")
    D, A = TASK_DIMS[args.task]

    def fake_make(num_envs, env_id, seed=None):
        env = SyntheticVecEnv(num_envs, D, A, seed=0 if seed is None else seed, **env_kw)
        return env, env.observation_space, env.action_space

    mod.make_sa_mujoco_env = fake_make
    mod.main(args, {})
    with open(os.path.join(args.log_dir, "progress.csv")) as f:
        rows = list(csv.DictReader(f))
    model_dir = os.path.join(args.log_dir, "torch_save")
    last = sorted(os.listdir(model_dir), key=lambda s: int(s[5:-3]))[-1]
    return rows, torch.load(os.path.join(model_dir, last)), sorted(os.listdir(args.log_dir))


def gen_main_runs(ref, out):
    runs = {}
    cfgs = {
        "ppo_lag": (dict(seed=3, num_envs=3, steps_per_epoch=3 * 70, total_steps=3 * 70 * 2), dict(episode_len=25, stagger=True, p_terminate=0.02)),
        "focops": (dict(seed=4, num_envs=2, steps_per_epoch=2 * 90, total_steps=2 * 90 * 2), dict(episode_len=30, stagger=True, p_terminate=0.02)),
        "cpo": (dict(seed=5, num_envs=3, steps_per_epoch=3 * 80, total_steps=3 * 80 * 2, task="SafetyCarButton1-v0"), dict(episode_len=20, stagger=True, p_terminate=0.02)),
        "trpo_lag": (dict(seed=6, num_envs=2, steps_per_epoch=2 * 100, total_steps=2 * 100 * 2), dict(episode_len=40, stagger=True, p_terminate=0.02)),
    }
    for algo, (akw, ekw) in cfgs.items():
        rows, actor_sd, files = run_reference_main(ref, algo, akw, ekw)
        runs[algo] = dict(args=akw, env=ekw, rows=rows, actor=actor_sd, files=files)
        print(algo, "rows:", len(rows), "files:", files)
    out["main_runs"] = runs


def gen_siblings(ref, out):
    """SURVEY 8f rank 2: main() of the sibling scripts ppo / pg / cppo_pid / trpo on the synthetic env, and a
    PIDLagrangian sequence (safepo/common/lagrange.py:108-200)."""
    runs = {}
    cfgs = {
        "ppo": (dict(seed=7, num_envs=3, steps_per_epoch=3 * 70, total_steps=3 * 70 * 2), dict(episode_len=25, stagger=True, p_terminate=0.02)),
        "pg": (dict(seed=8, num_envs=2, steps_per_epoch=2 * 90, total_steps=2 * 90 * 2), dict(episode_len=30, stagger=True, p_terminate=0.02)),
        "cppo_pid": (dict(seed=9, num_envs=3, steps_per_epoch=3 * 70, total_steps=3 * 70 * 3, cost_limit=5.0),
                     dict(episode_len=25, stagger=True, p_terminate=0.02)),
        "trpo": (dict(seed=10, num_envs=2, steps_per_epoch=2 * 100, total_steps=2 * 100 * 2), dict(episode_len=40, stagger=True, p_terminate=0.02)),
        "natural_pg": (dict(seed=11, num_envs=2, steps_per_epoch=2 * 100, total_steps=2 * 100 * 2), dict(episode_len=40, stagger=True, p_terminate=0.02)),
        "rcpo": (dict(seed=12, num_envs=3, steps_per_epoch=3 * 80, total_steps=3 * 80 * 2), dict(episode_len=20, stagger=True, p_terminate=0.02)),
        "cup": (dict(seed=14, num_envs=3, steps_per_epoch=3 * 70, total_steps=3 * 70 * 3, cost_limit=0.2),
                dict(episode_len=25, stagger=True, p_terminate=0.02)),
        "pcpo": (dict(seed=13, num_envs=3, steps_per_epoch=3 * 80, total_steps=3 * 80 * 2, task="SafetyCarButton1-v0", cost_limit=8.0),
                 dict(episode_len=20, stagger=True, p_terminate=0.02)),
    }
    for algo, (akw, ekw) in cfgs.items():
        rows, actor_sd, files = run_reference_main(ref, algo, akw, ekw)
        runs[algo] = dict(args=akw, env=ekw, rows=rows, actor=actor_sd, files=files)
        print(algo, "rows:", len(rows), "files:", files)
    out["main_runs"] = runs
    P = ref["lagrange"].PIDLagrangian(25.0, 0.001)
    jcs = [0.0, 50.0, 50.0, 10.0, 31.5, 2.0, 80.0, 80.0, 80.0, 26.0, 24.0, 3.0, 90.0, 12.5]
    seq = []
    for jc in jcs:
        P.update_lagrange_multiplier(jc)
        seq.append(P.lagrangian_multiplier)
    out["pid"] = dict(jc=jcs, lam=seq)


def gen_ma_gae(ref, out):
    """SURVEY 8 row G2: SeparatedReplayBuffer.compute_returns / compute_cost_returns (buffer.py:356-384) with a PopArt
    value normaliser (popart.py).  The buffer methods are called unbound on a bare namespace holding exactly the
    attributes they touch, so the arithmetic is the reference's own without building gymnasium spaces."""
    import importlib
    from types import SimpleNamespace
    buf_mod = ref["buffer"]
    popart_mod = importlib.import_module("safepo.common.popart")
    cases = []
    for (T, N, seed, gamma, lam) in ((8, 5, 0, 0.96, 0.95), (64, 3, 1, 0.99, 0.95), (1, 4, 2, 0.96, 0.95), (33, 16, 3, 0.96, 0.9)):
        g = torch.Generator().manual_seed(seed)
        pop = popart_mod.PopArt(1)
        trained = []
        for _ in range(3):                                   # move the running statistics off their initial zeros
            x = torch.randn(40, 1, generator=g) * 3 + 1.5
            trained.append((x.clone(), pop(x).clone()))
        value_preds = torch.randn(T + 1, N, 1, generator=g)
        cost_preds = torch.randn(T + 1, N, 1, generator=g)
        rewards = torch.randn(T, N, 1, generator=g)
        costs = torch.rand(T, N, 1, generator=g)
        masks = (torch.rand(T + 1, N, 1, generator=g) > 0.15).float()
        ns = SimpleNamespace(value_preds=value_preds.clone(), cost_preds=cost_preds.clone(), rewards=rewards, costs=costs, masks=masks,
                             gamma=gamma, gae_lambda=lam, returns=torch.zeros(T + 1, N, 1), cost_returns=torch.zeros(T + 1, N, 1))
        next_value, next_cost = value_preds[-1].clone(), cost_preds[-1].clone()
        buf_mod.SeparatedReplayBuffer.compute_returns(ns, next_value, pop)
        buf_mod.SeparatedReplayBuffer.compute_cost_returns(ns, next_cost, pop)
        cases.append(dict(T=T, N=N, gamma=gamma, lam=lam, popart_inputs=[t[0] for t in trained], popart_outputs=[t[1] for t in trained],
                          popart_state=(pop.running_mean.clone(), pop.running_mean_sq.clone(), pop.debiasing_term.clone()),
                          denorm_probe=pop.denormalize(value_preds[:2]).clone(), value_preds=value_preds, cost_preds=cost_preds,
                          rewards=rewards, costs=costs, masks=masks, returns=ns.returns.clone(), cost_returns=ns.cost_returns.clone()))
    out["ma_gae"] = cases


def gen_ma_update(ref, out):
    """MAPPO-Lag networks and two consecutive ppo_update calls through the reference's own MAPPO_L_Policy /
    MAPPO_L_Trainer (safepo/multi_agent/mappolag.py:46-199) at small dimensions (obs 10, share_obs 14, act 3, hidden 32,
    the yaml's layer_N = 2): initial state dicts, get_actions outputs (deterministic and sampled under a fixed seed), the
    sample, and after each update the returned scalars, lamda_lagr, the PopArt state and all three state dicts."""
    import yaml
    m = importlib.import_module("safepo.multi_agent.mappolag")
    cfg = yaml.safe_load(open(os.path.join(REF, "safepo", "multi_agent", "marl_cfg", "mappolag", "config.yaml")))
    cfg.update(device="cpu", algorithm_name="mappolag", n_rollout_threads=4, hidden_size=32)

    class Sp:
        def __init__(self, d):
            self.shape = (d,)

    # one intra-op thread: the parameter-shaped reductions of LayerNorm's backward split their rows over the threads, so the last
    # bit of a gradient depends on the thread count (the test pins the same setting)
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    torch.manual_seed(11)
    D, DS, A, N = 10, 14, 3, 24
    pol = m.MAPPO_L_Policy(cfg, Sp(D), Sp(DS), Sp(A))
    with torch.no_grad():       # move the LayerNorm affine parameters and biases off their trivial initial values
        for net in (pol.actor, pol.critic, pol.cost_critic):
            for k, v in net.state_dict().items():
                if k.endswith("bias") or ".2.weight" in k or "feature_norm" in k or k.endswith("log_std"):
                    v.add_(0.1 * torch.randn_like(v))
    tr = m.MAPPO_L_Trainer(cfg, pol)
    g = torch.Generator().manual_seed(12)
    obs, share = torch.randn(N, D, generator=g) * 2 + 0.5, torch.randn(N, DS, generator=g) * 3
    rnn, masks = np.zeros((N, 1, 32), dtype=np.float32), np.ones((N, 1), dtype=np.float32)
    init_state = {n: {k: v.clone() for k, v in getattr(pol, n).state_dict().items()} for n in ("actor", "critic", "cost_critic")}
    with torch.no_grad():
        det = pol.get_actions(share, obs, rnn, rnn, masks, deterministic=True, rnn_states_cost=rnn)
        torch.manual_seed(99)
        smp = pol.get_actions(share, obs, rnn, rnn, masks, deterministic=False, rnn_states_cost=rnn)
    acts = {"det": dict(values=det[0], actions=det[1], logp=det[2], cost=det[5]),
            "sampled": dict(values=smp[0], actions=smp[1], logp=smp[2], cost=smp[5], seed=99)}
    sample = dict(share_obs=share, obs=obs, actions=smp[1].clone(), value_preds=det[0].clone() + 0.1 * torch.randn(N, 1, generator=g),
                  returns=torch.randn(N, 1, generator=g) * 4 + 1, old_action_log_probs=smp[2].clone() + 0.05 * torch.randn(N, A, generator=g),
                  adv_targ=torch.randn(N, 1, generator=g), factor=torch.rand(N, 1, generator=g) + 0.5,
                  cost_preds=det[5].clone() + 0.1 * torch.randn(N, 1, generator=g), cost_returns=torch.randn(N, 1, generator=g).abs() * 30,
                  cost_adv_targ=torch.randn(N, 1, generator=g), aver_episode_costs=torch.rand(N, 1, generator=g) * 60)
    steps = []
    for _ in range(2):
        tup = (sample["share_obs"].numpy(), sample["obs"].numpy(), rnn, rnn, sample["actions"].numpy(), sample["value_preds"],
               sample["returns"], masks, masks, sample["old_action_log_probs"], sample["adv_targ"], None, sample["factor"],
               sample["cost_preds"], sample["cost_returns"], rnn, sample["cost_adv_targ"], sample["aver_episode_costs"])
        r = tr.ppo_update(tup)
        names = ("value_loss", "critic_grad_norm", "policy_loss", "dist_entropy", "actor_grad_norm", "imp_weights", "cost_loss", "cost_grad_norm")
        vn = tr.value_normalizer
        steps.append(dict(out={k: v.detach().clone() for k, v in zip(names, r)}, lamda_lagr=torch.as_tensor(tr.lamda_lagr).clone(),
                          popart=(vn.running_mean.clone(), vn.running_mean_sq.clone(), vn.debiasing_term.clone()),
                          state={n: {k: v.clone() for k, v in getattr(pol, n).state_dict().items()} for n in ("actor", "critic", "cost_critic")}))
    keep = ("actor_lr", "critic_lr", "opti_eps", "weight_decay", "clip_param", "huber_delta", "entropy_coef", "max_grad_norm", "cost_limit",
            "gamma", "lagrangian_coef_rate", "value_loss_coef", "lamda_lagr", "layer_N", "std_x_coef", "std_y_coef")
    torch.set_num_threads(threads)
    out["ma_update"] = dict(cfg={k: cfg[k] for k in keep}, dims=(D, DS, A, N), init=init_state, actions=acts, sample=sample, steps=steps)


def gen_ma_epoch(ref, out):
    """Two whole MAPPO-Lag training iterations of TWO agents through the reference's own Runner methods (collect / insert /
    compute / train of safepo/multi_agent/mappolag.py:402-504,583-597, called on a stand-in ``self`` that carries the real
    MAPPO_L_Policy / MAPPO_L_Trainer / SeparatedReplayBuffer objects -- the Runner's constructor needs environments that are not
    installable here) on a synthetic environment stream: T = 4 steps, 6 envs, hidden 32, learning_iters 2.  Stored: the initial
    state dicts, the env stream, the global-RNG seed, and after every iteration the buffers' returns / cost returns / factor,
    lamda_lagr, the PopArt state and every state dict."""
    import yaml
    m = importlib.import_module("safepo.multi_agent.mappolag")
    cfg = yaml.safe_load(open(os.path.join(REF, "safepo", "multi_agent", "marl_cfg", "mappolag", "config.yaml")))
    T, N, D, DS, A, H, NA = 4, 6, 10, 14, 3, 32, 2
    cfg.update(device="cpu", algorithm_name="mappolag", n_rollout_threads=N, hidden_size=H, episode_length=T, learning_iters=2,
               env_name="synthetic", entropy_coef=0.01)

    class Sp:
        def __init__(self, d):
            self.shape = (d,)

    class Log:
        def store(self, **kw):
            pass

    threads = torch.get_num_threads()
    torch.set_num_threads(1)          # LayerNorm's backward reductions depend on the intra-op thread count (see gen_ma_update)
    torch.manual_seed(21)
    policy = [m.MAPPO_L_Policy(cfg, Sp(D), Sp(DS), Sp(A)) for _ in range(NA)]
    with torch.no_grad():
        for pol in policy:
            for net in (pol.actor, pol.critic, pol.cost_critic):
                for k, v in net.state_dict().items():
                    if k.endswith("bias") or ".2.weight" in k or "feature_norm" in k or k.endswith("log_std"):
                        v.add_(0.1 * torch.randn_like(v))
    init_state = [{n: {k: v.clone() for k, v in getattr(pol, n).state_dict().items()} for n in ("actor", "critic", "cost_critic")} for pol in policy]
    fake = types.SimpleNamespace(config=cfg, num_agents=NA, logger=Log(), policy=policy,
                                 trainer=[m.MAPPO_L_Trainer(cfg, pol) for pol in policy],
                                 buffer=[m.SeparatedReplayBuffer(cfg, Sp(D), Sp(DS), Sp(A)) for _ in range(NA)])
    g = torch.Generator().manual_seed(22)
    obs0, share0 = torch.randn(N, NA, D, generator=g) * 2 + 0.5, torch.randn(N, NA, DS, generator=g) * 3
    for a in range(NA):                                    # Runner.warmup
        fake.buffer[a].share_obs[0].copy_(share0[:, a])
        fake.buffer[a].obs[0].copy_(obs0[:, a])
    stream, iters = [], []
    seed = 77
    torch.manual_seed(seed)
    train_episode_costs = torch.zeros(1, N)
    for it in range(2):
        steps = []
        for step in range(T):
            values, actions, action_log_probs, rnn_states, rnn_states_critic, cost_preds, rnn_states_cost = m.Runner.collect(fake, step)
            obs, share_obs = torch.randn(N, NA, D, generator=g) * 2 + 0.5, torch.randn(N, NA, DS, generator=g) * 3
            rewards, costs = torch.randn(N, NA, 1, generator=g), (torch.rand(N, NA, 1, generator=g) < 0.3).float()
            done_env = torch.rand(N, generator=g) < 0.2
            # all agents of an env finish together: an agent finishing alone zeroes its active mask, and MAPPO_L_Trainer.train
            # (mappolag.py:202-205) then takes torch.mean over a copy with NaNs written into it -- the reference's own update
            # turns to NaN in that case (it means nanmean), so only the all-or-none case is a usable fixture
            dones = done_env[:, None].expand(N, NA).clone()
            train_episode_costs += torch.mean(costs, dim=1).flatten()
            for t in range(N):
                if bool(torch.all(dones, dim=1)[t]):
                    train_episode_costs[:, t] = 0
            data = (obs, share_obs, rewards, costs, dones, None, values, actions, action_log_probs, rnn_states, rnn_states_critic,
                    cost_preds, rnn_states_cost, train_episode_costs.mean())
            m.Runner.insert(fake, data)
            steps.append(dict(obs=obs, share_obs=share_obs, rewards=rewards, costs=costs, dones=dones,
                              values=values.clone(), actions=[x.clone() for x in actions], action_log_probs=[x.clone() for x in action_log_probs],
                              cost_preds=cost_preds.clone()))
        m.Runner.compute(fake)
        after_compute = [dict(returns=b.returns.clone(), cost_returns=b.cost_returns.clone(), value_preds=b.value_preds.clone(),
                              cost_preds=b.cost_preds.clone(), masks=b.masks.clone(), active_masks=b.active_masks.clone()) for b in fake.buffer]
        m.Runner.train(fake)
        res = []
        for a in range(NA):
            tr, vn = fake.trainer[a], fake.trainer[a].value_normalizer
            res.append(dict(factor=fake.buffer[a].factor.clone(), lamda_lagr=torch.as_tensor(tr.lamda_lagr).clone(),
                            popart=(vn.running_mean.clone(), vn.running_mean_sq.clone(), vn.debiasing_term.clone()),
                            state={n: {k: v.clone() for k, v in getattr(policy[a], n).state_dict().items()} for n in ("actor", "critic", "cost_critic")}))
        stream.append(steps)
        iters.append(dict(after_compute=after_compute, agents=res))
        if it == 0:                                          # Runner.return_aver_cost after an iteration with finished episodes
            for a in range(NA):
                fake.buffer[a].return_aver_insert(torch.tensor(31.5))
    keep = ("actor_lr", "critic_lr", "opti_eps", "weight_decay", "clip_param", "huber_delta", "entropy_coef", "max_grad_norm", "cost_limit",
            "gamma", "gae_lambda", "lagrangian_coef_rate", "value_loss_coef", "lamda_lagr", "layer_N", "std_x_coef", "std_y_coef", "learning_iters",
            "num_mini_batch", "episode_length", "n_rollout_threads")
    torch.set_num_threads(threads)
    out["ma_epoch"] = dict(cfg={k: cfg[k] for k in keep}, dims=(T, N, D, DS, A, H, NA), init=init_state, obs0=obs0, share_obs0=share0, seed=seed,
                           stream=stream, iters=iters, aver_cost_after_first=31.5)


def main():
    sys.path.insert(0, ROOT)
    ref = import_reference()
    only = set(sys.argv[1:])      # e.g. `python make_golden.py siblings` regenerates one fixture
    for name, fn in (("forward", gen_forward), ("gae", gen_gae), ("lagrange", gen_lagrange), ("update", gen_update_chain),
                     ("dataloader", gen_dataloader), ("trust", gen_trust), ("main_runs", gen_main_runs), ("siblings", gen_siblings), ("ma_gae", gen_ma_gae), ("ma_update", gen_ma_update), ("ma_epoch", gen_ma_epoch)):
        if only and name not in only:
            continue
        out = {}
        fn(ref, out)
        path = os.path.join(HERE, f"{name}.pt")
        torch.save(out, path)
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
