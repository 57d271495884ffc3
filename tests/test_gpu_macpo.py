"""MACPO on the B200 against the CPU oracle (oracle/macpo_oracle.py, itself pinned bit for bit to the reference by
tests/test_macpo_cpu.py): the Fisher-vector product at three shapes, the surrogate gradients and CG solutions, a full
trpo_update per optim_case and for an all-rejected line search, two runner iterations of two agents and the CLI."""
import csv
import math
import os

import pytest
import torch

from oracle import ma_oracle as MA
from oracle import macpo_oracle as MO

pytestmark = pytest.mark.gpu

CFG = dict(critic_lr=5e-3, opti_eps=1e-5, weight_decay=0.0, clip_param=0.2, huber_delta=10.0, max_grad_norm=10.0, cost_limit=25.0, gamma=0.96,
           gae_lambda=0.95, value_loss_coef=1.0, layer_N=2, std_x_coef=1.0, std_y_coef=0.5, target_kl=0.016, searching_steps=10,
           conjugate_gradient_iters=10, step_fraction=0.5, fraction_coef=0.1)


def _states(D, DS, H, A, layer_N, seed):
    from safepo.multi_agent.mappolag import init_state
    g = torch.Generator().manual_seed(seed)
    out = []
    for head, d in (("actor", D), ("critic", DS), ("critic", DS)):
        st = init_state(d, H, layer_N, head, A, generator=g)
        out.append({k: v + 0.1 * torch.randn(v.shape, generator=g) for k, v in st.items()})
    return out, g


def _device(states, layer_N, cfg):
    from safepo.common.ma_model import MACPOTrainer, MultiAgentNets
    nets = MultiAgentNets(*states, "cuda", layer_N=layer_N)
    return nets, MACPOTrainer(nets, dict(cfg, layer_N=layer_N))


@pytest.mark.parametrize("shape", [(10, 128, 3, 100, 2), (38, 256, 5, 300, 1), (398, 512, 20, 2048, 2)])
def test_fvp_matches_double_backprop(shape):
    D, H, A, n, layer_N = shape
    states, g = _states(D, 14, H, A, layer_N, 7)
    obs = torch.randn(n, D, generator=g) * 2 + 0.5
    nets, tr = _device(states, layer_N, CFG)
    v = torch.zeros(tr._count, device="cuda")
    tv = tr._tangents(v)
    for k, t in tv.items():
        t.copy_(torch.randn(t.shape, generator=g).cuda())
    out = torch.full_like(v, float("nan"))
    tr.fvp(obs.cuda(), v, out)
    actor = MA.OracleMANet({k: x.double() for k, x in states[0].items()}, layer_N=layer_N)
    otr = MO.OracleMACPOTrainer.__new__(MO.OracleMACPOTrainer)
    otr.actor, otr.cfg = actor, CFG
    want = otr.fisher_vector_product(obs.double(), torch.zeros(n, A, dtype=torch.float64), torch.cat([tv[k].cpu().double().reshape(-1) for k in tv]))
    got = tr._tangents(out)
    i, worst = 0, 0.0
    for k, p in actor.p.items():
        w = want[i:i + p.numel()].view(p.shape)
        i += p.numel()
        err = float((got[k].cpu().double() - w).abs().max() / w.abs().max())
        worst = max(worst, err)
        assert err <= 5e-5, (k, err)
    pads = torch.ones(tr._count, dtype=torch.bool, device="cuda")
    for t in tr._tangents(pads).values():
        t.fill_(False)
    assert bool((out[pads] == 0).all())
    print(f"fvp {shape}: worst per-tensor error / max-abs = {worst:.2e}")


CASES = (("case0", 80.0, {}, False), ("case1", 25.5, {}, False), ("case2", 24.9, {}, False), ("case3", 0.0, {}, False), ("case4", 10.0, {}, True),
         ("rejected", 0.0, {"target_kl": 1e-6, "fraction_coef": 1e5}, False))


def _sample(D, DS, A, n, aver, zero_cost_adv, g, states):
    actor = MA.OracleMANet(states[0])
    obs, share = torch.randn(n, D, generator=g) * 2 + 0.5, torch.randn(n, DS, generator=g) * 3
    with torch.no_grad():
        dist = MA.ma_actor_dist(actor, obs)
        actions = dist.mean + dist.stddev * torch.randn(n, A, generator=g)
        logp = dist.log_prob(actions) + 0.05 * torch.randn(n, A, generator=g)
    return dict(share_obs=share, obs=obs, actions=actions, value_preds=torch.randn(n, 1, generator=g), returns=torch.randn(n, 1, generator=g) * 4 + 1,
                old_action_log_probs=logp, adv_targ=torch.randn(n, 1, generator=g), factor=torch.rand(n, 1, generator=g) + 0.5,
                cost_preds=torch.randn(n, 1, generator=g), cost_returns=torch.randn(n, 1, generator=g).abs() * 30,
                cost_adv_targ=torch.zeros(n, 1) if zero_cost_adv else torch.randn(n, 1, generator=g),
                aver_episode_costs=torch.full((n, 1), aver) + 0.01 * torch.randn(n, 1, generator=g))


def _rel(a, b):
    return float((a.cpu() - b).norm() / b.norm().clamp_min(1e-30))


@pytest.mark.parametrize("case", [c[0] for c in CASES])
def test_trpo_update_matches_oracle(case):
    _, aver, overrides, zero = next(c for c in CASES if c[0] == case)
    D, DS, H, A, n, layer_N = 10, 14, 128, 3, 256, 2
    cfg = dict(CFG, **overrides)
    states, g = _states(D, DS, H, A, layer_N, 11)
    s = _sample(D, DS, A, n, aver, zero, g, states)
    onets = tuple(MA.OracleMANet(st, layer_N=layer_N) for st in states)
    want = MO.OracleMACPOTrainer(*onets, cfg).trpo_update(s)
    nets, tr = _device(states, layer_N, cfg)
    got = tr.trpo_update({k: v.cuda() for k, v in s.items()})
    print(case, "oracle", want["optim_case"], want["accepted"], "device", got["optim_case"], got["accepted"])
    assert got["optim_case"] == want["optim_case"] and got["accepted"] == want["accepted"]
    packed = lambda v: torch.cat([t.reshape(-1) for t in tr._tangents(v).values()])      # noqa: E731
    assert _rel(packed(got["g"]), want["g"]) < 5e-3 and _rel(packed(got["b"]), want["b"]) < 5e-3 or float(want["b"].norm()) == 0
    assert _rel(packed(got["g_step_dir"]), want["g_step_dir"]) < 5e-3
    if want["optim_case"] != 4:
        assert _rel(packed(got["b_step_dir"]), want["b_step_dir"]) < 5e-3
        assert _rel(packed(got["x"]), want["x"]) < 5e-3
    step = max(float((onets[0].p[k].detach() - states[0][k]).abs().max()) for k in states[0])
    for k, v in onets[0].p.items():
        err = float((nets.actor.p[k].cpu() - v.detach()).abs().max())
        assert err <= 1e-2 * step + 1e-6, (k, err, step)
    for dn, on in ((nets.critic, onets[1]), (nets.cost_critic, onets[2])):
        for k, v in on.p.items():
            torch.testing.assert_close(dn.p[k].cpu(), v.detach(), rtol=1e-4, atol=1e-5)
    assert math.isclose(got["kl"], float(want["kl"]), rel_tol=1e-2, abs_tol=1e-7)
    assert math.isclose(got["ratio"], float(want["ratio"].mean()), rel_tol=1e-4)


def test_runner_two_iterations_matches_oracle():
    from safepo.multi_agent import macpo
    T, N, D, DS, A, H, NA, layer_N = 4, 32, 10, 14, 3, 128, 2, 2
    cfg = dict(CFG, episode_length=T, n_rollout_threads=N)
    g = torch.Generator().manual_seed(3)
    all_states = [_states(D, DS, H, A, layer_N, 20 + a)[0] for a in range(NA)]
    onets = [tuple(MA.OracleMANet(st, layer_N=layer_N) for st in states) for states in all_states]
    orun = MO.OracleMACPORunner(onets, cfg, T, N, D, DS, A)
    dnets = [macpo.MultiAgentNets(*states, "cuda", layer_N=layer_N) for states in all_states]
    drun = macpo.Runner(dnets, cfg, D, DS, A)
    obs0, share0 = torch.randn(N, NA, D, generator=g), torch.randn(N, NA, DS, generator=g)
    orun.warmup(obs0, share0)
    drun.warmup(obs0, share0)
    for it in range(2):
        for step in range(T):
            eps = [torch.randn(N, A, generator=g) for _ in range(NA)]
            ov, oa, ol, oc = orun.collect(step, eps=eps)
            dv, da, dl, dc = drun.collect(step, eps=eps)
            obs, share = torch.randn(N, NA, D, generator=g), torch.randn(N, NA, DS, generator=g)
            rew, cost = torch.randn(N, NA, 1, generator=g), (torch.rand(N, NA, 1, generator=g) < 0.3).float()
            dones = (torch.rand(N, generator=g) < 0.2)[:, None].expand(N, NA).clone()
            orun.insert(obs, share, rew, cost, dones, ov, oa, ol, oc)
            drun.insert(obs, share, rew, cost, dones, dv, da, dl, dc)
        orun.compute()
        drun.compute()
        perms = [[torch.randperm(T * N, generator=g)] for _ in range(NA)]
        order = [1, 0]
        outs = orun.train(agent_order=order, perms=[p[0] for p in perms])
        douts = drun.train(agent_order=order, perms=[[p[0].cuda()] for p in perms], collect_outputs=True)
        for a in range(NA):
            assert douts[a]["optim_case"] == outs[a]["optim_case"] and douts[a]["accepted"] == outs[a]["accepted"], (it, a)
            torch.testing.assert_close(drun.buffer[a].factor.cpu(), orun.buffer[a].factor, rtol=1e-3, atol=1e-4)
            for dn, on in zip((dnets[a].actor, dnets[a].critic, dnets[a].cost_critic), onets[a]):
                for k, v in on.p.items():
                    torch.testing.assert_close(dn.p[k].cpu(), v.detach(), rtol=1e-3, atol=1e-4)


def test_cli_synthetic_run(tmp_path):
    from safepo.multi_agent import macpo
    rows = macpo.main(["--env", "synthetic", "--num-envs", "64", "--obs-dim", "24", "--share-obs-dim", "30", "--act-dim", "4", "--hidden-size", "128",
                       "--iterations", "3", "--episode-len", "5", "--log-dir", str(tmp_path)])
    assert len(rows) == 3
    path = os.path.join(str(tmp_path), "progress.csv")
    with open(path) as f:
        table = list(csv.DictReader(f))
    assert table and "Misc/KL/agent0" in table[0]
    for r in table:
        for k, v in r.items():
            if v not in ("", None):
                assert math.isfinite(float(v)), (k, v)
