"""MACPO on the CPU: the oracle (oracle/macpo_oracle.py) pinned bit for bit against the reference's own MACPO_Trainer and
Runner (tests/golden/macpo.pt), the closed-form Fisher-vector product the kernels implement against the oracle's double
backprop in float64, and the host orchestration of MACPOTrainer / macpo.Runner through an emulated C-ABI."""
import pytest
import torch

from oracle import ma_oracle as MA
from oracle import macpo_oracle as MO


@pytest.fixture()
def one_thread():
    threads = torch.get_num_threads()
    torch.set_num_threads(1)        # LayerNorm's backward reductions depend on the intra-op thread count (as in the fixture)
    yield
    torch.set_num_threads(threads)


def _nets(init, layer_N):
    return tuple(MA.OracleMANet(init[n], layer_N=layer_N) for n in ("actor", "critic", "cost_critic"))


def _sample(c):
    s = dict(c["sample"])
    return s


def test_oracle_fvp_bit_exact(golden, one_thread):
    u = golden("macpo")["update"]
    actor, critic, cost_critic = _nets(u["init"], u["cfg"]["layer_N"])
    tr = MO.OracleMACPOTrainer(actor, critic, cost_critic, u["cfg"])
    s = u["cases"][0]["sample"]
    got = tr.fisher_vector_product(s["obs"], s["actions"], u["fvp"]["p"].clone())
    assert torch.equal(got, u["fvp"]["out"])


@pytest.mark.parametrize("case", ["case0", "case1", "case2", "case3", "case4", "rejected"])
def test_oracle_trpo_update_bit_exact(golden, one_thread, case):
    u = golden("macpo")["update"]
    c = next(x for x in u["cases"] if x["name"] == case)
    critics = u["cases"][0]["critics"]
    cfg = dict(u["cfg"], **c["cfg_overrides"])
    actor, critic, cost_critic = _nets(u["init"], cfg["layer_N"])
    tr = MO.OracleMACPOTrainer(actor, critic, cost_critic, cfg)
    out = tr.trpo_update(_sample(c))
    assert out["optim_case"] == c["optim_case"] and out["accepted"] == c["accepted"]
    for k, want in c["out"].items():
        got = out[k]
        assert torch.equal(torch.as_tensor(got).reshape(-1).float(), torch.as_tensor(want).reshape(-1).float()), k
    if c["vectors"] is not None:
        for k, want in c["vectors"].items():
            assert torch.equal(out[k], want), k
    for k, v in c["actor"].items():
        assert torch.equal(actor.p[k].detach(), v), k
    for n, net in (("critic", critic), ("cost_critic", cost_critic)):
        for k, v in critics[n].items():
            assert torch.equal(net.p[k].detach(), v), (n, k)
    for got, want in zip((tr.popart.running_mean, tr.popart.running_mean_sq, tr.popart.debiasing_term), critics["popart"]):
        assert torch.equal(got.reshape(-1), want.reshape(-1))


def test_fixture_covers_every_case(golden):
    cases = golden("macpo")["update"]["cases"]
    assert sorted(c["optim_case"] for c in cases if c["accepted"] >= 0) == [0, 1, 2, 3, 4]
    assert any(c["accepted"] == -1 for c in cases)


def test_oracle_runner_two_iterations_bit_exact(golden, one_thread):
    e = golden("macpo")["epoch"]
    T, N, D, DS, A, H, NA = e["dims"]
    cfg = e["cfg"]
    nets = [_nets(st, cfg["layer_N"]) for st in e["init"]]
    run = MO.OracleMACPORunner(nets, cfg, T, N, D, DS, A)
    run.warmup(e["obs0"], e["share_obs0"])
    torch.manual_seed(e["seed"])
    for it in range(2):
        for step in range(T):
            s = e["stream"][it][step]
            values, actions, logps, cost_preds = run.collect(step)
            run.insert(s["obs"], s["share_obs"], s["rewards"], s["costs"], s["dones"], values, actions, logps, cost_preds)
        run.compute()
        run.train()
        for a in range(NA):
            want = e["iters"][it]["agents"][a]
            b = run.buffer[a]
            assert torch.equal(b.factor, want["factor"]) and torch.equal(b.returns, want["returns"]), (it, a)
            assert torch.equal(b.cost_returns, want["cost_returns"]), (it, a)
            pop = run.trainer[a].popart
            for got, w in zip((pop.running_mean, pop.running_mean_sq, pop.debiasing_term), want["popart"]):
                assert torch.equal(got.reshape(-1), w.reshape(-1)), (it, a)
            for n, net in zip(("actor", "critic", "cost_critic"), run.nets[a]):
                for k, v in want["state"].get(n, {}).items():
                    assert torch.equal(net.p[k].detach(), v), (it, a, n, k)
        if it == 0:
            for b in run.buffer:
                b.aver_episode_costs = torch.tensor(e["aver_cost_after_first"])
    assert any(bool((e["iters"][1]["agents"][a]["factor"] != 1).any()) for a in range(NA))


def _random_actor(D, H, A, layer_N, seed, dtype):
    from safepo.multi_agent.mappolag import init_state
    g = torch.Generator().manual_seed(seed)
    st = init_state(D, H, layer_N, "actor", A, generator=g)
    st = {k: (v + 0.1 * torch.randn(v.shape, generator=g)).to(dtype) for k, v in st.items()}
    return MA.OracleMANet(st, layer_N=layer_N), g


@pytest.mark.parametrize("shape", [(10, 32, 3, 24, 2), (37, 64, 5, 50, 1)])
def test_closed_form_fvp_matches_double_backprop(shape):
    """The formula of the device FVP (forward tangents, J^T diag(2/(1e-8+2 std^2)) J / n, the quirky log_std block, damping) against
    the reference's double backprop, both in float64."""
    D, H, A, n, layer_N = shape
    actor, g = _random_actor(D, H, A, layer_N, 5, torch.float64)
    obs = (torch.randn(n, D, generator=g) * 2 + 0.5).double()
    tr = MO.OracleMACPOTrainer.__new__(MO.OracleMACPOTrainer)
    tr.actor, tr.cfg = actor, dict(std_x_coef=1.0, std_y_coef=0.5)
    count = sum(v.numel() for v in actor.p.values())
    for _ in range(3):
        v = torch.randn(count, generator=g, dtype=torch.float64)
        want = tr.fisher_vector_product(obs, torch.zeros(n, A, dtype=torch.float64), v)
        got = MO.closed_form_fvp(actor, obs, v)
        assert float((got - want).abs().max() / want.abs().max()) < 1e-10


def test_quirky_log_std_curvature():
    """At the default initialisation (log_std = 1, std = sigmoid(1) / 2) the log_std block of the reference's "KL" is ~0.54,
    not the Gaussian Fisher's ~0.15."""
    sg = torch.sigmoid(torch.tensor(1.0, dtype=torch.float64))
    s, ds, dds = 0.5 * sg, 0.5 * sg * (1 - sg), 0.5 * sg * (1 - sg) * (1 - 2 * sg)
    D = 1e-8 + 2 * s ** 2
    quirky = (1 / s ** 2 - 4 * s ** 2 / D ** 2 + 32 * s ** 4 / D ** 3) * ds ** 2 + (-1 / s - 4 * s ** 3 / D ** 2) * dds
    assert abs(float(quirky) - 0.54) < 0.01 and abs(float(2 / s ** 2 * ds ** 2) - 0.15) < 0.01


# ---- host orchestration through the emulated C-ABI (tests/macpo_emulator.py) ----
@pytest.fixture()
def emulated(monkeypatch):
    import sys, os
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import macpo_emulator
    return macpo_emulator.install(monkeypatch)


@pytest.mark.parametrize("case", ["case0", "case1", "case3", "case4", "rejected"])
def test_macpo_trainer_host_against_oracle(golden, one_thread, emulated, case):
    from safepo.common.ma_model import MACPOTrainer, MultiAgentNets
    u = golden("macpo")["update"]
    c = next(x for x in u["cases"] if x["name"] == case)
    cfg = dict(u["cfg"], **c["cfg_overrides"])
    nets = MultiAgentNets(u["init"]["actor"], u["init"]["critic"], u["init"]["cost_critic"], "cpu", layer_N=cfg["layer_N"])
    tr = MACPOTrainer(nets, cfg)
    out = tr.trpo_update(c["sample"])
    assert out["optim_case"] == c["optim_case"] and out["accepted"] == c["accepted"]
    step = max(float((c["actor"][k] - u["init"]["actor"][k]).abs().max()) for k in c["actor"])
    for k, v in c["actor"].items():
        assert float((nets.actor.p[k] - v).abs().max()) <= 1e-3 * step + 1e-7, k
    for n in ("critic", "cost_critic"):
        for k, v in u["cases"][0]["critics"][n].items():
            torch.testing.assert_close(getattr(nets, n).p[k], v, rtol=1e-5, atol=1e-6)
    assert abs(out["kl"] - float(c["out"]["kl"])) <= 1e-4 * abs(float(c["out"]["kl"])) + 1e-9
    assert abs(out["expected_improve"] - float(c["out"]["expected_improve"])) <= 1e-4 * abs(float(c["out"]["expected_improve"])) + 1e-9
    assert abs(out["cost_loss"] - float(c["out"]["cost_loss"])) <= 1e-5


def test_macpo_fvp_host_against_oracle(golden, one_thread, emulated):
    from safepo.common.ma_model import MACPOTrainer, MultiAgentNets
    u = golden("macpo")["update"]
    nets = MultiAgentNets(u["init"]["actor"], u["init"]["critic"], u["init"]["cost_critic"], "cpu", layer_N=u["cfg"]["layer_N"])
    tr = MACPOTrainer(nets, u["cfg"])
    v = torch.zeros(tr._count)
    i = 0
    for t in tr._tangents(v).values():
        t.copy_(u["fvp"]["p"][i:i + t.numel()].view(t.shape))
        i += t.numel()
    out = torch.zeros_like(v)
    tr.fvp(u["cases"][0]["sample"]["obs"].contiguous(), v, out)
    got = torch.cat([t.reshape(-1) for t in tr._tangents(out).values()])
    assert float((got - u["fvp"]["out"]).abs().max() / u["fvp"]["out"].abs().max()) < 1e-5


def test_macpo_runner_host_against_oracle(one_thread, emulated):
    from safepo.multi_agent import macpo
    T, N, D, DS, A, H, NA, layer_N = 4, 6, 10, 14, 3, 32, 2, 2
    cfg = dict(macpo.DEFAULT_CONFIG, episode_length=T, n_rollout_threads=N, hidden_size=H)
    g = torch.Generator().manual_seed(3)
    all_states = []
    for a in range(NA):
        st = [macpo.init_state(D, H, layer_N, "actor", A, generator=g), macpo.init_state(DS, H, layer_N, "critic", generator=g),
              macpo.init_state(DS, H, layer_N, "critic", generator=g)]
        all_states.append([{k: v + 0.1 * torch.randn(v.shape, generator=g) for k, v in s.items()} for s in st])
    onets = [tuple(MA.OracleMANet(s, layer_N=layer_N) for s in states) for states in all_states]
    orun = MO.OracleMACPORunner(onets, cfg, T, N, D, DS, A)
    drun = macpo.Runner([macpo.MultiAgentNets(*states, "cpu", layer_N=layer_N) for states in all_states], cfg, D, DS, A)
    obs0, share0 = torch.randn(N, NA, D, generator=g), torch.randn(N, NA, DS, generator=g)
    orun.warmup(obs0, share0)
    drun.warmup(obs0, share0)
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
    perms = [torch.randperm(T * N, generator=g) for _ in range(NA)]
    outs = orun.train(agent_order=[1, 0], perms=perms)
    douts = drun.train(agent_order=[1, 0], perms=[[p] for p in perms], collect_outputs=True)
    for a in range(NA):
        assert douts[a]["optim_case"] == outs[a]["optim_case"] and douts[a]["accepted"] == outs[a]["accepted"]
        for dn, on in zip((drun.nets[a].actor, drun.nets[a].critic, drun.nets[a].cost_critic), onets[a]):
            for k, v in on.p.items():
                torch.testing.assert_close(dn.p[k], v.detach(), rtol=1e-4, atol=1e-5)
    row = drun._agent_log(0, douts[0])
    assert {"Loss/Loss_actor_improve/agent0", "Loss/Loss_actor_expected_improve/agent0", "Misc/KL/agent0"} <= set(row)
