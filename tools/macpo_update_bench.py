"""Time the MACPO update on the device at config 5's per-agent shape (8192 rows = 8 steps x 1024 envs, obs 398 -> 512 x 3,
act 20): one Fisher-vector product and one whole trpo_update (critics, two surrogate gradients, 2 x 10 FVPs of CG, the line
search), with CUDA events.  Prints one JSON line with the card's name and power limit read in the same run.

    python tools/macpo_update_bench.py [--rows 8192] [--reps 20]

FLOP of one FVP from the shapes: the JVP and the VJP cost about two forwards each (a forward is 2 n (D H + 2 H H + H A)), so
~ 4 forwards."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "safe-policy-optimization_b200")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=8192)
    ap.add_argument("--obs-dim", type=int, default=398)
    ap.add_argument("--hidden", type=int, default=512)
    ap.add_argument("--act-dim", type=int, default=20)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    from safepo.common.ma_model import MACPOTrainer, MultiAgentNets
    from safepo.multi_agent.macpo import DEFAULT_CONFIG, init_state
    n, D, H, A = args.rows, args.obs_dim, args.hidden, args.act_dim
    g = torch.Generator().manual_seed(0)
    nets = MultiAgentNets(init_state(D, H, 2, "actor", A, generator=g), init_state(D, H, 2, "critic", generator=g),
                          init_state(D, H, 2, "critic", generator=g), "cuda")
    tr = MACPOTrainer(nets, DEFAULT_CONFIG)
    dev = "cuda"
    obs = torch.randn(n, D, device=dev)
    sample = dict(share_obs=torch.randn(n, D, device=dev), obs=obs, actions=torch.randn(n, A, device=dev) * 0.3,
                  value_preds=torch.randn(n, 1, device=dev), returns=torch.randn(n, 1, device=dev), old_action_log_probs=torch.zeros(n, A, device=dev),
                  adv_targ=torch.randn(n, 1, device=dev), factor=torch.ones(n, 1, device=dev), cost_preds=torch.randn(n, 1, device=dev),
                  cost_returns=torch.rand(n, 1, device=dev) * 30, cost_adv_targ=torch.randn(n, 1, device=dev),
                  aver_episode_costs=torch.full((n, 1), 20.0, device=dev))
    ws = tr._ws(n, nets.actor)
    tr._forward_train(nets.actor, obs, ws)
    v = torch.randn(tr._count, device=dev)
    out = torch.empty_like(v)
    for _ in range(3):
        tr.fvp(obs, v, out, ws)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.reps):
        tr.fvp(obs, v, out, ws)
    e1.record()
    torch.cuda.synchronize()
    fvp_ms = e0.elapsed_time(e1) / args.reps
    fwd = 2.0 * n * (D * H + 2 * H * H + H * A)
    fvp_flop = 4 * fwd
    for _ in range(2):
        tr.trpo_update(sample)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.reps // 4 or 1):
        tr.trpo_update(sample)
    e1.record()
    torch.cuda.synchronize()
    upd_ms = e0.elapsed_time(e1) / (args.reps // 4 or 1)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps(dict(card=q, rows=n, obs_dim=D, hidden=H, act_dim=A, fvp_ms=round(fvp_ms, 4), fvp_gflop=round(fvp_flop / 1e9, 2),
                          fvp_tflops=round(fvp_flop / fvp_ms / 1e9, 2), trpo_update_ms=round(upd_ms, 3))))


if __name__ == "__main__":
    main()
