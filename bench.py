#!/usr/bin/env python
"""Headline benchmark: env-steps/sec of PPO-Lag on SafetyPointGoal1-v0 shape
(obs 60, act 2), 1024 envs per GPU, 1000 steps per env per epoch (BASELINE.json
configs[1]), synthetic observations.

    python bench.py --gpus 1 --steps K --warmup W            # this repo (libspo kernels)
    python bench.py --impl reference --gpus 1 --steps K --warmup W   # the reference's CPU path (oracle port)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one epoch of the hot path: T=1000 fused forward/sample/store launches over
1024 envs, dual GAE + advantage statistics, then the PPO-Lag update (<= 40 passes of
16000 minibatch steps with the KL early stop of ppo_lag.py:347).  Two measurements:

  value : the environment stream is resident in HBM before the timed region starts
          (DeviceTapeRollout); CUDA events on the launching stream, barrier + synchronize
          on both sides, max over ranks.
  e2e   : the public trainer path with a HOST vector env: every env step copies that
          step's observations/rewards/costs/flags host->device from pinned memory and reads
          the actions back (bytes counted from the tensors copied).

Both arms run on ONE set of trainer objects (policy, optimizer state, buffer): the `value`
arm's W warm-up epochs warm every kernel of the `e2e` arm as well, which only swaps the rollout
front end (one extra warm-up epoch covers its copy path).  Each arm times exactly K epochs.

--dump-outputs DIR writes, after the timed epochs of the `value` arm, what its last epoch
handed back as DIR/<name>.npy (rank 0): the trained policy's parameters under their
state_dict names, the update's statistics, the Lagrange multiplier and a fixed, seeded
sample of rows of the epoch's batch.  The inputs depend on the arguments only, so two
builds run with the same arguments can be compared output for output.

Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement" for the roofline and
cpu_baseline definitions.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "safe-policy-optimization_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# BASELINE.json configs[1] (the headline; what the driver runs), configs[2] and configs[3] (per-GPU shard of the 4-GPU config)
WORKLOADS = {
    "ppo_lag": dict(algo="ppo_lag", task="SafetyPointGoal1-v0", D=60, A=2, envs=1024, batch=64,
                    metric="env-steps/sec PPO-Lag SafetyPointGoal1 @1024 envs/GPU",
                    text="BASELINE.json configs[1]: PPO-Lag SafetyPointGoal1-v0 shape (obs 60, act 2, hidden 64x64)",
                    update="batch 64, <=40 passes with KL early stop"),
    "cpo": dict(algo="cpo", task="SafetyCarButton1-v0", D=88, A=2, envs=1024, batch=128,
                metric="env-steps/sec CPO SafetyCarButton1 @1024 envs/GPU",
                text="BASELINE.json configs[2]: CPO SafetyCarButton1-v0 shape (obs 88, act 2, hidden 64x64)",
                update="2 x 15-iteration CG (33 FVPs over the full batch) + line search + 10 passes of batch-128 critic regression"),
    "focops": dict(algo="focops", task="SafetyAntVelocity-v1", D=27, A=8, envs=512, batch=64,
                   metric="env-steps/sec FOCOPS SafetyAntVelocity @512 envs/GPU",
                   text="BASELINE.json configs[3]: FOCOPS SafetyAntVelocity-v1 shape (obs 27, act 8, hidden 64x64), 2048 envs over 4 GPUs = 512 per GPU",
                   update="batch 64, <=40 passes with KL early stop, KL-projection loss"),
}
WL = WORKLOADS["ppo_lag"]
TASK, D_OBS, D_ACT = WL["task"], WL["D"], WL["A"]


def select_workload(name):
    global WL, TASK, D_OBS, D_ACT
    WL = WORKLOADS[name]
    TASK, D_OBS, D_ACT = WL["task"], WL["D"], WL["A"]


def bytes_per_sample_update():
    """SURVEY section 8(d): obs + act + logp/adv/targets gathered per sample per pass + the 8 B index."""
    return 4 * (D_OBS + D_ACT + 4) + 8


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=("spo", "reference"), default="spo")
    ap.add_argument("--config", choices=tuple(WORKLOADS), default="ppo_lag",
                    help="ppo_lag = BASELINE.json configs[1] (headline), cpo = configs[2], focops = configs[3] (per-GPU shard)")
    ap.add_argument("--num-envs", type=int, default=0, help="envs per GPU (0 = the workload's own)")
    ap.add_argument("--horizon", type=int, default=1000, help="steps per env per epoch (T)")
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--ref-horizon", type=int, default=0,
                    help="steps per env of the reference arm's measured mini-epoch (0 = sized from --cpu-seconds)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed epoch computed as DIR/<name>.npy (e.g. bench_outputs/)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------

def build_trainer(args, device, rank, resident, dp=None):
    """The public trainer objects of safepo.single_agent.<algo>, assembled once so that epochs can be timed individually."""
    import importlib
    from safepo import _lib as L
    from safepo.common.buffer import VectorizedOnPolicyBuffer
    from safepo.common.lagrange import Lagrange
    from safepo.common.logger import EpochLogger
    from safepo.common.model import ActorVCritic
    from safepo.common.synthetic_env import SyntheticVecEnv
    from safepo.single_agent._engine import (CriticRegression, DeviceTapeRollout, PolicyGradientUpdate, Rollout, TrustRegionUpdate,
                                             seed_all)
    from safepo.utils.config import single_agent_args

    algo = WL["algo"]
    mod = importlib.import_module(f"safepo.single_agent.{algo}")
    N, T = args.num_envs, args.horizon
    a, _ = single_agent_args(["--num-envs", str(N), "--steps-per-epoch", str(N * T), "--total-steps", str(N * T * 1000),
                              "--seed", str(rank), "--rng", "device", "--task", TASK])
    seed_all(rank)
    env = SyntheticVecEnv(N, D_OBS, D_ACT, episode_len=T, seed=rank)
    cfg = dict(mod.default_cfg)
    policy = ActorVCritic(D_OBS, D_ACT, cfg["hidden_sizes"]).to(device)
    buffer = VectorizedOnPolicyBuffer(env.observation_space, env.action_space, size=T, device=device, num_envs=N, gamma=cfg["gamma"])
    lagrange = None if algo == "cpo" else Lagrange(a.cost_limit, a.lagrangian_multiplier_init, a.lagrangian_multiplier_lr,
                                                   lagrangian_upper_bound=2.0 if algo == "focops" else None)
    log_dir = os.path.join(tempfile.mkdtemp(prefix="spo_bench_"), "exp", TASK, algo, f"rank{rank}")
    logger = EpochLogger(log_dir, seed=str(rank), verbose=False, use_tensorboard=False)
    roll = (DeviceTapeRollout if resident else Rollout)(env, policy, buffer, logger, a, device)
    tr = dict(env=env, policy=policy, buffer=buffer, lagrange=lagrange, logger=logger, roll=roll, T=T, N=N, dp=dp, device=device,
              algo=algo, args=a, cfg=cfg)
    if algo == "cpo":
        tr["trust"] = TrustRegionUpdate(policy, cfg, device, dp=dp)
        tr["critics"] = CriticRegression(policy, cfg, False, device, dp=dp)
    else:
        kind = L.LOSS_FOCOPS if algo == "focops" else L.LOSS_PPO_CLIP
        tr["upd"] = PolicyGradientUpdate(policy, cfg, kind, epochs=1000, host_rng=False, device=device, dp=dp)
    return tr


def one_epoch(tr):
    """Exactly the epoch body of run_policy_gradient / run_trust_region (the algorithms' main())."""
    tr["roll"].run(tr["T"])
    dp, lg = tr["dp"], tr["logger"]
    jc = lg.get_stats("Metrics/EpCost") if dp is None else dp.mean_episode_cost(lg, device=tr["device"])
    red = None if dp is None else dp.all_reduce_sum
    if tr["algo"] == "cpo":
        data = tr["buffer"].get(0.0, all_reduce=red)
        r = tr["trust"].run_cpo(data, jc - tr["args"].cost_limit)
        c = tr["critics"].run(data)
        res = {"stop_iter": int(r.get("Misc/AcceptanceStep", 0)), "steps": c["steps"]}
    else:
        tr["lagrange"].update_lagrange_multiplier(jc)
        data = tr["buffer"].get(tr["lagrange"].lagrangian_multiplier, all_reduce=red)
        res = tr["upd"].run(data)
    tr["buffer"].reset_segments()
    if not lg.logged:   # keep the logger's per-epoch state machine moving (A3)
        for k in ("Metrics/EpRet", "Metrics/EpCost", "Metrics/EpLen"):
            lg.log_tabular(k)
        lg.dump_tabular()
    return res


def timed_epochs(tr, K, W, world, device):
    import torch.distributed as dist
    from safepo import _lib as L
    for _ in range(W):
        one_epoch(tr)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = L.LAUNCHES["n"]
    h0, d0 = tr["roll"].bytes_h2d, tr["roll"].bytes_d2h
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stops, msteps = [], []
    with ClockSampler(device.index) as clk:
        flush = None
        if tr["N"] * tr["T"] * D_OBS * 4 < 126e6:      # inputs smaller than L2: evict them between timed epochs
            flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=device)
        e0.record()
        for _ in range(K):
            if flush is not None:
                flush.fill_(0.0)
            res = one_epoch(tr)
            stops.append(res["stop_iter"]); msteps.append(res["steps"])
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return dict(ms=ms, launches=L.LAUNCHES["n"] - l0, stops=stops, msteps=msteps, clocks=clk.summary(),
                h2d=(tr["roll"].bytes_h2d - h0) / K, d2h=(tr["roll"].bytes_d2h - d0) / K, last=res)


DUMP_ROWS = 65536   # batch rows dumped: 65536 x 4 (D + A + 11) bytes, 26 MB at the largest workload (cpo, D = 88)


def dump_outputs(tr, last, out_dir):
    """Write what the epoch just run handed back: the policy's parameters, the update's statistics, the Lagrange
    multiplier and the rows of a fixed, seeded sample of the epoch's batch (every field buffer.get() returned)."""
    S = tr["N"] * tr["T"]
    rows = np.sort(np.random.default_rng(0).choice(S, min(S, DUMP_ROWS), replace=False))
    idx = torch.as_tensor(rows, device=tr["device"])
    out = {f"policy.{k}": v for k, v in tr["policy"].state_dict().items()}
    for k, v in tr["buffer"].data.items():
        out[f"batch.{k}"] = v.reshape(S, *v.shape[2:])[idx]
    out["batch.adv"] = tr["buffer"].adv_mixed[idx]
    out["batch.row_index"] = rows.astype(np.float64)
    for k, v in last.items():
        out[f"update.{k}"] = np.float64(v)
    if tr["lagrange"] is not None:
        out["lagrange.multiplier"] = np.float64(tr["lagrange"].lagrangian_multiplier)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        a = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def time_dominant_kernel(tr, device):
    """Average duration of one launch of the workload's dominant kernel, CUDA events on the launching stream, 3 warm
    launches + 3 timed.  PPO-Lag / FOCOPS: spo_pg_update (one pass over the epoch's data).  CPO: spo_fvp over the full
    batch (the 33-per-epoch Fisher-vector product; SURVEY 8d: 98 560 FLOP and 4*D bytes per sample) plus, for the record,
    one critic-regression pass."""
    import ctypes as C
    from safepo import _lib as L
    pol = tr["policy"]
    data = tr["buffer"].get(0.0)
    S = data["obs"].shape[0]

    def timed(fn):
        times = []
        for i in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if i >= 3:
                times.append(e0.elapsed_time(e1))
        return float(np.mean(times))

    out = {}
    if tr["algo"] == "cpo":
        trust, crit = tr["trust"], tr["critics"]
        v = torch.randn(pol.n_actor, device=device)
        trust._old_dist(data)
        ms = timed(lambda: trust._fvp(data, v, trust.Fx))
        flops = S * 5 * 2 * (D_OBS * 64 + 64 * 64 + 64 * D_ACT)
        out = {"kernel": "spo_fvp (Fisher-vector product over the full batch, fp32 FFMA tile GEMMs)", "ms": ms, "bound": "tensor",
               "achieved": flops / (ms / 1e3) / 1e12, "unit": "TFLOP/s", "units_per_launch": S}
        batch = L.Batch(L.ptr(data["obs"]), None, None, L.ptr(data["target_value_r"]), L.ptr(data["target_value_c"]), None, None, None, S)
        crit.ctrl.zero_()
        B = tr["cfg"]["batch_size"]

        def crit_pass():
            perm = torch.randperm(S, device=device)
            L.check(L.lib().spo_pg_update(C.byref(pol.dims), L.ptr(pol.flat), L.ptr(crit.adam.m), L.ptr(crit.adam.v), L.ptr(crit.adam.t),
                                          C.byref(batch), L.ptr(perm), S, B, L.LOSS_CRITIC_ONLY, C.byref(crit.hp), L.ptr(crit.ctrl),
                                          L.stream()), "spo_pg_update")
        ms_c = timed(crit_pass)
        out["critic_pass_ms"] = ms_c
        out["us_per_minibatch_step"] = ms_c * 1e3 / ((S + B - 1) // B)
    else:
        upd = tr["upd"]
        kind = L.LOSS_FOCOPS if tr["algo"] == "focops" else L.LOSS_PPO_CLIP
        old_mean = old_std = None
        if kind == L.LOSS_FOCOPS:
            old_mean = torch.zeros(S, D_ACT, device=device)
            old_std = torch.ones(S, D_ACT, device=device)
        batch = L.Batch(L.ptr(data["obs"]), L.ptr(data["act"]), L.ptr(data["log_prob"]), L.ptr(data["target_value_r"]),
                        L.ptr(data["target_value_c"]), L.ptr(data["adv"]), L.ptr(old_mean), L.ptr(old_std), S)
        upd.ctrl.zero_()

        def upd_pass():
            perm = torch.randperm(S, device=device)
            L.check(L.lib().spo_pg_update(C.byref(pol.dims), L.ptr(pol.flat), L.ptr(upd.adam.m), L.ptr(upd.adam.v), L.ptr(upd.adam.t),
                                          C.byref(batch), L.ptr(perm), S, 64, kind, C.byref(upd.hp), L.ptr(upd.ctrl), L.stream()),
                    "spo_pg_update")
        ms = timed(upd_pass)
        steps = (S + 63) // 64
        extra = 8 * D_ACT if kind == L.LOSS_FOCOPS else 0        # old_mean / old_std rows
        out = {"kernel": f"spo_update_kernel (one {tr['algo']} pass = {steps} serial minibatch steps)", "ms": ms, "bound": "hbm",
               "achieved": steps * 64 * (bytes_per_sample_update() + extra) / (ms / 1e3) / 1e9, "unit": "GB/s",
               "units_per_launch": steps, "us_per_minibatch_step": ms * 1e3 / steps}
    tr["buffer"].reset_segments()
    return out


def cpu_baseline(args, kind="port", threads=4, horizon=None):
    """The reference's CPU path (oracle port, bit-identical to the reference's main() -- tests/test_oracle_golden.py)
    timed on this box's host cores: ONE TRULY EXECUTED PPO-Lag epoch of oracle.trainers.train() -- rollout loop with
    store / bootstrap forwards / per-path GAE, buffer.get(), Lagrange step, <= 40 passes of batch-64 minibatch steps with
    the KL early stop -- at the workload's N envs and a reduced horizon T_s, plus 3 mid-epoch vector env steps to
    separate the per-step rollout cost from the once-per-epoch closing step.  The epoch is then scaled linearly to the
    workload's horizon T (every component is linear in T at fixed N; the closing step is counted once):
        epoch_s(T) = (T - 1) * t_step + t_close + t_update(T_s) * T / T_s."""
    from collections import deque
    from oracle import spo_oracle as O
    from oracle import trainers as TR
    from safepo.common.synthetic_env import SyntheticVecEnv
    N, T = args.num_envs, args.horizon
    per_T = 2.5 * (N / 1024.0) * (0.5 if WL["algo"] == "cpo" else 1.0)     # rough seconds of oracle update per unit of horizon
    Ts = horizon or max(1, min(16, int((args.cpu_seconds - 4.0) / per_T)))
    torch.set_num_threads(threads)
    # (a) per-step rollout cost away from the epoch end
    torch.manual_seed(0)
    env = SyntheticVecEnv(N, D_OBS, D_ACT, episode_len=T, seed=0)
    pol = O.OraclePolicy(D_OBS, D_ACT)
    r = 3
    buf = TR.PathBuffer(N, r, D_OBS, D_ACT, 0.99)
    obs, _ = env.reset()
    obs = torch.as_tensor(obs, dtype=torch.float32)
    ep = (np.zeros(N), np.zeros(N), np.zeros(N))
    dq = (deque(maxlen=50), deque(maxlen=50), deque(maxlen=50))
    t0 = time.time()
    TR.rollout(pol, env, buf, obs, ep, dq, TR.StatLog(), r, epoch_T=10 ** 9)
    t_step = (time.time() - t0) / r
    # (b) one real epoch at horizon Ts through the trainer
    env = SyntheticVecEnv(N, D_OBS, D_ACT, episode_len=T, seed=0)
    a = TR.default_args(num_envs=N, steps_per_epoch=N * Ts, total_steps=N * Ts * 1000, seed=0, torch_threads=threads, task=TASK)
    t1 = time.time()
    seen = {}
    _, log, times = TR.train(WL["algo"], a, env, max_epochs=1,
                             hooks={"after_update": lambda epoch, pol_, data_, extra: seen.update(extra)})
    t_epoch = time.time() - t1
    t_roll, t_upd = times["rollout"][0], times["update"][0]
    passes = int(seen.get("Train/StopIter", -1))
    t_close = max(t_roll - (Ts - 1) * t_step, 0.0)
    S_full, S_s = N * T, N * Ts
    epoch_s = (T - 1) * t_step + t_close + t_upd * T / Ts
    B = WL["batch"]
    if WL["algo"] == "cpo":
        passes = 10                                   # critic regression: learning_iters = 10 (cpo.py:52), no early stop
    mb = passes * ((S_s + B - 1) // B) if passes > 0 else 0
    return {"value": S_full / epoch_s, "unit": "env-steps/s", "cores": threads, "kind": kind,
            "sample": (f"one executed {WL['algo']} epoch of the oracle port at {N} envs x {Ts} steps (S={S_s}: rollout {t_roll:.2f} s, "
                       f"update {t_upd:.2f} s incl. {passes} passes / {mb} minibatch steps of {B}, total {t_epoch:.2f} s) "
                       f"+ {r} mid-epoch vector steps ({t_step*1e3:.1f} ms each); scaled linearly to {T} steps/env"),
            "measured_epoch": {"horizon": Ts, "seconds": t_epoch, "env_steps_per_s": S_s / t_epoch, "passes": passes},
            "ms_per_minibatch_step": (t_upd / mb * 1e3) if (mb and WL["algo"] != "cpo") else None,
            "ms_per_vector_env_step": t_step * 1e3, "passes": passes}


def update_traffic_per_step():
    """dram__bytes_read.sum + dram__bytes_write.sum per minibatch step of the update kernel, from the committed
    `ncu --set full` capture (profiles/r02_update_traffic.json, written by tools/ncu_traffic.py); None if absent."""
    path = os.path.join(ROOT, "profiles", "r02_update_traffic.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        t = json.load(f)
    return float(t["dram_bytes_per_minibatch_step"]), t.get("source", "profiles/r02_update_traffic.json")


def run_spo(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl spo needs a CUDA device (there is no CPU fallback)")
    device = torch.device(f"cuda:{local}")
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    K, W = args.steps, max(args.warmup, 0)
    S = args.num_envs * args.horizon

    dp = None
    if world > 1:
        from safepo.common.dist import DataParallel
        dp = DataParallel()
    tr = build_trainer(args, device, rank, resident=True, dp=dp)
    val = timed_epochs(tr, K, W, world, device)
    if args.dump_outputs and rank == 0:
        dump_outputs(tr, val["last"], args.dump_outputs)      # before time_dominant_kernel trains the policy further
    dom = time_dominant_kernel(tr, device) if world == 1 else None
    e2e = None
    if not args.no_e2e:
        # same policy / optimizer / buffer objects, host-env rollout front end; one warm-up epoch for its copy path
        from safepo.common.synthetic_env import SyntheticVecEnv
        from safepo.single_agent._engine import Rollout
        tr2 = dict(tr)
        env2 = SyntheticVecEnv(args.num_envs, D_OBS, D_ACT, episode_len=args.horizon, seed=rank)
        tr2["env"] = env2
        tr2["roll"] = Rollout(env2, tr["policy"], tr["buffer"], tr["logger"], tr["roll"].args, device)
        e2e = timed_epochs(tr2, K, 1, world, device)
    if dp is not None:
        dp.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm, how = peaks()
    value = S * K * world / (val["ms"] / 1e3)
    passes = int(round(float(np.mean(val["stops"])))) or 1
    B = WL["batch"]
    if dom is None:   # per-launch timing is a single-GPU measurement; under torchrun derive the per-step figure from the epoch
        steps_per_pass = (S + B - 1) // B
        n_pass = 10 if WL["algo"] == "cpo" else max(passes, 1)
        ms = val["ms"] / K / n_pass
        dom = {"kernel": "spo_update_kernel (per-step figure derived from the epoch: all of the epoch attributed to the update passes)",
               "ms": ms, "bound": "hbm", "achieved": steps_per_pass * B * bytes_per_sample_update() / (ms / 1e3) / 1e9, "unit": "GB/s",
               "units_per_launch": steps_per_pass, "us_per_minibatch_step": ms * 1e3 / steps_per_pass}
    if dom["bound"] == "hbm":
        peak, peak_how = hbm, how
    else:
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peak, peak_how = float(json.load(f)["bf16_tflops"]), "measured dense bf16 (MEASURED_PEAKS.json); the kernel itself runs fp32 FFMA"
        except Exception:
            peak, peak_how = 1590.0, "fallback dense bf16 (B200_PROFILING.md); the kernel itself runs fp32 FFMA"
    traffic_step, traffic_src = update_traffic_per_step() if WL["algo"] == "ppo_lag" else (None, None)
    S_obs_mb = S * D_OBS * 4 / 1e6
    out = {
        "metric": WL["metric"], "value": value, "unit": "env-steps/s",
        "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": val["ms"] / K, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{WL['text']}, {args.num_envs} envs/GPU x {args.horizon} steps/epoch, {WL['update']}",
                   "samples_per_step_per_gpu": S, "stop_iter": val["stops"], "minibatch_steps_per_epoch": val["msteps"],
                   "us_per_minibatch_step": dom.get("us_per_minibatch_step"), "ms_per_dominant_launch": dom["ms"],
                   "l2": f"inputs larger than L2 ({S_obs_mb:.1f} MB observation buffer per epoch vs 126 MB L2)" if S_obs_mb > 126
                         else f"observation buffer {S_obs_mb:.1f} MB fits the 126 MB L2: a 256 MB scratch write flushes it between timed epochs",
                   "parallelism": (f"dp{world}: envs sharded, per-rank batch {B} (global batch {B * world}), in-kernel NVLink gradient sum per minibatch step"
                                   if world > 1 else "single")},
        "clocks": val["clocks"],
        "gpu_launches": val["launches"],
        "roofline": {"kernel": dom["kernel"], "bound": dom["bound"], "achieved": dom["achieved"], "peak": peak, "unit": dom["unit"],
                     "frac": dom["achieved"] / peak,
                     "traffic": (traffic_step * dom["units_per_launch"]) if traffic_step is not None else None, "traffic_source": traffic_src,
                     "peak_source": peak_how,
                     "note": ("serial-latency-bound chain of minibatch Adam steps (SURVEY H3): us_per_minibatch_step is the figure of merit"
                              if dom["bound"] == "hbm" else "fp32 FFMA tile GEMMs measured against the tensor roof the survey names for this kernel")},
    }
    if "critic_pass_ms" in dom:
        out["config"]["ms_per_critic_regression_pass"] = dom["critic_pass_ms"]
    if e2e is not None:
        out["e2e"] = {"value": S * K * world / (e2e["ms"] / 1e3), "unit": "env-steps/s", "h2d_bytes_per_step": e2e["h2d"],
                      "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": e2e["ms"] / K, "steps": K, "warmup": 1,
                      "stop_iter": e2e["stops"], "gpu_launches": e2e["launches"],
                      "note": "same trainer objects as the value arm (already warm); only the rollout front end differs"}
    if not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(args)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path (oracle port), all host threads
# ---------------------------------------------------------------------------------------

def pick_reference_threads():
    """The thread count the reference's path actually profits from on this host.  The reference pins
    torch.set_num_threads(4) (ppo_lag.py:73); its 64-row minibatch steps get slower, not faster, with more
    intra-op threads (128 threads on the GPU box: 1015 ms per minibatch step vs 2.3 ms with 4,
    profiles/r01_bench_reference_128threads.json).  A short probe of the dominant op picks the fastest of
    1..16 threads, so the arm is timed at the reference's best, not at an oversubscribed setting."""
    from oracle import spo_oracle as O
    torch.manual_seed(0)
    pol = O.OraclePolicy(D_OBS, D_ACT)
    opt = O.OracleOptim(pol)
    b = {"obs": torch.randn(64, D_OBS), "act": torch.randn(64, D_ACT), "log_prob": torch.full((64,), -2.5),
         "target_value_r": torch.randn(64), "target_value_c": torch.randn(64), "adv": torch.randn(64)}
    best, best_t = None, 1e9
    ncpu = os.cpu_count() or 4
    for t in (1, 2, 4, 8, 16):
        if t > ncpu:
            break
        torch.set_num_threads(t)
        for _ in range(5):
            O.minibatch_step(pol, opt, b, "ppo")
        t0 = time.time()
        n = 0
        while time.time() - t0 < 0.5:
            O.minibatch_step(pol, opt, b, "ppo")
            n += 1
        dt = (time.time() - t0) / n
        if dt < best_t:
            best, best_t = t, dt
    return best


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = pick_reference_threads()
    K, W = args.steps, max(args.warmup, 0)
    # every step = one executed mini-epoch of the oracle port (cpu_baseline); horizon sized so K+W of them end in minutes
    per = max(args.cpu_seconds * 6.0 / max(K + W, 1), 5.0)
    Ts = args.ref_horizon or max(1, min(16, int((per - 3.0) / 2.5)))
    vals = []
    for i in range(K + W):
        r = cpu_baseline(args, kind="port", threads=threads, horizon=Ts)
        if i >= W:
            vals.append(r)
    v = float(np.mean([r["value"] for r in vals]))
    S = args.num_envs * args.horizon
    out = {"impl": "reference", "metric": WL["metric"], "value": v, "unit": "env-steps/s",
           "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": S / v * 1e3, "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{WL['text']}, {args.num_envs} envs/GPU x {args.horizon} steps/epoch, {WL['update']}",
                      "sampling": f"each step executes one full epoch at {Ts} steps/env and scales it linearly to {args.horizon} (ms_per_step is the scaled epoch)",
                      "passes_observed": [r["passes"] for r in vals],
                      "measured_env_steps_per_s_at_reduced_horizon": float(np.mean([r["measured_epoch"]["env_steps_per_s"] for r in vals]))},
           "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": vals[-1]["sample"]},
           "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


if __name__ == "__main__":
    a = parse()
    select_workload(a.config)
    if a.num_envs <= 0:
        a.num_envs = WL["envs"]
    if a.impl == "reference":
        run_reference(a)
    else:
        run_spo(a)
