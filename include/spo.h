/*
 * libspo -- C-ABI of the B200-native SafePO hot path (rollout forward -> dual GAE ->
 * policy / critic update).  Plain pointers and sizes only; every pointer marked
 * "device" is a CUDA device pointer owned by the caller (PyTorch tensors in the shipped
 * host code); the library never allocates, frees or retains memory past a call.
 *
 * Each entry point names the reference code it replaces (paths relative to the
 * PKU-Alignment/Safe-Policy-Optimization checkout).
 *
 * Conventions
 *   - return value: 0 (SPO_OK) or a negative spo_status; message via spo_last_error()
 *     (thread-local).  Nothing aborts or throws across the boundary.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All
 *     work is asynchronous on that stream; asynchronous CUDA errors surface at the next
 *     call or at spo_sync_check().
 *   - there is no CPU fallback: unsupported dimensions return SPO_ERR_UNSUPPORTED.
 *
 * Packed parameter layout (fp32, one buffer of spo_param_count() floats):
 *     actor         : log_std[A] W1[H*D] b1[H] W2[H*H] b2[H] W3[A*H] b3[A]
 *     reward critic : W1[H*D] b1[H] W2[H*H] b2[H] W3[H] b3[1]
 *     cost critic   : (same)
 *   matrices are row-major [out][in] exactly as torch.nn.Linear stores them, so the actor
 *   slice is the flat vector of get_flat_params_from(policy.actor)
 *   (safepo/single_agent/cpo.py:70-78; log_std first) and nn.Parameter views into the
 *   buffer reproduce actor.state_dict() (safepo/common/model.py:73-76).
 *   Adam moments use the same layout; step counters are 3 int32 (actor, reward, cost).
 *
 * Rollout storage is env-major: element (env n, step t) of a per-step scalar lives at
 * n*T + t, rows of obs/act at (n*T + t)*D / *A -- the order buffer.get() produces
 * (safepo/common/buffer.py:149-153).
 */
#ifndef SPO_H_
#define SPO_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPO_VERSION 100

typedef enum spo_status {
  SPO_OK = 0,
  SPO_ERR_INVALID_ARG = -1,
  SPO_ERR_UNSUPPORTED = -2,
  SPO_ERR_CUDA = -3,
  SPO_ERR_NCCL = -4
} spo_status;

/* Network dimensions.  hidden must be 64 (two tanh layers of 64, the reference's
 * default_cfg for every MuJoCo task: ppo_lag.py:46, cpo.py:48, focops.py:48). */
typedef struct spo_dims {
  int obs_dim; /* D, 1..128 */
  int act_dim; /* A, 1..8   */
  int hidden;  /* H, 64     */
} spo_dims;

/* Env-major rollout arrays of one epoch, all device pointers (buffer.py:53-73). */
typedef struct spo_rollout {
  float *obs, *act;                  /* [N,T,D], [N,T,A] */
  float *reward, *cost;              /* [N,T] */
  float *value_r, *value_c, *logp;   /* [N,T] */
  uint8_t* seg_end;                  /* [N,T] 1 where a path closes (ppo_lag.py:200) */
  float *boot_r, *boot_c;            /* [N,T] bootstrap value of the path closing at t */
  int num_envs, steps;               /* N, T */
} spo_rollout;

int spo_version(void);
const char* spo_last_error(void);
int spo_sync_check(void* stream);

/* offsets (in floats) into the packed buffer; out arrays may be NULL.
 * net: 0 actor, 1 reward critic, 2 cost critic. */
int spo_param_count(const spo_dims* d, int* actor, int* critic, int* total);
int spo_param_offsets(const spo_dims* d, int net, int* log_std, int* w1, int* b1, int* w2, int* b2, int* w3, int* b3);

/* ---- F1/F2: ActorVCritic.step (safepo/common/model.py:149-170) fused with
 * VectorizedOnPolicyBuffer.store (safepo/common/buffer.py:84-95) ------------------------
 * obs [n,D] device.  eps [n,A] device or NULL (NULL: in-kernel Philox4x32-10 keyed by
 * (seed, offset), perf mode).  deterministic!=0: act = mean.  Outputs act [n,A], logp
 * [n], v_r [n], v_c [n] (device, any may be NULL).  If `store` is not NULL the kernel
 * also writes obs/act/logp/value_r/value_c of every env into slot t of the rollout
 * arrays (n must equal store->num_envs). */
int spo_policy_step(const spo_dims* d, const float* params, const float* obs, const float* eps,
                    uint64_t seed, uint64_t offset, int deterministic, int n,
                    float* act, float* logp, float* v_r, float* v_c,
                    const spo_rollout* store, int t, void* stream);

/* Reward/cost critic values only (the bootstrap forwards of ppo_lag.py:204-213). */
int spo_critic_values(const spo_dims* d, const float* params, const float* obs, int n,
                      float* v_r, float* v_c, void* stream);

/* Slot-t bookkeeping of the rollout loop (ppo_lag.py:187-234, SURVEY Appendix D):
 * writes reward/cost [n] into column t and derives seg_end/boot from the env flags:
 *   seg_end = epoch_end | terminated | truncated
 *   boot    = terminated ? 0 : truncated ? V(final_obs) : V(next_obs)
 * terminated/truncated: uint8 [n] device.  next_v_*: V(next_obs) [n] (used only when
 * epoch_end).  final_v_*: V(final_observation) [n] or NULL when no env truncated. */
int spo_store_transition(const spo_rollout* r, int t, const float* reward, const float* cost,
                         const uint8_t* terminated, const uint8_t* truncated, int epoch_end,
                         const float* next_v_r, const float* next_v_c,
                         const float* final_v_r, const float* final_v_c, void* stream);

/* ---- env I/O transforms around the forward (SURVEY 8f rank 1) ----
 * spo_obs_normalize: SafeNormalizeObservation (safepo/common/wrappers.py:42-49; gymnasium
 * NormalizeObservation + RunningMeanStd): with update != 0 folds the n rows into the running
 * statistics (mean/var: device float64 [obs_dim], updated in place; `count` is passed by value
 * and *count_out -- device, may be NULL -- receives count + n), then writes
 * out = (obs - mean) / sqrt(var + eps) as fp32 [n][obs_dim] (out may be NULL to update only, or
 * equal to obs for an in-place transform).
 * The caller owns the count bookkeeping (RunningMeanStd starts at mean 0, var 1, count 1e-4). */
int spo_obs_normalize(const float* obs, int n, int obs_dim, double* mean, double* var, double count,
                      double* count_out, int update, double eps, float* out, void* stream);

/* spo_action_rescale: SafeRescaleAction(env, min_action, max_action) (safepo/common/env.py:62,76;
 * gymnasium RescaleAction): clip to [min_action, max_action], map affinely onto [low, high]
 * (device fp32 [act_dim]), clip to [low, high].  act/out: device fp32 [n][act_dim]. */
int spo_action_rescale(const float* act, int n, int act_dim, const float* low, const float* high,
                       float min_action, float max_action, float* out, void* stream);

/* ---- G1: finish_path -> calculate_adv_and_value_targets -> discount_cumsum
 * (safepo/common/buffer.py:97-140,167-201) for every path of every env in one launch.
 * delta in fp32 ((r + gamma*v') - v, unfused), carry in fp64, outputs rounded to fp32.
 * disc_r = gamma*lam, disc_c = gamma*lam_c as doubles (buffer.py:199).
 * mode 0: warp-shuffle reverse affine scan (re-associates the fp64 carry);
 * mode 1: sequential recurrence per env, bit-exact with the reference. */
int spo_gae_dual(const float* reward, const float* cost, const float* value_r, const float* value_c,
                 const uint8_t* seg_end, const float* boot_r, const float* boot_c,
                 float gamma, double disc_r, double disc_c,
                 float* adv_r, float* adv_c, float* tgt_r, float* tgt_c,
                 int num_envs, int steps, int mode, void* stream);

/* ---- G2 (multi-agent path, config 5): SeparatedReplayBuffer.compute_returns / compute_cost_returns
 * (safepo/common/buffer.py:356-384): masked GAE on PopArt-de-normalised predictions, fp32 like the reference.
 * Time-major device arrays: rewards [T][N], value_preds [T+1][N] (row T = bootstrap), masks [T+1][N],
 * returns [T][N].  popart_mean / popart_sqrt_var: the de-biased running mean and sqrt(clamped variance) of the
 * value normaliser (popart.py:64-74); gamma_lambda = gamma * gae_lambda as the double product python forms.
 * (Round-1 status: compiled, first hardware run pending -- tests/test_zz_pending_gpu.py.) */
int spo_gae_masked(const float* rewards, const float* value_preds, const float* masks, float popart_mean,
                   float popart_sqrt_var, float gamma, double gamma_lambda, float* returns, int N, int T, void* stream);

/* ---- G3 + L1: buffer.get() statistics (buffer.py:154-160) and the Lagrange mix
 * (ppo_lag.py:280-281).  stats (device, 4 doubles) = {sum adv_r, sum adv_r^2, sum adv_c,
 * count}; spo_adv_stats overwrites them (all-reduce them across ranks before apply for
 * global statistics).  apply:
 *   a = (adv_r - mean) / (std_unbiased + 1e-8)   (if standardize_r)
 *   c = adv_c - mean_c                           (if standardize_c)
 *   mixed = (a - lam*c) / lam_plus_1
 * a/c overwrite adv_r/adv_c in place; mixed may be NULL. */
int spo_adv_stats(const float* adv_r, const float* adv_c, int64_t count, double* stats, void* stream);
int spo_adv_apply(float* adv_r, float* adv_c, int64_t count, const double* stats,
                  int standardize_r, int standardize_c, float lam, float lam_plus_1,
                  float* mixed, void* stream);

/* ---- U1/U3/C5: the minibatch update loop (ppo_lag.py:297-336, focops.py:309-357,
 * cpo.py:543-571) as ONE persistent launch per pass: for each of n_steps minibatches
 * gather `batch` rows by perm, forward+backward of the three nets, critic L2 term,
 * joint grad-norm clip, three Adam steps.  No host round trip inside. */
typedef enum spo_loss_kind {
  SPO_LOSS_PPO_CLIP = 0,   /* ppo_lag.py:315-319 */
  SPO_LOSS_FOCOPS = 1,     /* focops.py:323-337 ([B,1]x[B] broadcast semantics) */
  SPO_LOSS_CRITIC_ONLY = 2,/* cpo.py:543-571, trpo_lag.py:466-494 */
  SPO_LOSS_PG = 3,         /* pg.py:303-309: -(ratio * adv).mean(), the surrogate without the clip */
  SPO_LOSS_CUP_PROJECTION = 4 /* cup.py:355-404, second stage: ACTOR ONLY (critics untouched, clip norm over the actor),
                               * loss (c * ratio * adv [B] + KL(new||old) [B,1]).mean() with c passed in hp->focops_lam
                               * (c = lambda * (1 - gamma*0.95) / (1 - gamma)); needs old_mean/old_std, batch <= 64 */
} spo_loss_kind;

typedef struct spo_batch {
  const float *obs, *act, *logp;      /* [S,D], [S,A], [S] */
  const float *target_r, *target_c;   /* [S] */
  const float* adv;                   /* [S] mixed advantage (NULL for critic-only) */
  const float *old_mean, *old_std;    /* [S,A] each, FOCOPS only (focops.py:298-299) */
  int64_t count;                      /* S */
} spo_batch;

typedef struct spo_hparams {
  float lr_actor, lr_reward, lr_cost;
  float beta1, beta2, adam_eps;       /* 0.9, 0.999, 1e-8 */
  float max_grad_norm;                /* 40.0, ppo_lag.py:325 */
  float critic_l2;                    /* 0.001, ppo_lag.py:310-314 (0 disables) */
  float clip_lo, clip_hi;             /* 0.8, 1.2 (ppo_lag.py:318) */
  float focops_lam, focops_kl;        /* 1.5 (focops.py:45), target_kl */
  float value_coef;                   /* 1.0 (2.0 with use_value_coefficient) */
} spo_hparams;

/* Device control block shared by the update and KL kernels (zero it per epoch). */
typedef struct spo_update_ctrl {
  double loss_sum[3];   /* sums over minibatches of loss_r, loss_c, loss_pi */
  double kl_sum;        /* scratch of the KL pass */
  long long steps;      /* minibatch steps taken */
  int stop;             /* set when kl > target_kl (ppo_lag.py:347-348) */
  int passes;           /* Train/StopIter */
  float final_kl;       /* Train/KL */
  unsigned int ticket;  /* internal */
  float extra_sumsq;    /* squared norm of stale .grad that joins the joint clip (cpo.py:562) */
  int pad_;
} spo_update_ctrl;

/* perm: int64 device, n_steps*batch indices (the last step may be short: total =
 * perm_len).  adam_m/adam_v: packed like params.  adam_t: 3 int32 device step counters.
 * If ctrl->stop is already set the launch returns without touching anything. */
int spo_pg_update(const spo_dims* d, float* params, float* adam_m, float* adam_v, int* adam_t,
                  const spo_batch* data, const int64_t* perm, int64_t perm_len, int batch,
                  spo_loss_kind kind, const spo_hparams* hp, spo_update_ctrl* ctrl, void* stream);

/* ---- data-parallel variant (SURVEY section 8e): ranks own disjoint env shards and hold
 * identical replicas of the weights; every minibatch step each net's gradient is summed
 * over the ranks INSIDE the persistent kernel through peer-mapped memory over
 * NVLink/NVSwitch (no NCCL call, no extra launch): a CTA pushes its slice of the gradient into
 * peer-mapped staging memory of every peer as 8-byte {value, sequence} words (posted remote stores) and polls the
 * words it is owed -- no fence, no flag, no barrier; sums run in rank order, so all ranks obtain bit-identical
 * results and the replicas never diverge.  The result is scaled by 1/world (global minibatch = world * batch).
 *   grad_bufs[r] : rank r's staging memory, 2 * world * 3 * slot floats (slot from spo_comm_slot_floats):
 *                  [parity][source rank][net][slot] 8-byte {value, sequence} words
 *   flags[r]     : unused since round 2 (the sequence number inside every word is the flag); may be NULL
 *   seq_base     : number of minibatch steps all ranks have completed in earlier launches
 * Both pointer tables live in DEVICE memory (world entries each). */
typedef struct spo_comm {
  int world, rank;
  float* const* grad_bufs;
  unsigned int* const* flags;
  unsigned long long seq_base;
  unsigned int spin_limit;   /* 0 = default (~2e8 polls) before the kernel gives up and sets ctrl->stop = 2 */
} spo_comm;

int spo_comm_slot_floats(const spo_dims* d, int* slot_floats);
int spo_pg_update_dp(const spo_dims* d, float* params, float* adam_m, float* adam_v, int* adam_t,
                     const spo_batch* data, const int64_t* perm, int64_t perm_len, int batch,
                     spo_loss_kind kind, const spo_hparams* hp, spo_update_ctrl* ctrl,
                     const spo_comm* comm, void* stream);
/* Peer mapping helpers (CUDA IPC): the staging buffers must be plain cudaMalloc memory, so
 * these are the only entry points that allocate.  handle is 64 bytes. */
int spo_comm_alloc(size_t bytes, void** ptr);
int spo_comm_free(void* ptr);
int spo_comm_export(void* ptr, unsigned char* handle64);
int spo_comm_import(const unsigned char* handle64, void** ptr);
int spo_comm_close(void* imported_ptr);
/* KL early-stop test split in two for multi-GPU: accumulate the local sum into
 * ctrl->kl_sum, (all-reduce that double across ranks), then finalize with the global count. */
int spo_actor_kl_accumulate(const spo_dims* d, const float* params, const float* obs, const float* old_mean,
                            const float* old_log_std, int64_t count, spo_update_ctrl* ctrl, void* stream);
int spo_kl_finalize(spo_update_ctrl* ctrl, double denom, float target_kl, void* stream);

/* ---- U2: full-batch actor passes -------------------------------------------------------
 * spo_actor_forward: mean [S,A] of policy.actor(obs) (old_distribution, ppo_lag.py:277).
 * spo_actor_kl: KL(N(old_mean, exp(old_log_std)) || N(mean(obs), exp(log_std))) with
 *   reduce 0: .sum(-1).mean() (ppo_lag.py:338-344)   reduce 1: .mean() over S*A (cpo.py:489-491)
 *   result -> ctrl->final_kl, ctrl->passes += 1, ctrl->stop |= (kl > target_kl).
 *   Skipped (no-op) when ctrl->stop is already set. */
int spo_actor_forward(const spo_dims* d, const float* params, const float* obs, int64_t count,
                      float* mean_out, void* stream);
int spo_actor_kl(const spo_dims* d, const float* params, const float* obs, const float* old_mean,
                 const float* old_log_std, int64_t count, int reduce, float target_kl,
                 spo_update_ctrl* ctrl, void* stream);

/* ---- C1-C4: trust-region pieces (cpo.py:70-157,353-519; trpo_lag.py:363-442) -----------
 * All vectors are actor-flat [P_a] device fp32 (log_std first).
 * spo_surrogate_grad: loss = mean(ratio*adv) (cpo.py:356-359) and d loss / d theta.
 *   out_loss: device float.  grad may be NULL (loss only).
 * spo_fvp: (H + damping I) v with H the Hessian of mean_{S*A} KL(old||new) at new=old
 *   (cpo.py:132-157), evaluated in closed form (one JVP + one VJP through the mean MLP).
 * spo_linesearch_eval: with theta = params actor slice (already set to the trial
 *   point) writes out[0]=mean(ratio*adv_a), out[1]=mean(ratio*adv_b) (adv_b may be NULL),
 *   out[2]=mean_{S*A} KL(old||new)  (cpo.py:475-491). */
int spo_surrogate_grad(const spo_dims* d, const float* params, const float* obs, const float* act,
                       const float* logp_old, const float* adv, int64_t count,
                       float* out_loss, float* grad, void* stream);
int spo_fvp(const spo_dims* d, const float* params, const float* obs, int64_t count,
            const float* v, float damping, float* out, void* stream);
int spo_linesearch_eval(const spo_dims* d, const float* params, const float* obs, const float* act,
                        const float* logp_old, const float* adv_a, const float* adv_b,
                        const float* old_mean, const float* old_log_std, int64_t count,
                        float* out3, void* stream);
/* Conjugate gradient (cpo.py:81-106) fully on device: 1 + iters FVPs, all dots/axpys and
 * the residual_tol break evaluated on device (no host sync).  work: 4*P_a floats + 8. */
int spo_conjugate_gradient(const spo_dims* d, const float* params, const float* obs, int64_t count,
                           const float* b, int iters, float damping, float residual_tol, float eps,
                           float* x, float* work, void* stream);

/* The solver above split at the Fisher-vector product, for data-parallel ranks (SURVEY section 8e, exchange 3'): every
 * FVP result is averaged over the ranks before the step that consumes it.  Same work layout (r | p | z | - | scalars):
 *   spo_cg_begin(b, x, work);
 *   repeat iters times: spo_fvp(..., v = work + P_a, out = work + 2*P_a); all-reduce(mean) of work + 2*P_a; spo_cg_update(x, work, ...)
 * (cpo.py:81-106; the residual break stays a device flag). */
int spo_cg_begin(const spo_dims* d, const float* b, float* x, float* work, void* stream);
int spo_cg_update(const spo_dims* d, float* x, float* work, float residual_tol, float eps, void* stream);

/* ---- multi-agent nets (MAPPO-Lag, BASELINE config 5; SURVEY section 8f rank 3), first slice: the forward ----
 * spo_ma_mlp_layer: one [Linear -> ELU -> LayerNorm] block of MLPLayer (safepo/utils/mlp.py:18-27), optionally preceded by
 *   the input LayerNorm of MLPBase (feature_norm, mlp.py:46-47,57-58): out[n][H] = LN_out(ELU(LN_in?(in)[n][K] W[H][K]^T + b)).
 *   K even, H a multiple of 128 up to 512; all pointers device fp32 (in / W 8-byte, out 16-byte aligned).
 * spo_ma_head: the output layer on the features, one warp per row.  log_std == NULL: plain Linear (v_out of
 *   MultiAgentCritic, model.py:330,361).  Otherwise the DiagGaussian head (distributions.py:38-42, act.py:37-43):
 *   std = sigmoid(log_std / std_x_coef) * std_y_coef, action = mean + std * eps (eps [n][O] device, NULL = the mode), and the
 *   per-dimension log-probabilities logp [n][O] (may be NULL). */
int spo_ma_mlp_layer(const float* in, int n, int K, const float* W, const float* b, const float* ln_w, const float* ln_b, int H,
                     const float* ln_in_w, const float* ln_in_b, float* out, void* stream);
int spo_ma_head(const float* feat, int n, int H, const float* W, const float* b, int O, const float* log_std, float std_x_coef,
                float std_y_coef, const float* eps, float* out, float* logp, void* stream);

/* ---- multi-agent nets, second slice: the UPDATE (MAPPO_L_Trainer.ppo_update, safepo/multi_agent/mappolag.py:135-199) ----
 * The host side (safepo/common/ma_model.py: MultiAgentTrainer) strings these together per net: training forward (activations
 * kept), loss head, then per layer LayerNorm/ELU backward, dW = dz^T x, dx = dz W, and clip + Adam on the packed parameters.
 * All pointers are device fp32; every sum over rows is a fixed-order two-stage reduction (per-CTA partials in `part`, then
 * spo_ma_partial_reduce), so results do not depend on scheduling.
 *
 * spo_ma_mlp_layer_train: spo_ma_mlp_layer that also keeps pre[n][H] = ELU(z) (the input of the output LayerNorm; 16-byte
 *   aligned) and, with the input LayerNorm, xn[n][K] = LN_in(in) (may be NULL otherwise).
 * spo_ma_ln_elu_bwd: dy[n][H] = d loss / d LN output -> dz[n][H] = d loss / d (x W^T + b) (mlp.py:18-27 backwards);
 *   part[ceil(n/32)][3][H] = per-CTA column sums {dy * xhat (d ln weight), dy (d ln bias), dz (d bias)}.
 * spo_ma_ln_in_bwd: parameter gradients of the input LayerNorm (mlp.py:46-47): part[ceil(n/32)][2][K] = {dxn * xhat, dxn}.
 * spo_ma_partial_reduce: out_s[j] = scale * sum_b part[b * stride + s * len + j], s < nseg <= 3 (out_s NULL = skipped).
 * spo_ma_gemm_nn: C[M][N] = A[M][Kd] B[Kd][N].   spo_ma_gemm_tn: part[z][M][N] = sum over the z-th slice of the R rows of
 *   A[r][M] B[r][N]  (follow with spo_ma_partial_reduce(part, slices, M*N, 1, M*N, C, ...)).
 * spo_ma_actor_loss: DiagGaussian head + clipped surrogate (mappolag.py:147-166, distributions.py:8-9,38-42): per-dimension
 *   log-probs of `actions` under mean = feat W^T + b, std = sigmoid(log_std / x) * y;  imp[n] = prod_j exp(logp_j - old_logp_j);
 *   loss_row = -factor * min(imp * adv, clamp(imp, clip_lo, clip_hi) * adv), adv = adv_targ - *lamda * cost_adv_targ (lamda: device
 *   scalar);  dmean[n][A] = d mean_rows(loss_row) / d mean;  part[ceil(n/32)][66] = {sum loss_row, 0, sum dmean_j (32), sum dstd_j (32)}.
 * spo_ma_actor_finalize: scalars[0] = policy_loss, scalars[1] = dist_entropy (act.py:57-60); g_b[A] = d / d bias of the mean layer,
 *   g_log_std[A] = d (policy_loss - entropy_coef * entropy) / d log_std.
 * spo_ma_value_loss: clipped one-sided-Huber value loss (mappolag.py:121-133, util.py:19-22) on v[n] against the two PopArt
 *   normalisations of the returns; dv[n] = scale * dL/dv (scale = value_loss_coef / n); part[ceil(n/256)][2] = {sum L_row, sum dv}.
 * spo_ma_popart_normalize: PopArt.forward on [n] values (popart.py:76-112): updates state = {running_mean, running_mean_sq,
 *   debiasing_term} with the batch moments (weight beta), then out = (x - mean) / sqrt(var).
 * spo_ma_lagrange_step: lamda <- relu(lamda - delta * rate), delta = -mean((mean(aver_costs) - cost_limit)(1 - gamma) + imp * cost_adv)
 *   (mappolag.py:169-172).
 * spo_ma_clip_adam: clip_grad_norm_(max_grad_norm) over the packed gradient + one torch.optim.Adam step (step >= 1 is the new
 *   step count); work[>= 1024] scratch, norm_out[0] = the gradient norm before clipping, norm_out[1] = the clip coefficient. */
int spo_ma_mlp_layer_train(const float* in, int n, int K, const float* W, const float* b, const float* ln_w, const float* ln_b, int H,
                           const float* ln_in_w, const float* ln_in_b, float* out, float* pre, float* xn, void* stream);
int spo_ma_ln_elu_bwd(const float* dy, const float* pre, const float* ln_w, int n, int H, float* dz, float* part, void* stream);
int spo_ma_ln_in_bwd(const float* dxn, const float* x, int n, int K, float* part, void* stream);
int spo_ma_partial_reduce(const float* part, int nblk, int stride, int nseg, int len, float* out0, float* out1, float* out2, float scale,
                          void* stream);
int spo_ma_gemm_nn(const float* A, const float* B, float* C, int M, int N, int Kd, void* stream);
int spo_ma_gemm_tn(const float* A, const float* B, float* part, int R, int M, int N, int slices, void* stream);
int spo_ma_actor_loss(const float* feat, int n, int H, const float* W, const float* b, const float* log_std, int A, const float* actions,
                      const float* old_logp, const float* adv, const float* cost_adv, const float* factor, const float* lamda,
                      float clip_lo, float clip_hi, float std_x_coef, float std_y_coef, float* dmean, float* imp, float* part, void* stream);
int spo_ma_actor_finalize(const float* part, int nblk, int n, const float* log_std, int A, float std_x_coef, float std_y_coef, float entropy_coef,
                          float* g_b, float* g_log_std, float* scalars, void* stream);
int spo_ma_value_loss(const float* v, const float* value_preds, const float* ret_norm_clipped, const float* ret_norm_orig, int n, float clip,
                      float huber_delta, float scale, float* dv, float* part, void* stream);
int spo_ma_popart_normalize(const float* x, int n, float* state, double beta, float epsilon, float* out, void* stream);
int spo_ma_lagrange_step(const float* imp, const float* cost_adv, const float* aver_episode_costs, int n, float cost_limit, double gamma,
                         float rate, float* lamda, void* stream);
int spo_ma_clip_adam(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int count, float max_grad_norm, double lr, double beta1,
                     double beta2, double eps, double weight_decay, int step, float* work, float* norm_out, void* stream);

/* ---- MACPO trust region on the multi-agent nets (safepo/multi_agent/macpo.py:153-380; csrc/spo_ma_trust.cu) ----
 * The Fisher-vector product of fisher_vector_product (macpo.py:187-198: double backprop of kl_divergence, :153-166) in closed form:
 * spo_ma_ln_in_jvp: tangent of the input LayerNorm, out[n][K] = dln_w xhat + dln_b (the observations carry no tangent).
 * spo_ma_gemm_nt_pair: C[M][N] = A1[M][K1] B1[N][K1]^T + A2[M][K2] B2[N][K2]^T (+ bias[N], may be NULL): the tangent
 *   z' = x' W^T + x W'^T + b' of a Linear layer (and mu' of the mean head).
 * spo_ma_ln_elu_jvp: in place on t[n][H]: z' -> y' through ELU (kept pre = ELU(z)) and LayerNorm (ln_w; tangents dln_w, dln_b).
 * spo_ma_fvp_head: dmean[n][A] = dmu * 2 / (1e-8 + 2 std^2) / n, part[ceil(n/32)][A] = per-CTA column sums (the mean bias).
 * spo_ma_fvp_finish: out = g + damping v on a packed buffer, except out[ls_off + j] = (h_j + damping) v[ls_off + j] with h the
 *   log_std block of the reference's KL, whose log term has the sign of KL(new || old)'s (macpo.py:163-164):
 *   h = f_ss s'^2 + f_s s'', f_s = -1/s - 4 s^3 / D^2, f_ss = 1/s^2 - 4 s^2 / D^2 + 32 s^4 / D^3, D = 1e-8 + 2 s^2.
 * Conjugate gradient (macpo.py:168-185) over `count` floats; state[4] = {rdotr, done, p.Ap, new rdotr}, part[256] scratch:
 *   spo_ma_cg_begin: x = 0, r = p = b, rdotr = b.b.  spo_ma_cg_update: alpha = rdotr / (p.Ap + 1e-8), x += alpha p,
 *   r -= alpha Ap, p = r + (r.r / rdotr) p; sets done once r.r < residual_tol, after which further updates are no-ops.
 * spo_ma_dot: out = x.y (fixed-order two-stage sum).  spo_ma_axpby: out = a x + b y (y may be NULL).
 * spo_ma_clip_norm: x *= max_norm / |x| when |x| > max_norm (macpo.py:343-345); nrm2 = x.x before.
 * spo_ma_linesearch_eval (macpo.py:349-368): on the features of the trial weights, scalars[5] = {-mean(imp factor adv),
 *   mean(imp factor cost_adv), mean_rows(sum_j kl_divergence), mean(imp), entropy}, imp = prod_j exp(logp_j - old_logp_j),
 *   old_mean[n][A] / old_std[A] of the weights before the step.  part[ceil(n/32)][4] scratch. */
int spo_ma_ln_in_jvp(const float* x, int n, int K, const float* dln_w, const float* dln_b, float* out, void* stream);
int spo_ma_gemm_nt_pair(const float* A1, const float* B1, int K1, const float* A2, const float* B2, int K2, const float* bias, float* C, int M, int N,
                    void* stream);
int spo_ma_ln_elu_jvp(float* t, const float* pre, const float* ln_w, const float* dln_w, const float* dln_b, int n, int H, void* stream);
int spo_ma_fvp_head(const float* dmu, int n, int A, const float* log_std, float std_x_coef, float std_y_coef, float* dmean, float* part,
                    void* stream);
int spo_ma_fvp_finish(const float* g, const float* v, int count, int ls_off, int A, const float* log_std, float std_x_coef, float std_y_coef,
                      float damping, float* out, void* stream);
int spo_ma_dot(const float* x, const float* y, int count, float* part, float* out, void* stream);
int spo_ma_cg_begin(const float* b, float* x, float* r, float* p, int count, float* state, float* part, void* stream);
int spo_ma_cg_update(float* p, const float* Ap, float* x, float* r, int count, float* state, float* part, float residual_tol, void* stream);
int spo_ma_axpby(float* out, float a, const float* x, float b, const float* y, int count, void* stream);
int spo_ma_clip_norm(float* x, int count, float max_norm, float* part, float* nrm2, void* stream);
int spo_ma_linesearch_eval(const float* feat, int n, int H, const float* W, const float* b, const float* log_std, int A, const float* actions,
                           const float* old_logp, const float* adv, const float* cost_adv, const float* factor, const float* old_mean,
                           const float* old_std, float std_x_coef, float std_y_coef, float* part, float* scalars, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPO_H_ */
