// Multi-agent trust-region pieces: the device side of MACPO_Trainer.trpo_update (safepo/multi_agent/macpo.py:200-380) on the
// MAPPO-Lag networks of spo_ma.cu / spo_ma_update.cu.
//
// The Fisher-vector product of the reference (macpo.py:187-198, double backprop of kl_divergence, :153-166) is computed in
// closed form as J^T M J v + the log_std block + 0.1 v:
//   * forward tangents (JVP) block by block: z' = x' W^T + x W'^T + b'  (ma_gemm_nt_pair_kernel, one tile product over both operand
//     pairs), then ELU' from the kept pre-activations and the LayerNorm tangent (ma_ln_elu_jvp_kernel); the input LayerNorm
//     contributes gamma_in' xhat_in + beta_in' (ma_ln_in_jvp_kernel), the observations carry no tangent;
//   * the head: mu' = f' W_m^T + f W_m'^T + b_m', dmean = mu' 2 / (1e-8 + 2 std^2) / n (ma_fvp_head_kernel); the vector-Jacobian
//     half is the existing backward chain of spo_ma_update.cu;
//   * the log_std block of the reference's "KL" (its log term has the sign of KL(new || old)'s): with D = 1e-8 + 2 s^2,
//     f_s = -1/s - 4 s^3 / D^2 and f_ss = 1/s^2 - 4 s^2 / D^2 + 32 s^4 / D^3 at coincidence, so h = f_ss s'^2 + f_s s''
//     (~ 4/s^2 s'^2 - 2/s s'', not the Gaussian Fisher's 2/s^2 s'^2) (ma_fvp_finish_kernel).
// Conjugate gradient over a vector of any length with the reference's eps placement and a device "done" flag (no host sync),
// and the line-search evaluation head (surrogates and the quirky KL against the kept old mean / std).  Every reduction is a
// two-stage sum in a fixed order.
#include <math.h>
#include "spo_common.cuh"
#include "spo_mma.cuh"

namespace {

constexpr int TR_ROWS = 32;        // rows per CTA of the row-wise kernels (as spo_ma_update.cu)
constexpr int TR_THREADS = 256;
constexpr int DOT_BLOCKS = 256;    // fixed grid of the vector reductions: the summation order depends only on the length
constexpr float kLogSqrt2Pi = 0.91893853320467274178f;

// ------------------------------------------------------------------------------------------------------------------
// C[M][N] = A1[M][K1] B1[N][K1]^T + A2[M][K2] B2[N][K2]^T (+ bias[N]): the tangent of a Linear layer.  mma.sync 3xTF32 tiles
// (spo_mma.cuh), 128 x 64 output tile, 32-deep chunks over the concatenated K, operands staged k-major as in spo_ma_update.cu.
// ------------------------------------------------------------------------------------------------------------------
constexpr int GTM = 128, GTN = 64, GK = 32;
constexpr int LDA_S = GTM + 8, LDB_S = GTN + 8;

struct NtPairArgs {
  const float *A1, *B1, *A2, *B2, *bias;
  float* C;
  int M, N, K1, K2;
};

__global__ void __launch_bounds__(256) ma_gemm_nt_pair_kernel(const NtPairArgs a) {
  __shared__ __align__(16) float As[GK * LDA_S];   // [k][m]
  __shared__ __align__(16) float Bs[GK * LDB_S];   // [k][n]
  const int tid = threadIdx.x, wid = tid >> 5;
  const int m0 = blockIdx.y * GTM, n0 = blockIdx.x * GTN;
  const int wm = (wid & 1) * 64, wn = (wid >> 1) * 16;
  float acc[4][2][4];
  spo_mma_zero<4>(acc);
  for (int pair = 0; pair < 2; ++pair) {
    const float* A = pair ? a.A2 : a.A1;
    const float* B = pair ? a.B2 : a.B1;
    const int K = pair ? a.K2 : a.K1;
    for (int k0 = 0; k0 < K; k0 += GK) {
      {   // A tile 128 x 32: thread -> row tid >> 1, sixteen consecutive k
        const int r = tid >> 1, kb = (tid & 1) * 16, gm = m0 + r;
        const float* src = A + static_cast<size_t>(gm) * K + k0 + kb;
#pragma unroll
        for (int e = 0; e < 16; ++e) As[(kb + e) * LDA_S + r] = (gm < a.M && k0 + kb + e < K) ? src[e] : 0.f;
      }
      {   // B tile 64 x 32 (rows of B = output columns): thread -> row tid >> 2, eight consecutive k
        const int r = tid >> 2, kb = (tid & 3) * 8, gn = n0 + r;
        const float* src = B + static_cast<size_t>(gn) * K + k0 + kb;
#pragma unroll
        for (int e = 0; e < 8; ++e) Bs[(kb + e) * LDB_S + r] = (gn < a.N && k0 + kb + e < K) ? src[e] : 0.f;
      }
      __syncthreads();
      spo_warp_mma_3xtf32<4>(acc, As, 1, LDA_S, Bs, LDB_S, 1, wm, wn, GK);
      __syncthreads();
    }
  }
  const int lane = tid & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int gm = m0 + wm + 16 * mt + g + ((e >> 1) << 3), gn = n0 + wn + 8 * nt + 2 * t + (e & 1);
        if (gm < a.M && gn < a.N) a.C[static_cast<size_t>(gm) * a.N + gn] = acc[mt][nt][e] + (a.bias ? a.bias[gn] : 0.f);
      }
}

// ------------------------------------------------------------------------------------------------------------------
// Tangent of ELU then LayerNorm (mlp.py:18-27), in place on t[n][H] (= z' on entry, y' on exit); pre = ELU(z) kept by the
// training forward.  p' = z' (pre > 0 ? 1 : pre + 1);  y' = gamma rstd (p' - mean(p') - xhat mean(p' xhat)) + gamma' xhat + beta'
// One warp per row, row statistics as in the forward / ma_ln_elu_bwd_kernel (lane l owns columns 128 cb + 4 l .. + 3).
// ------------------------------------------------------------------------------------------------------------------
struct LnEluJvpArgs {
  float* t;
  const float *pre, *ln_w, *dln_w, *dln_b;
  int n;
};

template <int HB>
__global__ void __launch_bounds__(TR_THREADS) ma_ln_elu_jvp_kernel(const LnEluJvpArgs a) {
  constexpr int H = 128 * HB;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float gam[4 * HB], dgam[4 * HB], dbet[4 * HB];
#pragma unroll
  for (int cb = 0; cb < HB; ++cb) {
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(a.ln_w + 128 * cb + 4 * lane));
    const float4 dg4 = __ldg(reinterpret_cast<const float4*>(a.dln_w + 128 * cb + 4 * lane));
    const float4 db4 = __ldg(reinterpret_cast<const float4*>(a.dln_b + 128 * cb + 4 * lane));
    gam[4 * cb] = g4.x; gam[4 * cb + 1] = g4.y; gam[4 * cb + 2] = g4.z; gam[4 * cb + 3] = g4.w;
    dgam[4 * cb] = dg4.x; dgam[4 * cb + 1] = dg4.y; dgam[4 * cb + 2] = dg4.z; dgam[4 * cb + 3] = dg4.w;
    dbet[4 * cb] = db4.x; dbet[4 * cb + 1] = db4.y; dbet[4 * cb + 2] = db4.z; dbet[4 * cb + 3] = db4.w;
  }
  for (int r = 0; r < 4; ++r) {
    const int g = blockIdx.x * TR_ROWS + 4 * wid + r;
    if (g >= a.n) break;                                   // warp-uniform
    float e[4 * HB], d[4 * HB];
    float s = 0.f;
#pragma unroll
    for (int cb = 0; cb < HB; ++cb) {
      const float4 e4 = *reinterpret_cast<const float4*>(a.pre + static_cast<size_t>(g) * H + 128 * cb + 4 * lane);
      const float4 d4 = *reinterpret_cast<const float4*>(a.t + static_cast<size_t>(g) * H + 128 * cb + 4 * lane);
      e[4 * cb] = e4.x; e[4 * cb + 1] = e4.y; e[4 * cb + 2] = e4.z; e[4 * cb + 3] = e4.w;
      d[4 * cb] = d4.x; d[4 * cb + 1] = d4.y; d[4 * cb + 2] = d4.z; d[4 * cb + 3] = d4.w;
      s += (e4.x + e4.y) + (e4.z + e4.w);
    }
    s = spo_warp_sum(s);
    const float mean = s / static_cast<float>(H);
    float q = 0.f;
#pragma unroll
    for (int c = 0; c < 4 * HB; ++c) { const float u = e[c] - mean; q = fmaf(u, u, q); }
    q = spo_warp_sum(q);
    const float rstd = rsqrtf(q / static_cast<float>(H) + 1e-5f);
    float xh[4 * HB];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int c = 0; c < 4 * HB; ++c) {
      xh[c] = (e[c] - mean) * rstd;
      d[c] *= (e[c] > 0.f ? 1.f : e[c] + 1.f);            // ELU'(z) = ELU(z) + 1 for z <= 0
      s1 += d[c];
      s2 = fmaf(d[c], xh[c], s2);
    }
    s1 = spo_warp_sum(s1) / static_cast<float>(H);
    s2 = spo_warp_sum(s2) / static_cast<float>(H);
    float o[4 * HB];
#pragma unroll
    for (int c = 0; c < 4 * HB; ++c) o[c] = fmaf(gam[c] * rstd, d[c] - s1 - xh[c] * s2, fmaf(dgam[c], xh[c], dbet[c]));
#pragma unroll
    for (int cb = 0; cb < HB; ++cb)
      *reinterpret_cast<float4*>(a.t + static_cast<size_t>(g) * H + 128 * cb + 4 * lane) = make_float4(o[4 * cb], o[4 * cb + 1], o[4 * cb + 2], o[4 * cb + 3]);
  }
}

// tangent of the input LayerNorm's output (mlp.py:46-47) for observations without tangent: out = gamma' xhat + beta'
struct LnInJvpArgs {
  const float *x, *dln_w, *dln_b;
  float* out;
  int n, K;
};

__global__ void __launch_bounds__(TR_THREADS) ma_ln_in_jvp_kernel(const LnInJvpArgs a) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, K = a.K;
  for (int r = 0; r < 4; ++r) {
    const int g = blockIdx.x * TR_ROWS + 4 * wid + r;
    if (g >= a.n) break;
    const float* x = a.x + static_cast<size_t>(g) * K;
    float s = 0.f;
    for (int k = lane; k < K; k += 32) s += x[k];
    s = spo_warp_sum(s);
    const float mean = s / static_cast<float>(K);
    float v = 0.f;
    for (int k = lane; k < K; k += 32) { const float d = x[k] - mean; v = fmaf(d, d, v); }
    v = spo_warp_sum(v);
    const float rstd = rsqrtf(v / static_cast<float>(K) + 1e-5f);
    for (int k = lane; k < K; k += 32) a.out[static_cast<size_t>(g) * K + k] = fmaf(a.dln_w[k], (x[k] - mean) * rstd, a.dln_b[k]);
  }
}

__device__ __forceinline__ float std_of(float log_std, float x_coef, float y_coef) {
  return __fmul_rn(__fdiv_rn(1.f, 1.f + expf(-__fdiv_rn(log_std, x_coef))), y_coef);     // as spo_ma_head_kernel
}

// ------------------------------------------------------------------------------------------------------------------
// FVP head: dmean[n][A] = dmu * 2 / (1e-8 + 2 std^2) / n;  part[blk][j] = sum over the CTA's 32 rows of dmean[.][j] (bias block)
// ------------------------------------------------------------------------------------------------------------------
struct FvpHeadArgs {
  const float *dmu, *log_std;
  float *dmean, *part;
  int n, A;
  float x_coef, y_coef;
};

__global__ void __launch_bounds__(TR_THREADS) ma_fvp_head_kernel(const FvpHeadArgs a) {
  const int j = threadIdx.x & 31, rw = threadIdx.x >> 5;
  __shared__ float red[TR_THREADS / 32][32];
  float acc = 0.f;
  if (j < a.A) {
    const float s = std_of(a.log_std[j], a.x_coef, a.y_coef);
    const float w = __fdiv_rn(__fdiv_rn(2.f, 1e-8f + 2.f * s * s), static_cast<float>(a.n));
    for (int r = rw; r < TR_ROWS; r += TR_THREADS / 32) {
      const int g = blockIdx.x * TR_ROWS + r;
      if (g >= a.n) break;
      const float d = a.dmu[static_cast<size_t>(g) * a.A + j] * w;
      a.dmean[static_cast<size_t>(g) * a.A + j] = d;
      acc += d;
    }
  }
  red[rw][j] = acc;
  __syncthreads();
  if (threadIdx.x < a.A) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < TR_THREADS / 32; ++w) s += red[w][threadIdx.x];
    a.part[static_cast<size_t>(blockIdx.x) * a.A + threadIdx.x] = s;
  }
}

// out = g + damping v over the packed buffer; the log_std segment [ls_off, ls_off + A) gets h v + damping v instead
struct FvpFinishArgs {
  const float *g, *v, *log_std;
  float* out;
  int count, ls_off, A;
  float x_coef, y_coef, damping;
};

__global__ void __launch_bounds__(256) ma_fvp_finish_kernel(const FvpFinishArgs a) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= a.count) return;
  const float v = a.v[i];
  float g = a.g[i];
  const int j = i - a.ls_off;
  if (j >= 0 && j < a.A) {
    const float sg = __fdiv_rn(1.f, 1.f + expf(-__fdiv_rn(a.log_std[j], a.x_coef)));
    const float s = sg * a.y_coef;
    const float ds = a.y_coef * sg * (1.f - sg) / a.x_coef;
    const float dds = ds * (1.f - 2.f * sg) / a.x_coef;
    const float D = 1e-8f + 2.f * s * s;
    const float f_s = -1.f / s - 4.f * s * s * s / (D * D);
    const float f_ss = 1.f / (s * s) - 4.f * s * s / (D * D) + 32.f * s * s * s * s / (D * D * D);
    g = (f_ss * ds * ds + f_s * dds) * v;
  }
  a.out[i] = fmaf(a.damping, v, g);
}

// ------------------------------------------------------------------------------------------------------------------
// Vector reductions and the conjugate-gradient steps.  state = {rdotr, done, pAp, new_rdotr, scratch...}
// ------------------------------------------------------------------------------------------------------------------
enum { CG_RDOTR = 0, CG_DONE = 1, CG_PAP = 2, CG_NEW = 3 };

__global__ void __launch_bounds__(256) ma_dot_partial_kernel(const float* x, const float* y, int count, float* part) {
  __shared__ float red[8];
  float s = 0.f;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < count; i += DOT_BLOCKS * 256) s = fmaf(x[i], y[i], s);
  s = spo_warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
    part[blockIdx.x] = t;
  }
}

// out = sum of the DOT_BLOCKS partials in order; also_rdotr: state[CG_RDOTR] = out, state[CG_DONE] = 0 (CG begin)
__global__ void ma_dot_final_kernel(const float* part, float* out, float* state_begin) {
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int b = 0; b < DOT_BLOCKS; ++b) t += part[b];
    *out = t;
    if (state_begin) { state_begin[CG_RDOTR] = t; state_begin[CG_DONE] = 0.f; }
  }
}

__global__ void __launch_bounds__(256) ma_copy2_kernel(const float* b, float* x, float* r, float* p, int count) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= count) return;
  const float v = b[i];
  x[i] = 0.f; r[i] = v; p[i] = v;
}

// x += alpha p; r -= alpha Ap with alpha = rdotr / (p.Ap + 1e-8) (macpo.py:176-178), skipped once the solve has converged
__global__ void __launch_bounds__(256) ma_cg_xr_kernel(const float* p, const float* Ap, float* x, float* r, int count, const float* st) {
  if (st[CG_DONE] != 0.f) return;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= count) return;
  const float alpha = st[CG_RDOTR] / (st[CG_PAP] + 1e-8f);
  x[i] = fmaf(alpha, p[i], x[i]);
  r[i] = fmaf(-alpha, Ap[i], r[i]);
}

// p = r + (new_rdotr / rdotr) p (macpo.py:180-181)
__global__ void __launch_bounds__(256) ma_cg_p_kernel(const float* r, float* p, int count, const float* st) {
  if (st[CG_DONE] != 0.f) return;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= count) return;
  const float beta = st[CG_NEW] / st[CG_RDOTR];
  p[i] = fmaf(beta, p[i], r[i]);
}

// rdotr = new_rdotr; the solve stops when rdotr < residual_tol (macpo.py:182-184)
__global__ void ma_cg_commit_kernel(float* st, float tol) {
  if (threadIdx.x == 0 && st[CG_DONE] == 0.f) {
    st[CG_RDOTR] = st[CG_NEW];
    if (st[CG_NEW] < tol) st[CG_DONE] = 1.f;
  }
}

// out = a x + b y  (y may be null)
__global__ void __launch_bounds__(256) ma_axpby_kernel(float* out, float a, const float* x, float b, const float* y, int count) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= count) return;
  out[i] = y ? fmaf(a, x[i], b * y[i]) : a * x[i];
}

// x *= max_norm / |x| when |x| > max_norm (macpo.py:343-345); nrm2 = x.x
__global__ void __launch_bounds__(256) ma_clip_norm_kernel(float* x, int count, const float* nrm2, float max_norm) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= count) return;
  const float nrm = sqrtf(*nrm2);
  if (nrm > max_norm) x[i] = x[i] * max_norm / nrm;
}

// ------------------------------------------------------------------------------------------------------------------
// Line-search head (macpo.py:349-368): mean on the trial weights, per-dimension log-probs, imp = prod_j exp(logp_j - old_logp_j),
//   part[blk] = { sum imp * factor * adv, sum imp * factor * cost_adv, sum kl_row, sum imp }
//   kl_row = sum_j log s_old - log s + (s_old^2 + (mu_old - mu)^2) / (1e-8 + 2 s^2) - 1/2     (the reference's kl_divergence)
// One warp per row (4 rows per warp, 32 per CTA); lane j < A owns action dimension j.
// ------------------------------------------------------------------------------------------------------------------
constexpr int LS_PART = 4;

struct LsArgs {
  const float *feat, *W, *b, *log_std, *actions, *old_logp, *adv, *cost_adv, *factor, *old_mean, *old_std;
  float* part;
  int n, H, A;
  float x_coef, y_coef;
};

__global__ void __launch_bounds__(TR_THREADS) ma_linesearch_kernel(const LsArgs a) {
  __shared__ float red[TR_THREADS / 32][LS_PART];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, A = a.A, H = a.H;
  float std = 1.f, bj = 0.f, so = 1.f;
  if (lane < A) {
    std = std_of(a.log_std[lane], a.x_coef, a.y_coef);
    bj = a.b[lane];
    so = a.old_std[lane];
  }
  const float log_s = logf(std), log_so = logf(so), den = 1e-8f + 2.f * std * std;
  float s_adv = 0.f, s_cadv = 0.f, s_kl = 0.f, s_imp = 0.f;
  for (int r = 0; r < 4; ++r) {
    const int g = blockIdx.x * TR_ROWS + 4 * wid + r;
    if (g >= a.n) break;                                   // warp-uniform
    const float* f = a.feat + static_cast<size_t>(g) * H;
    float mu = 0.f;
    for (int j = 0; j < A; ++j) {
      float s = 0.f;
      for (int k = lane; k < H; k += 32) s = fmaf(f[k], __ldg(a.W + j * H + k), s);
      s = spo_warp_sum(s);
      if (lane == j) mu = s + bj;
    }
    float ratio = 1.f, kl = 0.f;
    if (lane < A) {
      const size_t e = static_cast<size_t>(g) * A + lane;
      const float diff = __fsub_rn(a.actions[e], mu);
      const float q = __fdiv_rn(-__fmul_rn(diff, diff), __fmul_rn(2.f, __fmul_rn(std, std)));
      const float logp = __fsub_rn(__fsub_rn(q, log_s), kLogSqrt2Pi);
      ratio = expf(__fsub_rn(logp, a.old_logp[e]));
      const float dm = a.old_mean[e] - mu;
      kl = log_so - log_s + (so * so + dm * dm) / den - 0.5f;
    }
    float imp = ratio;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) imp *= __shfl_xor_sync(0xffffffffu, imp, m);
    kl = spo_warp_sum(kl);
    if (lane == 0) {
      const float w = imp * a.factor[g];
      s_adv += w * a.adv[g];
      s_cadv += w * a.cost_adv[g];
      s_kl += kl;
      s_imp += imp;
    }
  }
  if (lane == 0) { red[wid][0] = s_adv; red[wid][1] = s_cadv; red[wid][2] = s_kl; red[wid][3] = s_imp; }
  __syncthreads();
  if (threadIdx.x < LS_PART) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < TR_THREADS / 32; ++w) s += red[w][threadIdx.x];
    a.part[static_cast<size_t>(blockIdx.x) * LS_PART + threadIdx.x] = s;
  }
}

// scalars = { -mean(imp f adv), mean(imp f cost_adv), mean(kl_row), mean(imp), entropy }   (one CTA)
__global__ void ma_linesearch_final_kernel(const float* part, int nblk, int n, const float* log_std, int A, float x_coef, float y_coef,
                                           float* scalars) {
  if (threadIdx.x != 0) return;
  float t[LS_PART] = {0.f, 0.f, 0.f, 0.f};
  for (int b = 0; b < nblk; ++b)
    for (int k = 0; k < LS_PART; ++k) t[k] += part[static_cast<size_t>(b) * LS_PART + k];
  const float nf = static_cast<float>(n);
  scalars[0] = -(t[0] / nf);
  scalars[1] = t[1] / nf;
  scalars[2] = t[2] / nf;
  scalars[3] = t[3] / nf;
  float e = 0.f;
  for (int j = 0; j < A; ++j) e += 0.5f + kLogSqrt2Pi + logf(std_of(log_std[j], x_coef, y_coef));
  scalars[4] = e / static_cast<float>(A);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline int blocks256(int count) { return (count + 255) / 256; }

int dot_launch(const float* x, const float* y, int count, float* part, float* out, float* state_begin, cudaStream_t st) {
  ma_dot_partial_kernel<<<DOT_BLOCKS, 256, 0, st>>>(x, y, count, part);
  ma_dot_final_kernel<<<1, 32, 0, st>>>(part, out, state_begin);
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

}  // namespace

extern "C" {

int spo_ma_gemm_nt_pair(const float* A1, const float* B1, int K1, const float* A2, const float* B2, int K2, const float* bias, float* C, int M, int N,
                    void* stream) {
  SPO_REQUIRE(A1 && B1 && A2 && B2 && C && M > 0 && N > 0 && K1 > 0 && K2 > 0, SPO_ERR_INVALID_ARG, "spo_ma_gemm_nt_pair: null argument or empty shape");
  dim3 grid((N + GTN - 1) / GTN, (M + GTM - 1) / GTM, 1);
  SPO_REQUIRE(grid.y <= 65535, SPO_ERR_UNSUPPORTED, "spo_ma_gemm_nt_pair: M=%d too large", M);
  ma_gemm_nt_pair_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(NtPairArgs{A1, B1, A2, B2, bias, C, M, N, K1, K2});
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_ln_elu_jvp(float* t, const float* pre, const float* ln_w, const float* dln_w, const float* dln_b, int n, int H, void* stream) {
  SPO_REQUIRE(t && pre && ln_w && dln_w && dln_b && n > 0, SPO_ERR_INVALID_ARG, "spo_ma_ln_elu_jvp: null argument or n<=0");
  SPO_REQUIRE(H >= 128 && H <= 512 && (H & 127) == 0, SPO_ERR_UNSUPPORTED, "spo_ma_ln_elu_jvp: H=%d must be a multiple of 128 up to 512", H);
  SPO_REQUIRE(aligned16(t) && aligned16(pre) && aligned16(ln_w) && aligned16(dln_w) && aligned16(dln_b), SPO_ERR_INVALID_ARG,
              "spo_ma_ln_elu_jvp: 16-byte alignment required");
  LnEluJvpArgs a{t, pre, ln_w, dln_w, dln_b, n};
  const int grid = (n + TR_ROWS - 1) / TR_ROWS;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (H / 128) {
    case 1: ma_ln_elu_jvp_kernel<1><<<grid, TR_THREADS, 0, st>>>(a); break;
    case 2: ma_ln_elu_jvp_kernel<2><<<grid, TR_THREADS, 0, st>>>(a); break;
    case 3: ma_ln_elu_jvp_kernel<3><<<grid, TR_THREADS, 0, st>>>(a); break;
    default: ma_ln_elu_jvp_kernel<4><<<grid, TR_THREADS, 0, st>>>(a); break;
  }
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_ln_in_jvp(const float* x, int n, int K, const float* dln_w, const float* dln_b, float* out, void* stream) {
  SPO_REQUIRE(x && dln_w && dln_b && out && n > 0 && K > 0, SPO_ERR_INVALID_ARG, "spo_ma_ln_in_jvp: null argument or empty shape");
  ma_ln_in_jvp_kernel<<<(n + TR_ROWS - 1) / TR_ROWS, TR_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(LnInJvpArgs{x, dln_w, dln_b, out, n, K});
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_fvp_head(const float* dmu, int n, int A, const float* log_std, float std_x_coef, float std_y_coef, float* dmean, float* part,
                    void* stream) {
  SPO_REQUIRE(dmu && log_std && dmean && part && n > 0, SPO_ERR_INVALID_ARG, "spo_ma_fvp_head: null argument or n<=0");
  SPO_REQUIRE(A >= 1 && A <= 32, SPO_ERR_UNSUPPORTED, "spo_ma_fvp_head: act_dim=%d must be in 1..32", A);
  ma_fvp_head_kernel<<<(n + TR_ROWS - 1) / TR_ROWS, TR_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      FvpHeadArgs{dmu, log_std, dmean, part, n, A, std_x_coef, std_y_coef});
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_fvp_finish(const float* g, const float* v, int count, int ls_off, int A, const float* log_std, float std_x_coef, float std_y_coef,
                      float damping, float* out, void* stream) {
  SPO_REQUIRE(g && v && log_std && out && count > 0 && ls_off >= 0 && A >= 1 && ls_off + A <= count, SPO_ERR_INVALID_ARG,
              "spo_ma_fvp_finish: null argument or bad shape");
  ma_fvp_finish_kernel<<<blocks256(count), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      FvpFinishArgs{g, v, log_std, out, count, ls_off, A, std_x_coef, std_y_coef, damping});
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_dot(const float* x, const float* y, int count, float* part, float* out, void* stream) {
  SPO_REQUIRE(x && y && part && out && count > 0, SPO_ERR_INVALID_ARG, "spo_ma_dot: null argument or count<=0");
  return dot_launch(x, y, count, part, out, nullptr, static_cast<cudaStream_t>(stream));
}

int spo_ma_cg_begin(const float* b, float* x, float* r, float* p, int count, float* state, float* part, void* stream) {
  SPO_REQUIRE(b && x && r && p && state && part && count > 0, SPO_ERR_INVALID_ARG, "spo_ma_cg_begin: null argument or count<=0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  ma_copy2_kernel<<<blocks256(count), 256, 0, st>>>(b, x, r, p, count);
  return dot_launch(b, b, count, part, state + CG_RDOTR, state, st);
}

int spo_ma_cg_update(float* p, const float* Ap, float* x, float* r, int count, float* state, float* part, float residual_tol, void* stream) {
  SPO_REQUIRE(p && Ap && x && r && state && part && count > 0, SPO_ERR_INVALID_ARG, "spo_ma_cg_update: null argument or count<=0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = dot_launch(p, Ap, count, part, state + CG_PAP, nullptr, st);
  if (rc != SPO_OK) return rc;
  ma_cg_xr_kernel<<<blocks256(count), 256, 0, st>>>(p, Ap, x, r, count, state);
  rc = dot_launch(r, r, count, part, state + CG_NEW, nullptr, st);
  if (rc != SPO_OK) return rc;
  ma_cg_p_kernel<<<blocks256(count), 256, 0, st>>>(r, p, count, state);
  ma_cg_commit_kernel<<<1, 32, 0, st>>>(state, residual_tol);
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_axpby(float* out, float a, const float* x, float b, const float* y, int count, void* stream) {
  SPO_REQUIRE(out && x && count > 0, SPO_ERR_INVALID_ARG, "spo_ma_axpby: null argument or count<=0");
  ma_axpby_kernel<<<blocks256(count), 256, 0, static_cast<cudaStream_t>(stream)>>>(out, a, x, b, y, count);
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_clip_norm(float* x, int count, float max_norm, float* part, float* nrm2, void* stream) {
  SPO_REQUIRE(x && part && nrm2 && count > 0, SPO_ERR_INVALID_ARG, "spo_ma_clip_norm: null argument or count<=0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int rc = dot_launch(x, x, count, part, nrm2, nullptr, st);
  if (rc != SPO_OK) return rc;
  ma_clip_norm_kernel<<<blocks256(count), 256, 0, st>>>(x, count, nrm2, max_norm);
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

int spo_ma_linesearch_eval(const float* feat, int n, int H, const float* W, const float* b, const float* log_std, int A, const float* actions,
                           const float* old_logp, const float* adv, const float* cost_adv, const float* factor, const float* old_mean,
                           const float* old_std, float std_x_coef, float std_y_coef, float* part, float* scalars, void* stream) {
  SPO_REQUIRE(feat && W && b && log_std && actions && old_logp && adv && cost_adv && factor && old_mean && old_std && part && scalars && n > 0 && H > 0,
              SPO_ERR_INVALID_ARG, "spo_ma_linesearch_eval: null argument or empty shape");
  SPO_REQUIRE(A >= 1 && A <= 32, SPO_ERR_UNSUPPORTED, "spo_ma_linesearch_eval: act_dim=%d must be in 1..32", A);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nblk = (n + TR_ROWS - 1) / TR_ROWS;
  ma_linesearch_kernel<<<nblk, TR_THREADS, 0, st>>>(
      LsArgs{feat, W, b, log_std, actions, old_logp, adv, cost_adv, factor, old_mean, old_std, part, n, H, A, std_x_coef, std_y_coef});
  ma_linesearch_final_kernel<<<1, 32, 0, st>>>(part, nblk, n, log_std, A, std_x_coef, std_y_coef, scalars);
  SPO_CUDA_TRY(cudaGetLastError());
  return SPO_OK;
}

}  // extern "C"
