// K4 -- distribution heads: softmax / Categorical re-normalisation / inverse-CDF sampling /
// log-prob, and the Gaussian counterpart.
//
// Replaces  random_choice_prob_index / select_action   USTC_lab/server/utils.py:20-47
//           CategoricalActor._distribution + log_prob     nn/actor.py:90-101
//           GaussionActor._distribution + log_prob        nn/actor.py:58-70
//           sample / log_prob / play-mode lines           server/forward.py:137-144
// The random draw is an INPUT (uniforms / standard normals), so results are reproducible and
// the (probs, u) -> action map is bit-exact with the reference's numpy expression:
//     (p.cumsum(axis=1) > u[:,None]).argmax(axis=1)
// i.e. sequential fp32 prefix sum (__fadd_rn, never reassociated), strict '>', first hit,
// no hit => 0.  These kernels are tiny (<= 8A+16 B per row); one thread per row, except the Beta head's fp64 inverse-CDF
// solve, which runs one thread per (row, dimension).
// ACTION_MASK (categorical.cuh): the categorical head takes an optional mask [B, A]; the draw then inverts the CDF of the masked
// q, and no hit gives the first allowed action (0 without a mask, as above), so a masked action is never emitted.
// MultiDiscrete (categorical.cuh): the same head per branch, on the branch's slice, with draws u [B, K] and actions [B, K].
#include "common.cuh"
#include "beta.cuh"
#include "categorical.cuh"

namespace ddrl {

constexpr float kEps = 1.1920928955078125e-07f;   // torch.finfo(float32).eps
constexpr float kLogSqrt2Pi = 0.918938533204672741780329736406f;

// mask (categorical_row_mask) / j0 (categorical_first_allowed): only allowed actions are hits, and no hit gives j0
__device__ __forceinline__ int inverse_cdf(const float* __restrict__ p, int A, float u, const float* __restrict__ mask = nullptr,
                                           int j0 = 0) {
  float c = 0.f;
  for (int j = 0; j < A; ++j) {
    c = __fadd_rn(c, p[j]);
    if (c > u && categorical_allowed(mask, j)) return j;
  }
  return j0;  // numpy argmax of an all-False row (0 without a mask)
}

__device__ __forceinline__ int argmax_first(const float* __restrict__ p, int A, const float* __restrict__ mask = nullptr,
                                            int j0 = 0) {
  int best = j0;
  float bv = p[j0];
  for (int j = j0 + 1; j < A; ++j)
    if (categorical_allowed(mask, j) && p[j] > bv) { bv = p[j]; best = j; }
  return best;
}

__global__ void sample_probs_kernel(const float* __restrict__ probs, int ld, const float* __restrict__ u, int B, int A,
                                    float* __restrict__ action, float* __restrict__ logp) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float* p = probs + (size_t)b * ld;
  if (u) {
    const int a = inverse_cdf(p, A, u[b]);
    action[b] = (float)a;
    if (logp) logp[b] = logf(p[a]);            // server/utils.py:43
  } else {
    action[b] = (float)argmax_first(p, A);     // server/utils.py:45 / server/forward.py:143
    if (logp) logp[b] = 0.f;
  }
}

constexpr int kMaxA = kCatMaxA;

// logits -> softmax -> Categorical(probs): q = p / sum(p); logits' = log(clamp(q, eps, 1-eps)).  mask: [B, A] (row stride A) or
// null (categorical.cuh).  kBranched (MultiDiscrete): branch i samples its own slice with u[b, i] into action[b, i]; the row's
// log-prob is categorical_logp_row of the emitted actions.  Without it (the categorical actor) K = 1 and n_0 = A at compile time.
template <bool kBranched>
__global__ void categorical_head_kernel(const float* __restrict__ logits, int ld, const float* __restrict__ u, int B, int A,
                                        CatBranches br, float* __restrict__ action, float* __restrict__ logp,
                                        float* __restrict__ probs_out, const float* __restrict__ mask) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int K = kBranched ? br.K : 1;
  const float* x = logits + (size_t)b * ld;
  const float* mrow = mask ? mask + (size_t)b * A : nullptr;
  float q[kMaxA];
  for (int i = 0, o = 0; i < K; ++i) {
    const int n = kBranched ? br.n[i] : A;
    const float* mk = categorical_row_mask(mrow ? mrow + o : nullptr, n);
    const int j0 = categorical_first_allowed(mk, n);
    const float s2 = categorical_softmax(x + o, mk, n, j0, q + o);   // F.softmax (nn/actor.py:94)
    if (u) {
      for (int j = 0; j < n; ++j) q[o + j] = q[o + j] / s2;        // categorical.py:70
      const int a = inverse_cdf(q + o, n, u[(size_t)b * K + i], mk, j0);
      action[(size_t)b * K + i] = (float)a;
      if (!kBranched) logp[b] = logf(fminf(fmaxf(q[a], kEps), 1.f - kEps));
    } else {
      action[(size_t)b * K + i] = (float)argmax_first(q + o, n, mk, j0);   // play mode works on the raw softmax output
    }
    o += n;
  }
  if (probs_out) for (int j = 0; j < A; ++j) probs_out[(size_t)b * A + j] = q[j];
  if (!u) {
    logp[b] = 0.f;
  } else if (kBranched) {
    float s2[kCatMaxBranches];
    logp[b] = categorical_logp_row<true>(x, mrow, A, br, action + (size_t)b * K, q, s2);   // q is scratch now
  }
}

__global__ void gaussian_head_kernel(const float* __restrict__ mu, int ld, const float* __restrict__ log_std,
                                     const float* __restrict__ eps, int B, int A, float* __restrict__ action,
                                     float* __restrict__ logp) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float lp = 0.f;
  for (int j = 0; j < A; ++j) {
    const float m = mu[(size_t)b * ld + j];
    if (eps) {
      const float sd = expf(log_std[j]);
      const float a = __fadd_rn(m, __fmul_rn(sd, eps[(size_t)b * A + j]));   // torch.normal: mul then add
      action[(size_t)b * A + j] = a;
      const float z = a - m;
      lp += -(z * z) / (2.f * (sd * sd)) - logf(sd) - kLogSqrt2Pi;          // normal.py:87-102
    } else {
      action[(size_t)b * A + j] = m;                                         // server/forward.py:141
    }
  }
  logp[b] = lp;
}

// Beta head (beta.cuh): thread (r, j) of a block handles dimension j of the block's row r.  Sampling (u given): x = I^-1(u) in
// fp64, clamped into [eps, 1 - eps], a = low + (high - low) * fp32(x) (mul then add); the row's log-prob is then beta_logp of the
// emitted action.  Play mode (u null): the mean low + (high - low) * alpha / (alpha + beta), log-prob 0.  conc_out [B, 2A]
// (optional) receives alpha | beta.
constexpr int kBetaHeadThreads = 128;

__global__ void __launch_bounds__(kBetaHeadThreads) beta_head_kernel(const float* __restrict__ z, int ld,
                                                                    const float* __restrict__ low, const float* __restrict__ high,
                                                                    const float* __restrict__ u, int B, int A,
                                                                    float* __restrict__ action, float* __restrict__ logp,
                                                                    float* __restrict__ conc_out) {
  __shared__ float act_s[kBetaHeadThreads];
  const int rows = kBetaHeadThreads / A;
  const int r = threadIdx.x / A, j = threadIdx.x - r * A;
  const long long b = (long long)blockIdx.x * rows + r;
  const bool live = r < rows && b < B;
  if (live) {
    const float* zr = z + b * ld;
    const float al = beta_conc(zr[j]), be = beta_conc(zr[A + j]);
    if (conc_out) { conc_out[b * 2 * A + j] = al; conc_out[b * 2 * A + A + j] = be; }
    const float w = high[j] - low[j];
    float a;
    if (u) {
      const float x = (float)beta_clamp_x(beta_inc_inv(al, be, u[b * A + j]));
      a = __fadd_rn(low[j], __fmul_rn(w, x));
    } else {
      a = __fadd_rn(low[j], __fmul_rn(w, __fdiv_rn(al, __fadd_rn(al, be))));
    }
    action[b * A + j] = a;
    act_s[threadIdx.x] = a;
  }
  __syncthreads();
  if (live && j == 0) logp[b] = u ? beta_logp(z + b * ld, low, high, act_s + threadIdx.x, A) : 0.f;
}

}  // namespace ddrl

using namespace ddrl;

extern "C" int ddrl_sample_categorical_probs(const float* probs, int ld, const float* u, int B, int A, float* action,
                                             float* logp, void* stream) {
  if (B < 0 || A < 1 || ld < A) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!probs || !action) return DDRL_E_ARG;
  sample_probs_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(probs, ld, u, B, A, action, logp);
  DDRL_LAUNCHED("sample_probs_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_categorical_head_m(const float* logits, int ld, const float* u, int B, int A, float* action,
                                       float* logp, float* probs_out, const float* mask, void* stream) {
  if (B < 0 || A < 1 || A > kMaxA || ld < A) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!logits || !action || !logp) return DDRL_E_ARG;
  categorical_head_kernel<false><<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(logits, ld, u, B, A, CatBranches{}, action,
                                                                                     logp, probs_out, mask);
  DDRL_LAUNCHED("categorical_head_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_multi_categorical_head(const float* logits, int ld, const float* u, int B, int K, const int32_t* nvec,
                                           float* action, float* logp, float* probs_out, const float* mask, void* stream) {
  CatBranches br;
  int A = 0;
  const int e = cat_branches(K, nvec, &br, &A);
  if (e != DDRL_OK) return e;
  if (B < 0 || ld < A) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!logits || !action || !logp) return DDRL_E_ARG;
  categorical_head_kernel<true><<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(logits, ld, u, B, A, br, action, logp,
                                                                                    probs_out, mask);
  DDRL_LAUNCHED("multi_categorical_head_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_categorical_head(const float* logits, int ld, const float* u, int B, int A, float* action,
                                     float* logp, float* probs_out, void* stream) {
  return ddrl_categorical_head_m(logits, ld, u, B, A, action, logp, probs_out, nullptr, stream);
}

extern "C" int ddrl_gaussian_head(const float* mu, int ld, const float* log_std, const float* eps, int B, int A,
                                  float* action, float* logp, void* stream) {
  if (B < 0 || A < 1 || ld < A) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!mu || !log_std || !action || !logp) return DDRL_E_ARG;
  gaussian_head_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(mu, ld, log_std, eps, B, A, action, logp);
  DDRL_LAUNCHED("gaussian_head_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_beta_head(const float* head, int ld, const float* low, const float* high, const float* u, int B, int A,
                              float* action, float* logp, float* conc_out, void* stream) {
  if (B < 0 || A < 1 || A > kBetaMaxA || ld < 2 * A) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  if (!head || !low || !high || !action || !logp) return DDRL_E_ARG;
  const int rows = kBetaHeadThreads / A;
  beta_head_kernel<<<ceil_div(B, rows), kBetaHeadThreads, 0, (cudaStream_t)stream>>>(head, ld, low, high, u, B, A, action, logp,
                                                                                      conc_out);
  DDRL_LAUNCHED("beta_head_kernel");
  return DDRL_OK;
}
