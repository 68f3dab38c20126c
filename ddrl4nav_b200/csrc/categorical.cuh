// The categorical softmax with an optional action mask (ACTION_MASK), shared by the head kernel (heads.cu) and by the loss and
// log-prob pre-pass kernels (ppo_loss.cu), so that all three compute the same bits from the same logits and mask.
//
// mask: the row's [A] fp32 mask (action j allowed iff mask[j] != 0), or null when every action is allowed.  The masked softmax
// is torch's softmax(logits.masked_fill(~m, -inf)): the max is taken over the allowed entries only, masked entries get p = 0
// exactly (no expf; their logits are never read), and the rest is the unmasked arithmetic in the same order.  An all-ones mask
// therefore gives the bits of no mask.  A row that allows no action is treated as allowing every action.
//
// MultiDiscrete (DDRL_DIST_MULTI_CATEGORICAL): K independent branches over one head row of width A = n_1 + ... + n_K, branch i on
// the columns [o_i, o_i + n_i), o_i = n_1 + ... + n_{i-1}.  Every branch runs the categorical arithmetic above on its own slice
// (its own mask slice, and its own "allows nothing" rule).  The kernels take the branch table by value, so captured graphs need
// nothing more; they are templates over kBranched, and the categorical actor is the kBranched = false instantiation (one branch
// of width A, at compile time), which keeps its code, registers and bits.
#pragma once

#include "common.cuh"

namespace ddrl {

constexpr float kCatEps = 1.1920928955078125e-07f;   // torch.finfo(float32).eps: the Categorical clamp
constexpr int kCatMaxA = 64;                          // head width of a categorical / MultiDiscrete actor
constexpr int kCatMaxBranches = 8;

// the MultiDiscrete branch table: K branches of n[0..K) actions
struct CatBranches {
  int K;
  int n[kCatMaxBranches];
};

// checks a host branch table (1 <= K <= 8, every n_i >= 1: else DDRL_E_ARG; sum n_i <= 64: else DDRL_E_UNSUPPORTED) and copies it
// into *br, with *A = sum n_i
inline int cat_branches(int K, const int32_t* nvec, CatBranches* br, int* A) {
  if (!nvec || K < 1 || K > kCatMaxBranches) return DDRL_E_ARG;
  *br = CatBranches{};
  br->K = K;
  int sum = 0;
  for (int i = 0; i < K; ++i) {
    if (nvec[i] < 1 || nvec[i] > kCatMaxA) return DDRL_E_ARG;
    br->n[i] = nvec[i];
    sum += nvec[i];
  }
  if (sum > kCatMaxA) return DDRL_E_UNSUPPORTED;
  *A = sum;
  return DDRL_OK;
}

// the row's mask as the kernels read it: null without a mask, and null for a row that allows nothing
__device__ __forceinline__ const float* categorical_row_mask(const float* __restrict__ mask, int A) {
  if (!mask) return nullptr;
  for (int j = 0; j < A; ++j)
    if (mask[j] != 0.f) return mask;
  return nullptr;
}

__device__ __forceinline__ bool categorical_allowed(const float* __restrict__ mask, int j) { return !mask || mask[j] != 0.f; }

// first allowed action (0 without a mask); `mask` comes from categorical_row_mask, so one exists
__device__ __forceinline__ int categorical_first_allowed(const float* __restrict__ mask, int A) {
  int j = 0;
  if (mask)
    while (j < A - 1 && mask[j] == 0.f) ++j;
  return j;
}

// F.softmax of x[0..A) over the allowed entries into p[0..A) (j0 = categorical_first_allowed); returns s2 = sum(p), the divisor
// of the Categorical re-normalisation q = p / s2 (torch/distributions/categorical.py:70)
__device__ __forceinline__ float categorical_softmax(const float* __restrict__ x, const float* __restrict__ mask, int A, int j0,
                                                     float* p) {
  float m = x[j0];
  for (int j = j0 + 1; j < A; ++j)
    if (categorical_allowed(mask, j)) m = fmaxf(m, x[j]);
  float s = 0.f;
  for (int j = 0; j < A; ++j) { p[j] = categorical_allowed(mask, j) ? expf(x[j] - m) : 0.f; s += p[j]; }
  float s2 = 0.f;
  for (int j = 0; j < A; ++j) { p[j] = p[j] / s; s2 += p[j]; }
  return s2;
}

// log-prob of the taken action a (clamped into [0, A)) under Categorical(logits = x[0..A)) with the row's mask (or null): the
// masked softmax -> q = p / sum(p) -> clamp(eps, 1 - eps) -> log chain of torch.  Leaves the softmax p[0..A) and s2 = sum(p) for
// the loss kernel's gradient.
__device__ __forceinline__ float categorical_logp(const float* __restrict__ x, const float* __restrict__ mask, int A, float action,
                                                  float* p, float* s2_out) {
  mask = categorical_row_mask(mask, A);
  const float s2 = categorical_softmax(x, mask, A, categorical_first_allowed(mask, A), p);
  int a = (int)action;                      // Categorical.log_prob: value.long()
  a = a < 0 ? 0 : (a >= A ? A - 1 : a);     // the reference raises on an action outside [0, A); never read out of bounds
  const float qa = p[a] / s2;
  const float ca = fminf(fmaxf(qa, kCatEps), 1.f - kCatEps);
  *s2_out = s2;
  return logf(ca);
}

// log-prob of the taken action row act[0..K) of one head row x[0..A) (mask: the row's [A] mask or null): categorical_logp of each
// branch on its slice, added in branch order in fp32.  Leaves each branch's softmax in p[o_i ..) and its sum in s2[i].  The loss
// kernel, the log-prob pre-pass and the MultiDiscrete head all call it, so equal logits, masks and actions give equal bits.
template <bool kBranched>
__device__ __forceinline__ float categorical_logp_row(const float* __restrict__ x, const float* __restrict__ mask, int A,
                                                      const CatBranches& br, const float* __restrict__ act, float* p, float* s2) {
  if (!kBranched) return categorical_logp(x, mask, A, act[0], p, s2);
  float lp = 0.f;                           // 0 + l_0 == l_0 exactly (l_0 < 0): K = 1 gives the categorical bits
  for (int i = 0, o = 0; i < br.K; ++i) {
    const int n = br.n[i];
    lp += categorical_logp(x + o, mask ? mask + o : nullptr, n, act[i], p + o, s2 + i);
    o += n;
  }
  return lp;
}

}  // namespace ddrl
