// The categorical softmax with an optional action mask (ACTION_MASK), shared by the head kernel (heads.cu) and by the loss and
// log-prob pre-pass kernels (ppo_loss.cu), so that all three compute the same bits from the same logits and mask.
//
// mask: the row's [A] fp32 mask (action j allowed iff mask[j] != 0), or null when every action is allowed.  The masked softmax
// is torch's softmax(logits.masked_fill(~m, -inf)): the max is taken over the allowed entries only, masked entries get p = 0
// exactly (no expf; their logits are never read), and the rest is the unmasked arithmetic in the same order.  An all-ones mask
// therefore gives the bits of no mask.  A row that allows no action is treated as allowing every action.
#pragma once

namespace ddrl {

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

}  // namespace ddrl
