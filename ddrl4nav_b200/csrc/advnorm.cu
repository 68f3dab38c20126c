// Advantage normalisation of one optimiser step's rows (non-reference option NORM_ADV of nn/ppo.py):
//   out = (a - mean) / (std + eps),  std = unbiased standard deviation (torch's Tensor.std()).
//
// The rows of one step are at most a few 10^4 per rank, so ONE block does the whole job: every thread sums a fixed strided
// subset in fp64, the block adds the partials in a fixed tree, and the result is bit-reproducible run to run without the
// engine's deterministic mode.  A data-parallel learner takes the moments {n, sum a, sum a^2} of its local rows
// (ddrl_adv_moments), all-reduces them, and normalises with the global moments; a single device passes m3 = NULL and the
// normalising launch computes the local moments itself.
#include "common.cuh"

namespace ddrl {

constexpr int kAdvThreads = 1024;

// {sum a, sum a^2} of a[0..n), valid in every thread
__device__ __forceinline__ void adv_block_moments(const float* __restrict__ a, int n, double* s1, double* s2) {
  __shared__ double scratch[32];
  __shared__ double tot[2];
  double x = 0.0, xx = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = (double)a[i];
    x += v;
    xx += v * v;
  }
  x = block_sum(x, scratch);
  xx = block_sum(xx, scratch);
  if (threadIdx.x == 0) { tot[0] = x; tot[1] = xx; }
  __syncthreads();
  *s1 = tot[0];
  *s2 = tot[1];
}

__global__ void __launch_bounds__(kAdvThreads) adv_moments_kernel(const float* __restrict__ a, int n, double* __restrict__ m3) {
  double s1, s2;
  adv_block_moments(a, n, &s1, &s2);
  if (threadIdx.x == 0) { m3[0] = (double)n; m3[1] = s1; m3[2] = s2; }
}

__global__ void __launch_bounds__(kAdvThreads) adv_normalize_kernel(const float* a, int n, const double* __restrict__ m3,
                                                                    float eps, float* out) {
  double cnt, s1, s2;
  if (m3) { cnt = m3[0]; s1 = m3[1]; s2 = m3[2]; }
  else { cnt = (double)n; adv_block_moments(a, n, &s1, &s2); }
  if (cnt <= 1.0) {                    // torch's std of one element is nan; a one-row minibatch keeps its advantage
    if (out != a) for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = a[i];
    return;
  }
  const double mean = s1 / cnt;
  const double var = fmax((s2 - s1 * mean) / (cnt - 1.0), 0.0);
  const double inv = 1.0 / (sqrt(var) + (double)eps);
  // each thread rewrites exactly the elements it read above, so out == a is safe
  for (int i = threadIdx.x; i < n; i += blockDim.x) out[i] = (float)(((double)a[i] - mean) * inv);
}

}  // namespace ddrl

using namespace ddrl;

extern "C" int ddrl_adv_moments(const float* adv, int n, double* m3, void* stream) {
  if (n < 0 || !m3 || (n > 0 && !adv)) return DDRL_E_ARG;
  adv_moments_kernel<<<1, kAdvThreads, 0, (cudaStream_t)stream>>>(adv, n, m3);
  prof_work(4.0 * n);
  DDRL_LAUNCHED("adv_moments_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_adv_normalize(const float* adv, int n, const double* m3, float eps, float* out, void* stream) {
  if (n < 0 || (n > 0 && (!adv || !out)) || !(eps >= 0.f)) return DDRL_E_ARG;
  if (n == 0) return DDRL_OK;
  adv_normalize_kernel<<<1, kAdvThreads, 0, (cudaStream_t)stream>>>(adv, n, m3, eps, out);
  prof_work((m3 ? 8.0 : 12.0) * n);
  DDRL_LAUNCHED("adv_normalize_kernel");
  return DDRL_OK;
}
