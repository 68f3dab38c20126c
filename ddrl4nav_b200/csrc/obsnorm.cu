// Running observation normalisation (non-reference option NORM_OBS of nn/ppo.py), gym RunningMeanStd conventions:
//
//   ddrl_obs_moments      column sums of d = x - shift and d^2 in fp64 over a row-major fp32 [B, D]
//   ddrl_obs_rms_update   Chan's parallel merge of one batch into the running {mean, var, count}, then the applied form
//                         mean32 = fp32(mean), scale32 = fp32(1 / sqrt(var + 1e-8))
//   ddrl_obs_normalize    out = min(max((x - mean32) * scale32, -clip), clip)
//
// The statistics must be the same bits on every data-parallel rank and in every predictor, so the moments use a reduction
// order that depends on (B, D) only: rows are cut into fixed chunks of kMomChunkRows, each block sums one chunk of one column
// tile (row lane l of the block takes rows l, l + 8, ... of the chunk in order, then the 8 lanes are added in order), and a
// second launch adds the chunk partials in chunk order.  The vector and the scalar load paths visit every column's rows in the
// same order, so alignment changes the speed, never the bits.  Shifting by the running mean keeps the fp64 sums well
// conditioned; every rank shifts by the same mean, so the sums of the ranks can simply be all-reduced.
#include <algorithm>

#include "common.cuh"

namespace ddrl {

constexpr int kMomThreads = 256;
constexpr int kMomLanes = 8;                        // row lanes of a block
constexpr int kMomColThreads = kMomThreads / kMomLanes;   // 32: one warp per row lane reads one contiguous row segment
constexpr int kMomChunkRows = 256;                  // rows per partial: fixes the reduction order for given (B, D)
constexpr int kMomUnroll = 4;
constexpr int kNormThreads = 256;
constexpr int kNormUnroll = 4;
constexpr int kRmsThreads = 1024;

inline int64_t obs_moment_chunks(int B) { return B > 0 ? ceil_div64(B, kMomChunkRows) : 0; }

template <int VEC>
__device__ __forceinline__ void load_cols(const float* p, float* v) {
  if constexpr (VEC == 4) {
    const float4 q = ld_stream4(reinterpret_cast<const float4*>(p));
    v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
  } else {
    v[0] = ld_stream(p);
  }
}

// grid (column tiles of kMomColThreads * VEC columns, row chunks); part: [chunks][2D] = {sum d, sum d^2} per chunk
template <int VEC>
__global__ void __launch_bounds__(kMomThreads) obs_moments_kernel(const float* __restrict__ x, int B, int D,
                                                                  const double* __restrict__ shift, double* __restrict__ part) {
  constexpr int kTile = kMomColThreads * VEC;
  __shared__ double s_sum[kMomLanes][kTile];
  __shared__ double s_sq[kMomLanes][kTile];
  const int ct = threadIdx.x % kMomColThreads, lane = threadIdx.x / kMomColThreads;
  const int64_t tile0 = (int64_t)blockIdx.x * kTile;
  const int64_t col = tile0 + (int64_t)ct * VEC;      // VEC == 4 only when D % 4 == 0: col < D covers all four columns
  const int r0 = blockIdx.y * kMomChunkRows, r1 = min(B, r0 + kMomChunkRows);
  double s1[VEC], s2[VEC], sh[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    s1[v] = 0.0;
    s2[v] = 0.0;
    sh[v] = col < D ? shift[col + v] : 0.0;
  }
  if (col < D) {
    for (int r = r0 + lane; r < r1; r += kMomLanes * kMomUnroll) {
      float val[kMomUnroll][VEC];
#pragma unroll
      for (int k = 0; k < kMomUnroll; ++k) {
        const int row = r + k * kMomLanes;
        if (row < r1) load_cols<VEC>(x + (int64_t)row * D + col, val[k]);
      }
#pragma unroll
      for (int k = 0; k < kMomUnroll; ++k) {
        if (r + k * kMomLanes >= r1) break;
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          const double d = (double)val[k][v] - sh[v];
          s1[v] += d;
          s2[v] += d * d;
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    s_sum[lane][ct * VEC + v] = s1[v];
    s_sq[lane][ct * VEC + v] = s2[v];
  }
  __syncthreads();
  double* out = part + (int64_t)blockIdx.y * 2 * D;
  for (int t = threadIdx.x; t < kTile; t += blockDim.x) {
    const int64_t c = tile0 + t;
    if (c >= D) break;
    double a = 0.0, b = 0.0;
#pragma unroll
    for (int l = 0; l < kMomLanes; ++l) {
      a += s_sum[l][t];
      b += s_sq[l][t];
    }
    out[c] = a;
    out[D + c] = b;
  }
}

// sums[i] = sum over chunks c, in order, of part[c][i], i < 2D
__global__ void __launch_bounds__(256) obs_moments_reduce_kernel(const double* __restrict__ part, int64_t chunks, int64_t n2,
                                                                 double* __restrict__ sums) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int64_t c = 0; c < chunks; ++c) s += part[c * n2 + i];
    sums[i] = s;
  }
}

// ONE block: every thread reads the count before thread 0 rewrites it
__global__ void __launch_bounds__(kRmsThreads) obs_rms_update_kernel(double* __restrict__ mean, double* __restrict__ var,
                                                                     double* __restrict__ count, const double* __restrict__ sums,
                                                                     double n, int D, float* __restrict__ mean32,
                                                                     float* __restrict__ scale32) {
  const double c = *count;
  const double tot = c + n;
  for (int j = threadIdx.x; j < D; j += blockDim.x) {
    double m = mean[j], v = var[j];
    if (n > 0.0) {
      const double delta = sums[j] / n;                            // batch mean - running mean (the sums are shifted by it)
      const double bvar = fmax(sums[D + j] / n - delta * delta, 0.0);   // population variance of the batch
      m = m + delta * n / tot;
      v = (v * c + bvar * n + delta * delta * c * n / tot) / tot;
      mean[j] = m;
      var[j] = v;
    }
    mean32[j] = (float)m;
    scale32[j] = (float)(1.0 / sqrt(v + 1e-8));
  }
  __syncthreads();
  if (n > 0.0 && threadIdx.x == 0) *count = tot;
}

// grid (column groups, row stripes); each thread keeps its columns' mean / scale in registers and walks rows y, y + gridDim.y, ...
// Plain coherent loads: x may be out (each element is read, then written, by the same thread).
template <int VEC>
__global__ void __launch_bounds__(kNormThreads) obs_normalize_kernel(const float* x, int B, int D, const float* __restrict__ mean32,
                                                                     const float* __restrict__ scale32, float clip, float* out) {
  const int64_t col = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * VEC;
  if (col >= D) return;
  float m[VEC], s[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    m[v] = mean32[col + v];
    s[v] = scale32[col + v];
  }
  const int step = gridDim.y;
  for (int r = blockIdx.y; r < B; r += step * kNormUnroll) {
    float val[kNormUnroll][VEC];
#pragma unroll
    for (int k = 0; k < kNormUnroll; ++k) {
      const int row = r + k * step;
      if (row >= B) continue;
      const float* p = x + (int64_t)row * D + col;
      if constexpr (VEC == 4) {
        const float4 q = __ldcs(reinterpret_cast<const float4*>(p));
        val[k][0] = q.x; val[k][1] = q.y; val[k][2] = q.z; val[k][3] = q.w;
      } else {
        val[k][0] = __ldcs(p);
      }
    }
#pragma unroll
    for (int k = 0; k < kNormUnroll; ++k) {
      const int row = r + k * step;
      if (row >= B) continue;
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        // a subtract, a multiply and a clamp, each rounded on its own: torch reproduces it to the bit
        float y = __fmul_rn(__fsub_rn(val[k][v], m[v]), s[v]);
        if (clip > 0.f) y = y < -clip ? -clip : (y > clip ? clip : y);     // NaN passes through, as in torch.clamp
        val[k][v] = y;
      }
      float* q = out + (int64_t)row * D + col;
      if constexpr (VEC == 4) __stcs(reinterpret_cast<float4*>(q), make_float4(val[k][0], val[k][1], val[k][2], val[k][3]));
      else __stcs(q, val[k][0]);
    }
  }
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

}  // namespace ddrl

using namespace ddrl;

extern "C" int64_t ddrl_obs_moments_ws_bytes(int B, int D) {
  if (B < 0 || D < 1) return DDRL_E_ARG;
  const int64_t chunks = obs_moment_chunks(B);
  return chunks > 1 ? chunks * 2 * (int64_t)D * (int64_t)sizeof(double) : 0;
}

extern "C" int ddrl_obs_moments(const float* x, int B, int D, const double* shift, double* sums, void* ws, int64_t ws_bytes,
                                void* stream) {
  if (B < 0 || D < 1 || !shift || !sums || (B > 0 && !x)) return DDRL_E_ARG;
  const int64_t chunks = obs_moment_chunks(B);
  if (chunks > 65535) return DDRL_E_ARG;
  cudaStream_t s = (cudaStream_t)stream;
  if (B == 0) {
    DDRL_CUDA(cudaMemsetAsync(sums, 0, 2 * (size_t)D * sizeof(double), s));
    return DDRL_OK;
  }
  const int64_t need = ddrl_obs_moments_ws_bytes(B, D);
  if (need > 0 && (!ws || ws_bytes < need)) return DDRL_E_ARG;
  double* part = need > 0 ? static_cast<double*>(ws) : sums;     // one chunk: its partial is the result
  const bool vec = D % 4 == 0 && aligned16(x);
  const int64_t tile = (int64_t)kMomColThreads * (vec ? 4 : 1);
  const dim3 grid((unsigned)ceil_div64(D, tile), (unsigned)chunks);
  prof_work(4.0 * (double)B * D);
  if (vec) obs_moments_kernel<4><<<grid, kMomThreads, 0, s>>>(x, B, D, shift, part);
  else obs_moments_kernel<1><<<grid, kMomThreads, 0, s>>>(x, B, D, shift, part);
  DDRL_LAUNCHED("obs_moments_kernel");
  if (need > 0) {
    const int64_t n2 = 2 * (int64_t)D;
    const int blocks = (int)std::min<int64_t>(ceil_div64(n2, 256), 8LL * kNumSMs);
    prof_work(8.0 * (double)(chunks + 1) * n2);
    obs_moments_reduce_kernel<<<blocks, 256, 0, s>>>(part, chunks, n2, sums);
    DDRL_LAUNCHED("obs_moments_reduce_kernel");
  }
  return DDRL_OK;
}

extern "C" int ddrl_obs_rms_update(double* mean, double* var, double* count, const double* sums, double n, int D, float* mean32,
                                   float* scale32, void* stream) {
  if (!mean || !var || !count || !mean32 || !scale32 || D < 1 || !(n >= 0.0) || (n > 0.0 && !sums)) return DDRL_E_ARG;
  prof_work(8.0 * 5 * D);
  obs_rms_update_kernel<<<1, kRmsThreads, 0, (cudaStream_t)stream>>>(mean, var, count, sums, n, D, mean32, scale32);
  DDRL_LAUNCHED("obs_rms_update_kernel");
  return DDRL_OK;
}

extern "C" int ddrl_obs_normalize(const float* x, int B, int D, const float* mean32, const float* scale32, float clip, float* out,
                                  void* stream) {
  if (B < 0 || D < 1 || !mean32 || !scale32 || (B > 0 && (!x || !out)) || clip != clip) return DDRL_E_ARG;
  if (B == 0) return DDRL_OK;
  const bool vec = D % 4 == 0 && aligned16(x) && aligned16(out) && aligned16(mean32) && aligned16(scale32);
  const int64_t per_row = vec ? D / 4 : D;
  const int gx = (int)ceil_div64(per_row, kNormThreads);
  const int gy = (int)std::min<int64_t>(std::min(B, 65535), std::max<int64_t>(1, ceil_div64(8LL * kNumSMs, gx)));
  const dim3 grid((unsigned)gx, (unsigned)gy);
  prof_work(8.0 * (double)B * D);
  if (vec) obs_normalize_kernel<4><<<grid, kNormThreads, 0, (cudaStream_t)stream>>>(x, B, D, mean32, scale32, clip, out);
  else obs_normalize_kernel<1><<<grid, kNormThreads, 0, (cudaStream_t)stream>>>(x, B, D, mean32, scale32, clip, out);
  DDRL_LAUNCHED("obs_normalize_kernel");
  return DDRL_OK;
}
