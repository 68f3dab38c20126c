// Multi-tensor row gather: dst row i of every job = src row rows[i], all jobs in ONE launch.
//
// Used by the minibatch learner (nn/ppo.py) to copy the rows of one shuffled minibatch -- every observation slot, the
// actions, old log-probs, advantages and the V return rows -- into persistent minibatch buffers.  Row sizes span four
// orders of magnitude (a Pong row is 4 x 84 x 84 fp32 = 112896 B, a log-prob is 4 B), so the work is mapped to the BYTES,
// not to the rows: job j is n_rows x W_j units (W_j = row_bytes / 16 on the vector path, row_bytes / 4 otherwise), the
// units of all jobs form one flat index space, and a grid-stride loop hands consecutive units to consecutive threads.  A
// wide row is then read and written by whole warps in 512 B runs; a 4 B row costs one scattered sector per unit, which is
// what a gather of 4 B rows costs anyway.  Each thread keeps kUnroll independent loads in flight before it stores.
//
// Out-of-range indices are clamped to [0, src_rows), as the PPO loss clamps action indices: the kernel never reads
// outside a job's source.
#include <limits.h>

#include <algorithm>

#include "common.cuh"

namespace ddrl {

constexpr int kGatherThreads = 256;
constexpr int kGatherUnroll = 4;

struct GatherParams {
  const char* src[DDRL_GATHER_MAX_JOBS];
  char* dst[DDRL_GATHER_MAX_JOBS];
  int64_t src_stride[DDRL_GATHER_MAX_JOBS];
  int64_t dst_stride[DDRL_GATHER_MAX_JOBS];
  int64_t begin[DDRL_GATHER_MAX_JOBS + 1];   // first flat unit of each job; begin[n_jobs] = total
  uint32_t units_per_row[DDRL_GATHER_MAX_JOBS];
  int32_t last_row[DDRL_GATHER_MAX_JOBS];    // src_rows - 1 (clamped to the int32 index range)
  uint8_t vec[DDRL_GATHER_MAX_JOBS];         // 1: 16 B units, 0: 4 B units
  int n_jobs;
};

__global__ void __launch_bounds__(kGatherThreads) gather_rows_kernel(const int32_t* __restrict__ rows,
                                                                     const __grid_constant__ GatherParams p) {
  const int64_t total = p.begin[p.n_jobs];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t base = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; base < total; base += stride * kGatherUnroll) {
    uint4 v[kGatherUnroll];
    char* d[kGatherUnroll];
    bool wide[kGatherUnroll];
#pragma unroll
    for (int k = 0; k < kGatherUnroll; ++k) {
      const int64_t u = base + k * stride;
      d[k] = nullptr;
      wide[k] = false;
      if (u >= total) continue;
      int j = 0;
      while (j + 1 < p.n_jobs && u >= p.begin[j + 1]) ++j;
      const uint64_t off = (uint64_t)(u - p.begin[j]);
      const uint32_t W = p.units_per_row[j];
      const uint64_t i = (off >> 32) == 0 ? (uint64_t)((uint32_t)off / W) : off / W;
      const uint64_t c = off - i * W;
      const int r = min(max(__ldg(rows + i), 0), p.last_row[j]);
      wide[k] = p.vec[j] != 0;
      const char* s = p.src[j] + (int64_t)r * p.src_stride[j];
      d[k] = p.dst[j] + (int64_t)i * p.dst_stride[j];
      if (wide[k]) {
        v[k] = __ldg(reinterpret_cast<const uint4*>(s) + c);
        d[k] += c * 16;
      } else {
        v[k].x = __ldg(reinterpret_cast<const unsigned int*>(s) + c);
        d[k] += c * 4;
      }
    }
#pragma unroll
    for (int k = 0; k < kGatherUnroll; ++k) {
      if (!d[k]) continue;
      if (wide[k]) *reinterpret_cast<uint4*>(d[k]) = v[k];
      else *reinterpret_cast<unsigned int*>(d[k]) = v[k].x;
    }
  }
}

}  // namespace ddrl

extern "C" int ddrl_gather_rows(const int32_t* rows, int n_rows, const ddrl_gather_job* jobs, int n_jobs, void* stream) {
  using namespace ddrl;
  if (!jobs || n_jobs < 1 || n_jobs > DDRL_GATHER_MAX_JOBS || n_rows < 0 || (n_rows > 0 && !rows)) return DDRL_E_ARG;
  GatherParams p{};
  p.n_jobs = n_jobs;
  int64_t total = 0;
  double bytes = 0.0;
  for (int j = 0; j < n_jobs; ++j) {
    const ddrl_gather_job& g = jobs[j];
    const uintptr_t sa = (uintptr_t)g.src, da = (uintptr_t)g.dst;
    if (!g.src || !g.dst || g.row_bytes <= 0 || g.row_bytes % 4 || g.src_stride < 0 || g.dst_stride < 0 || g.src_stride % 4 ||
        g.dst_stride % 4 || sa % 4 || da % 4 || g.src_rows < 0 || (n_rows > 0 && g.src_rows < 1))
      return DDRL_E_ARG;
    const bool vec = sa % 16 == 0 && da % 16 == 0 && g.src_stride % 16 == 0 && g.dst_stride % 16 == 0 && g.row_bytes % 16 == 0;
    const int64_t W = g.row_bytes / (vec ? 16 : 4);
    if (W > UINT32_MAX) return DDRL_E_ARG;
    p.src[j] = static_cast<const char*>(g.src);
    p.dst[j] = static_cast<char*>(g.dst);
    p.src_stride[j] = g.src_stride;
    p.dst_stride[j] = g.dst_stride;
    p.units_per_row[j] = (uint32_t)W;
    p.last_row[j] = (int32_t)std::min<int64_t>(g.src_rows - 1, INT_MAX);
    p.vec[j] = vec ? 1 : 0;
    p.begin[j] = total;
    total += W * n_rows;
    bytes += 2.0 * (double)g.row_bytes * n_rows;
  }
  p.begin[n_jobs] = total;
  if (total == 0) return DDRL_OK;
  const int64_t per_block = (int64_t)kGatherThreads * kGatherUnroll;
  const int blocks = (int)std::min<int64_t>((total + per_block - 1) / per_block, 8LL * kNumSMs);
  prof_work(bytes);
  gather_rows_kernel<<<blocks, kGatherThreads, 0, (cudaStream_t)stream>>>(rows, p);
  DDRL_LAUNCHED("gather_rows_kernel");
  return DDRL_OK;
}
