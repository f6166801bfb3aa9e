// Helpers shared by the elementwise forward (elementwise.cu) and backward (backward.cu) kernels.
// Thread mapping used everywhere: blockIdx.y = (sample, plane); a thread owns one 16-byte chunk
// (8 channels of one voxel) per loop trip, consecutive threads consecutive voxels (coalesced).
#pragma once

#include "common.cuh"

namespace vdm {


constexpr int kEwThreads = 256;

// Reduce per-thread (sum[L], sq[L]) over the block, then 2L fp64 atomics into stats[c0..c0+L) (L = 8 bf16 or 4 fp32 lanes).
template <int L = 8>
__device__ __forceinline__ void block_flush_stats(float (&sum)[L], float (&sq)[L], double* __restrict__ stats8) {
  __shared__ float s_part[kEwThreads / 32][2 * L];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < L; ++j) {
    sum[j] = warp_sum(sum[j]);
    sq[j] = warp_sum(sq[j]);
  }
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < L; ++j) {
      s_part[warp][j] = sum[j];
      s_part[warp][L + j] = sq[j];
    }
  }
  __syncthreads();
  if (threadIdx.x < 2 * L) {
    float acc = 0.f;
#pragma unroll
    for (int w = 0; w < kEwThreads / 32; ++w) acc += s_part[w][threadIdx.x];
    // stats layout: [channel][2]; threadIdx.x < L -> sums, >= L -> sums of squares
    atomicAdd(stats8 + 2 * (threadIdx.x % L) + (threadIdx.x / L), (double)acc);
  }
  __syncthreads();
}

template <typename T = bf16x8>
__device__ __forceinline__ const T* plane_ptr(const VdmTensor& t, int b, int plane, int64_t voxels) {
  return reinterpret_cast<const T*>(t.data) + ((int64_t)b * t.planes + t.plane0 + plane) * voxels;
}
template <typename T = bf16x8>
__device__ __forceinline__ T* plane_ptr_mut(const VdmTensor& t, int b, int plane, int64_t voxels) {
  return reinterpret_cast<T*>(t.data) + ((int64_t)b * t.planes + t.plane0 + plane) * voxels;
}

// ---- GroupNorm scale/shift of the L (8 bf16 or 4 fp32) channels of one plane ----------------------
// y = x*scale + shift  ==  gamma*(x-mean)*rstd + beta ; stats are [B][C][2] for exactly this tensor.
template <int L = 8>
__device__ __forceinline__ void plane_scale_shift(const double* __restrict__ stats_b, int C, int groups, int pl,
                                                  double voxels, const float* __restrict__ gamma,
                                                  const float* __restrict__ beta, float eps, float* s_scale,
                                                  float* s_shift, float* s_mean, float* s_rstd) {
  if (threadIdx.x < L) {
    const int c = pl * L + threadIdx.x;
    const int cpg = C / groups;
    const int g0 = (c / cpg) * cpg;
    double s1 = 0.0, s2 = 0.0;
    for (int k = 0; k < cpg; ++k) {
      s1 += stats_b[2 * (g0 + k)];
      s2 += stats_b[2 * (g0 + k) + 1];
    }
    const double n = voxels * cpg;
    const double mean = s1 / n;
    double var = s2 / n - mean * mean;
    if (var < 0.0) var = 0.0;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float sc = gamma[c] * rstd;
    s_scale[threadIdx.x] = sc;
    s_shift[threadIdx.x] = beta[c] - (float)mean * sc;
    if (s_mean) {
      s_mean[threadIdx.x] = (float)mean;
      s_rstd[threadIdx.x] = rstd;
    }
  }
}

// 8 keep-flags for chunk `chunk` of dropout layer `tag`: bit j set = keep element j.
__device__ __forceinline__ uint32_t dropout_keep8(uint64_t chunk, uint32_t tag, uint64_t seed, uint32_t thresh16) {
  const uint4 w = philox4x32_7(make_uint4((uint32_t)chunk, (uint32_t)(chunk >> 32), tag, kStreamTagDropout),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const uint32_t r[4] = {w.x, w.y, w.z, w.w};
  uint32_t keep = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    keep |= ((r[i] & 0xffffu) >= thresh16 ? 1u : 0u) << (2 * i);
    keep |= ((r[i] >> 16) >= thresh16 ? 1u : 0u) << (2 * i + 1);
  }
  return keep;
}

static inline dim3 ew_grid(int64_t voxels, int batch_planes) {
  int64_t blocks = (voxels + kEwThreads * 4 - 1) / (kEwThreads * 4);
  const int64_t cap = ((int64_t)kNumSMs * 8 + batch_planes - 1) / batch_planes;  // 8 CTAs of 256 threads per SM
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return dim3((unsigned)blocks, (unsigned)batch_planes);
}

// A window of `channels` channels, L per 16-byte plane (8 bf16 or 4 fp32), inside a 16-byte aligned planar buffer.
template <int L>
static inline bool view_ok(const VdmTensor* t, int channels) {
  return t && t->data && channels >= L && channels % L == 0 && t->plane0 >= 0 && t->planes >= t->plane0 + channels / L &&
         (reinterpret_cast<uintptr_t>(t->data) & 15) == 0;
}

// blockIdx.y = (sample, plane) of an L-lane tensor must fit the 65535 limit of gridDim.y.
#define VDM_CHECK_PLANES(L, batch, channels, who) \
  VDM_CHECK_ARG((int64_t)(batch) * ((channels) / (L)) <= 65535, "%s: batch * planes exceeds 65535", who)

// Arguments of the GroupNorm + SiLU passes, forward (x, y) and backward (x, dy).
template <int L>
static inline int check_gn(const char* who, const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels,
                           int groups, const double* stats, const float* gamma, const float* beta, float dropout_p) {
  VDM_CHECK_ARG(view_ok<L>(x, channels) && view_ok<L>(y, channels) && stats && gamma && beta, "%s: bad tensor argument", who);
  VDM_CHECK_ARG(batch >= 1 && voxels >= 1, "%s: bad shape", who);
  VDM_CHECK_PLANES(L, batch, channels, who);
  VDM_CHECK_ARG(groups >= 1 && channels % groups == 0, "%s: %d channels not divisible into %d groups", who, channels, groups);
  VDM_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, "%s: dropout_p %f out of [0,1)", who, dropout_p);
  return VDM_OK;
}

// Pooling and up-sampling grids: fewer than 2^31 voxels (the kernels split a plane index with 32-bit divisions) and, when
// `even`, every extent even.  `noun` ("grid" or "fine grid") names the grid in the message.
static inline int check_grid(const char* who, const char* noun, int depth, int height, int width, bool even) {
  VDM_CHECK_ARG((int64_t)depth * height * width < ((int64_t)1 << 31), "%s: grid too large for 32-bit voxel indices", who);
  VDM_CHECK_ARG(!even || (depth >= 2 && height >= 2 && width >= 2 && depth % 2 == 0 && height % 2 == 0 && width % 2 == 0),
                "%s: %s (%d,%d,%d) must be even", who, noun, depth, height, width);
  return VDM_OK;
}

}  // namespace vdm
