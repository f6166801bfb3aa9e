// Fused elementwise passes of the ResNet blocks (all HBM-bound, channel-planar bf16, 16-byte accesses).
//
// Stand in for the ATen group_norm / silu / dropout / avg_pool3d / interpolate(nearest) / cat
// launches issued by mltools' ResNetBlock / ResNetDown (blocks.py:129-170 in the traceback of
// model_test.ipynb:686-692).  The reference runs each as its own full-tensor pass; here
//   * GroupNorm statistics are per-channel (sum, sumsq) pairs produced by whichever kernel
//     writes the tensor (conv epilogue, pool, up-sampling) and reduced to groups on the fly,
//   * normalise + affine + SiLU (+ dropout) is one read and one write,
//   * channel concatenation costs nothing: producers write into plane windows of one buffer.
//
// Thread mapping used everywhere: blockIdx.y = (sample, plane); a thread owns one 16-byte chunk
// (8 channels of one voxel) per loop trip, consecutive threads consecutive voxels (coalesced).
#include "ew_common.cuh"

namespace vdm {

// ---- channel statistics -------------------------------------------------------------------
__global__ void __launch_bounds__(kEwThreads)
channel_stats_kernel(VdmTensor x, int planes, int64_t voxels, double* __restrict__ stats, int stats_channels,
                     int stats_c0) {
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const bf16x8* xp = plane_ptr(x, b, pl, voxels);
  float sum[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < voxels; i += (int64_t)gridDim.x * kEwThreads) {
    float f[8];
    unpack8(xp[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      sum[j] += f[j];
      sq[j] += f[j] * f[j];
    }
  }
  block_flush_stats(sum, sq, stats + ((int64_t)b * stats_channels + stats_c0 + pl * 8) * 2);
}

// STREAM: evict-first loads/stores for tensors far larger than L2 (level-0 activations: +20% on the 96-channel
// layer, r01z); small tensors keep default caching so the conv that follows reads them from L2.
// F32: fp32 channel-planar tensors (TF32 inference mode), exp-based SiLU, no dropout.
template <bool STREAM, bool F32 = false>
__global__ void __launch_bounds__(kEwThreads)
gn_silu_kernel(VdmTensor x, VdmTensor y, int planes, int64_t voxels, int groups, const double* __restrict__ stats,
               const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float dropout_p,
               uint64_t seed, const int32_t* __restrict__ seed_step, uint32_t layer_tag) {
  using T = typename Unit<F32>::T;
  constexpr int L = Unit<F32>::L;
  if (seed_step) seed += (uint64_t)(uint32_t)(*seed_step);
  __shared__ float s_scale[L], s_shift[L];
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const int C = planes * L;
  plane_scale_shift<L>(stats + (int64_t)b * C * 2, C, groups, pl, (double)voxels, gamma, beta, eps, s_scale, s_shift,
                       nullptr, nullptr);
  __syncthreads();
  float sc[L], sh[L];                      // bf16: halved, silu(y) = h + h tanh(h), h = y / 2 (silu_half)
#pragma unroll
  for (int j = 0; j < L; ++j) {
    sc[j] = F32 ? s_scale[j] : 0.5f * s_scale[j];
    sh[j] = F32 ? s_shift[j] : 0.5f * s_shift[j];
  }
  const T* xp = plane_ptr<T>(x, b, pl, voxels);
  T* yp = plane_ptr_mut<T>(y, b, pl, voxels);
  const bool drop = dropout_p > 0.f;
  const uint32_t thresh16 = (uint32_t)(dropout_p * 65536.0f + 0.5f);
  const float keep_scale = drop ? 1.0f / (1.0f - dropout_p) : 1.0f;
  const uint64_t chunk0 = ((uint64_t)b * planes + pl) * (uint64_t)voxels;
  // kGnUnroll independent 16-byte loads in flight per thread (memory-level parallelism: r01f measured the one-load-per-
  // trip version at ~50% of the HBM roofline, two loads at ~73%)
  constexpr int U = 4;
  const int64_t stride = (int64_t)gridDim.x * kEwThreads;
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < voxels; i += U * stride) {
    T v[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t ii = i + k * stride;
      if (ii < voxels) v[k] = STREAM ? ld_stream(xp + ii) : xp[ii];
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t ii = i + k * stride;
      if (ii >= voxels) break;
      float f[L];
      unpack_unit(v[k], f);
#pragma unroll
      for (int j = 0; j < L; ++j) f[j] = F32 ? silu_f32(fmaf(f[j], sc[j], sh[j])) : silu_half(fmaf(f[j], sc[j], sh[j]));
      if constexpr (!F32) {
        if (drop) {
          const uint32_t keep = dropout_keep8(chunk0 + (uint64_t)ii, layer_tag, seed, thresh16);
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = ((keep >> j) & 1u) ? f[j] * keep_scale : 0.f;
        }
      }
      T out;
      pack_unit(f, out);
      if (STREAM) st_stream(yp + ii, out);
      else yp[ii] = out;
    }
  }
}

// ---- GroupNorm coefficients for the conv kernel's fused input transform ----------------------------------------
// coef[b][c] = (a, b) with  silu(gn(x)) = h + h * tanh(h),  h = a * x + b = (gamma * rstd * x + beta - mean * gamma * rstd) / 2:
// the per-(sample, channel) pair conv3d_planar_kernel's transform warps apply to the landed halo tile (csrc/conv3d.cu).
// One thread per (sample, channel); group sums are re-derived per thread from the fp64 (sum, sumsq) table.
__global__ void gn_coef_kernel(const double* __restrict__ stats, int batch, int C, int groups, double voxels,
                               const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                               float2* __restrict__ coef) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= batch * C) return;
  const int b = i / C, c = i - b * C;
  const int cpg = C / groups;
  const int g0 = (c / cpg) * cpg;
  const double* sb = stats + (int64_t)b * C * 2;
  double s1 = 0.0, s2 = 0.0;
  for (int k = 0; k < cpg; ++k) {
    s1 += sb[2 * (g0 + k)];
    s2 += sb[2 * (g0 + k) + 1];
  }
  const double n = voxels * cpg;
  const double mean = s1 / n;
  double var = s2 / n - mean * mean;
  if (var < 0.0) var = 0.0;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float sc = gamma[c] * rstd;
  const float sh = beta[c] - (float)mean * sc;      // same roundings as plane_scale_shift (the unfused kernels)
  coef[i] = make_float2(0.5f * sc, 0.5f * sh);
}

// ---- GroupNorm + SiLU of a channel window of a wider norm, optionally through a nearest x2 up-sampling ------------
// The up blocks normalise cat([upsample(h_coarse), skip]).  Nearest-neighbour up-sampling commutes with every
// pointwise operation and leaves per-channel means and variances unchanged, so the up-sampled tensor is never
// written: this kernel reads the COARSE channels [c_off, c_off + 8*planes) of the C_total-channel norm and writes
// silu(gn(.)) at the fine resolution (UP), or handles the skip channels of the same norm in place (!UP).
// stats: double [B][C_total][2] of the FINE-resolution concat (for up-sampled channels: 8x the coarse sums).
// (D, H, W) is the grid of y.
template <bool UP>
__global__ void __launch_bounds__(kEwThreads)
gn_silu_view_kernel(VdmTensor x, VdmTensor y, int planes, int c_off, int C_total, int groups, int D, int H, int W,
                    const double* __restrict__ stats, const float* __restrict__ gamma, const float* __restrict__ beta,
                    float eps, double stats_voxels) {
  __shared__ float s_scale[8], s_shift[8];
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const int64_t vf = (int64_t)D * H * W;
  plane_scale_shift(stats + (int64_t)b * C_total * 2, C_total, groups, (c_off >> 3) + pl, stats_voxels, gamma, beta, eps,
                    s_scale, s_shift, nullptr, nullptr);
  __syncthreads();
  float sc[8], sh[8];                      // halved: silu(y) = h + h tanh(h), h = y / 2 (silu_half)
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc[j] = 0.5f * s_scale[j];
    sh[j] = 0.5f * s_shift[j];
  }
  bf16x8* yp = plane_ptr_mut(y, b, pl, vf);
  const int64_t stride = (int64_t)gridDim.x * kEwThreads;
  if (UP) {
    const int Hc = H >> 1, Wc = W >> 1;
    const bf16x8* cp = plane_ptr(x, b, pl, vf >> 3);
    // one thread per (fine d, fine h, COARSE w): one 16-byte read (repeats hit L1/L2), two adjacent 16-byte stores
    const int64_t vh = vf >> 1;
    for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < vh; i += stride) {
      unsigned v = (unsigned)i;
      const int wc = (int)(v % (unsigned)Wc); v /= (unsigned)Wc;
      const int h = (int)(v % (unsigned)H);
      const int d = (int)(v / (unsigned)H);
      float f[8];
      unpack8(cp[((int64_t)(d >> 1) * Hc + (h >> 1)) * Wc + wc], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = silu_half(fmaf(f[j], sc[j], sh[j]));
      const bf16x8 val = pack8(f);
      bf16x8* dst = yp + ((int64_t)d * H + h) * W + 2 * wc;
      st_stream(dst, val);
      st_stream(dst + 1, val);
    }
  } else {
    const bf16x8* xp = plane_ptr(x, b, pl, vf);
    constexpr int U = 4;                       // independent 16-byte loads in flight per thread (see gn_silu_kernel)
    for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < vf; i += U * stride) {
      bf16x8 v[U];
#pragma unroll
      for (int k = 0; k < U; ++k)
        if (i + k * stride < vf) v[k] = ld_stream(xp + i + k * stride);
#pragma unroll
      for (int k = 0; k < U; ++k) {
        const int64_t ii = i + k * stride;
        if (ii >= vf) break;
        float f[8];
        unpack8(v[k], f);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = silu_half(fmaf(f[j], sc[j], sh[j]));
        st_stream(yp + ii, pack8(f));
      }
    }
  }
}

// ---- 2x2x2 average pooling (+ stats of the output) ---------------------------------------------
// (F32: fp32 channel-planar, statistics of the fp32 values)
template <bool F32 = false>
__global__ void __launch_bounds__(kEwThreads)
avgpool2_kernel(VdmTensor x, VdmTensor y, int planes, int D, int H, int W, double* __restrict__ stats,
                int stats_channels, int stats_c0) {
  using T = typename Unit<F32>::T;
  constexpr int L = Unit<F32>::L;
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const int Do = D >> 1, Ho = H >> 1, Wo = W >> 1;
  const int64_t vin = (int64_t)D * H * W, vout = (int64_t)Do * Ho * Wo;
  const T* xp = plane_ptr<T>(x, b, pl, vin);
  T* yp = plane_ptr_mut<T>(y, b, pl, vout);
  float sum[L] = {}, sq[L] = {};
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < vout; i += (int64_t)gridDim.x * kEwThreads) {
    unsigned v = (unsigned)i;
    const int wo = (int)(v % (unsigned)Wo); v /= (unsigned)Wo;
    const int ho = (int)(v % (unsigned)Ho);
    const int dz = (int)(v / (unsigned)Ho);
    float acc[L] = {};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int d = 2 * dz + (k >> 2), h = 2 * ho + ((k >> 1) & 1), w = 2 * wo + (k & 1);
      float f[L];
      unpack_unit(xp[((int64_t)d * H + h) * W + w], f);
#pragma unroll
      for (int j = 0; j < L; ++j) acc[j] += f[j];
    }
#pragma unroll
    for (int j = 0; j < L; ++j) acc[j] *= 0.125f;
    T packed;
    pack_unit(acc, packed);
    yp[i] = packed;
    if (stats) {
      float r[L];
      unpack_unit(packed, r);  // statistics of the stored (rounded) tensor
#pragma unroll
      for (int j = 0; j < L; ++j) {
        sum[j] += r[j];
        sq[j] += r[j] * r[j];
      }
    }
  }
  if (stats) block_flush_stats<L>(sum, sq, stats + ((int64_t)b * stats_channels + stats_c0 + pl * L) * 2);
}

// ---- nearest x2 up-sampling into a plane window of y (+ stats of the output) -------------------
// (D, H, W) is the FINE grid.  One thread per FINE voxel: fully coalesced 16-byte stores (the 8x repeated
// coarse reads hit L1/L2).  r01f: the one-thread-per-coarse-voxel version (8 scattered stores per thread)
// ran at ~1.2 TB/s.
// (F32: fp32 channel-planar)
template <bool F32 = false>
__global__ void __launch_bounds__(kEwThreads)
upsample2_kernel(VdmTensor coarse, VdmTensor y, int planes, int D, int H, int W, double* __restrict__ stats,
                 int stats_channels, int stats_c0) {
  using T = typename Unit<F32>::T;
  constexpr int L = Unit<F32>::L;
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const int Hc = H >> 1, Wc = W >> 1;
  const int64_t vc = (int64_t)(D >> 1) * Hc * Wc, vf = (int64_t)D * H * W;
  const T* cp = plane_ptr<T>(coarse, b, pl, vc);
  T* yp = plane_ptr_mut<T>(y, b, pl, vf);
  float sum[L] = {}, sq[L] = {};
  // one thread per (fine d, fine h, COARSE w): one 16-byte read, two adjacent 16-byte stores (32 contiguous bytes)
  const int64_t vh = vf >> 1;
  const bool big = vf * planes > ((int64_t)4 << 20);   // > 64 MB per sample: written once, read later from HBM anyway
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < vh; i += (int64_t)gridDim.x * kEwThreads) {
    unsigned v = (unsigned)i;
    const int wc = (int)(v % (unsigned)Wc); v /= (unsigned)Wc;
    const int h = (int)(v % (unsigned)H);
    const int d = (int)(v / (unsigned)H);
    const T val = cp[((int64_t)(d >> 1) * Hc + (h >> 1)) * Wc + wc];
    T* dst = yp + ((int64_t)d * H + h) * W + 2 * wc;
    if (big) { st_stream(dst, val); st_stream(dst + 1, val); }
    else { dst[0] = val; dst[1] = val; }
    if (stats) {
      float r[L];
      unpack_unit(val, r);
#pragma unroll
      for (int j = 0; j < L; ++j) {
        sum[j] += 2.f * r[j];
        sq[j] += 2.f * r[j] * r[j];
      }
    }
  }
  if (stats) block_flush_stats<L>(sum, sq, stats + ((int64_t)b * stats_channels + stats_c0 + pl * L) * 2);
}

// ---- periodic one-voxel halo (circular convolutions) ---------------------------------------------------
// One thread per PADDED voxel: coalesced 16-byte stores, reads coalesced except at the wrapped faces.
__global__ void __launch_bounds__(kEwThreads)
pad_circular_kernel(VdmTensor x, VdmTensor y, int planes, int D, int H, int W) {
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const int Dp = D + 2, Hp = H + 2, Wp = W + 2;
  const int64_t vin = (int64_t)D * H * W, vout = (int64_t)Dp * Hp * Wp;
  const bf16x8* xp = plane_ptr(x, b, pl, vin);
  bf16x8* yp = plane_ptr_mut(y, b, pl, vout);
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < vout; i += (int64_t)gridDim.x * kEwThreads) {
    unsigned v = (unsigned)i;
    const int wp = (int)(v % (unsigned)Wp); v /= (unsigned)Wp;
    const int hp = (int)(v % (unsigned)Hp);
    const int dp = (int)(v / (unsigned)Hp);
    const int d = dp == 0 ? D - 1 : (dp == Dp - 1 ? 0 : dp - 1);
    const int h = hp == 0 ? H - 1 : (hp == Hp - 1 ? 0 : hp - 1);
    const int w = wp == 0 ? W - 1 : (wp == Wp - 1 ? 0 : wp - 1);
    yp[i] = xp[((int64_t)d * H + h) * W + w];
  }
}

}  // namespace vdm

using namespace vdm;

extern "C" int vdm_pad_circular(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                                int channels, void* stream) {
  VDM_CHECK_ARG(view_ok<8>(x, channels) && view_ok<8>(y, channels) && batch >= 1, "vdm_pad_circular: bad argument");
  VDM_CHECK_PLANES(8, batch, channels, "vdm_pad_circular");
  VDM_CHECK_ARG(depth >= 1 && height >= 1 && width >= 1 && (int64_t)(depth + 2) * (height + 2) * (width + 2) < ((int64_t)1 << 31),
                "vdm_pad_circular: bad grid (%d,%d,%d)", depth, height, width);
  const int planes = channels / 8;
  const int64_t vout = (int64_t)(depth + 2) * (height + 2) * (width + 2);
  pad_circular_kernel<<<ew_grid(vout, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(*x, *y, planes, depth, height, width);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_channel_stats(const VdmTensor* x, int batch, int64_t voxels, int channels, double* stats,
                                 int stats_channels, int stats_c0, void* stream) {
  VDM_CHECK_ARG(view_ok<8>(x, channels) && stats && batch >= 1 && voxels >= 1, "vdm_channel_stats: bad argument");
  VDM_CHECK_PLANES(8, batch, channels, "vdm_channel_stats");
  if (stats_channels <= 0) stats_channels = channels;
  const int planes = channels / 8;
  channel_stats_kernel<<<ew_grid(voxels, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
      *x, planes, voxels, stats, stats_channels, stats_c0);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

// bf16 (vdm_gn_silu, vdm_gn_silu_step) and fp32 (vdm_gn_silu_f32, no dropout) GroupNorm + SiLU.
template <bool F32>
static int gn_silu_launch(const char* who, const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels,
                          int groups, const double* stats, const float* gamma, const float* beta, float eps,
                          float dropout_p, uint64_t seed, const int32_t* seed_step, uint32_t layer_tag, void* stream) {
  constexpr int L = Unit<F32>::L;
  if (const int rc = check_gn<L>(who, x, y, batch, voxels, channels, groups, stats, gamma, beta, dropout_p)) return rc;
  const int planes = channels / L;
  const dim3 grid = ew_grid(voxels, batch * planes);
  constexpr int kElemBytes = 16 / L;
  if ((int64_t)batch * channels * voxels * kElemBytes > (int64_t)96 << 20)
    gn_silu_kernel<true, F32><<<grid, kEwThreads, 0, (cudaStream_t)stream>>>(
        *x, *y, planes, voxels, groups, stats, gamma, beta, eps, dropout_p, seed, seed_step, layer_tag);
  else
    gn_silu_kernel<false, F32><<<grid, kEwThreads, 0, (cudaStream_t)stream>>>(
        *x, *y, planes, voxels, groups, stats, gamma, beta, eps, dropout_p, seed, seed_step, layer_tag);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_gn_silu_step(const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels,
                                int groups, const double* stats, const float* gamma, const float* beta, float eps,
                                float dropout_p, uint64_t seed, const int32_t* seed_step, uint32_t layer_tag, void* stream) {
  return gn_silu_launch<false>("vdm_gn_silu", x, y, batch, voxels, channels, groups, stats, gamma, beta, eps, dropout_p,
                               seed, seed_step, layer_tag, stream);
}

extern "C" int vdm_gn_silu(const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels, int groups,
                           const double* stats, const float* gamma, const float* beta, float eps, float dropout_p,
                           uint64_t seed, uint32_t layer_tag, void* stream) {
  return gn_silu_launch<false>("vdm_gn_silu", x, y, batch, voxels, channels, groups, stats, gamma, beta, eps, dropout_p,
                               seed, nullptr, layer_tag, stream);
}

extern "C" int vdm_gn_silu_f32(const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels, int groups,
                               const double* stats, const float* gamma, const float* beta, float eps, void* stream) {
  return gn_silu_launch<true>("vdm_gn_silu_f32", x, y, batch, voxels, channels, groups, stats, gamma, beta, eps, 0.f, 0,
                              nullptr, 0, stream);
}

extern "C" int vdm_gn_coef(const double* stats, int batch, int channels, int groups, int64_t voxels, const float* gamma,
                           const float* beta, float eps, float* coef, void* stream) {
  VDM_CHECK_ARG(stats && gamma && beta && coef && batch >= 1 && channels >= 1 && voxels >= 1, "vdm_gn_coef: bad argument");
  VDM_CHECK_ARG(groups >= 1 && channels % groups == 0, "vdm_gn_coef: %d channels not divisible into %d groups", channels, groups);
  const int n = batch * channels;
  gn_coef_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(stats, batch, channels, groups, (double)voxels, gamma, beta, eps,
                                                                    reinterpret_cast<float2*>(coef));
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_gn_silu_view(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                                int channels, int c_off, int channels_total, int groups, const double* stats,
                                const float* gamma, const float* beta, float eps, int upsample, void* stream) {
  VDM_CHECK_ARG(view_ok<8>(x, channels) && view_ok<8>(y, channels) && stats && gamma && beta, "vdm_gn_silu_view: bad tensor argument");
  VDM_CHECK_ARG(batch >= 1 && depth >= 1 && height >= 1 && width >= 1, "vdm_gn_silu_view: bad shape");
  VDM_CHECK_PLANES(8, batch, channels, "vdm_gn_silu_view");
  VDM_CHECK_ARG(c_off >= 0 && c_off % 8 == 0 && c_off + channels <= channels_total,
                "vdm_gn_silu_view: channel window [%d, %d) outside the %d-channel norm (c_off must be a multiple of 8)", c_off,
                c_off + channels, channels_total);
  VDM_CHECK_ARG(groups >= 1 && channels_total % groups == 0, "vdm_gn_silu_view: %d channels not divisible into %d groups",
                channels_total, groups);
  if (const int rc = check_grid("vdm_gn_silu_view", "fine grid", depth, height, width, upsample != 0)) return rc;
  const int64_t vf = (int64_t)depth * height * width;
  const int planes = channels / 8;
  if (upsample == 1) {
    gn_silu_view_kernel<true><<<ew_grid(vf / 2, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
        *x, *y, planes, c_off, channels_total, groups, depth, height, width, stats, gamma, beta, eps, (double)vf);
  } else if (upsample == 2) {
    // x AND y on the half-resolution grid; the statistics are those of the (depth, height, width) concat the channels
    // belong to (sums over the up-sampled tensor = 8x the coarse sums): the polyphase up-conv reads this tensor
    gn_silu_view_kernel<false><<<ew_grid(vf / 8, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
        *x, *y, planes, c_off, channels_total, groups, depth / 2, height / 2, width / 2, stats, gamma, beta, eps, (double)vf);
  } else {
    gn_silu_view_kernel<false><<<ew_grid(vf, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
        *x, *y, planes, c_off, channels_total, groups, depth, height, width, stats, gamma, beta, eps, (double)vf);
  }
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

// 2x2x2 average pooling of a bf16 (vdm_avgpool2) or fp32 (vdm_avgpool2_f32) planar tensor.
template <bool F32>
static int avgpool2_launch(const char* who, const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height,
                           int width, int channels, double* stats, int stats_channels, int stats_c0, void* stream) {
  constexpr int L = Unit<F32>::L;
  VDM_CHECK_ARG(view_ok<L>(x, channels) && view_ok<L>(y, channels) && batch >= 1, "%s: bad argument", who);
  VDM_CHECK_PLANES(L, batch, channels, who);
  if (const int rc = check_grid(who, "grid", depth, height, width, true)) return rc;
  if (stats_channels <= 0) stats_channels = channels;
  const int planes = channels / L;
  const int64_t vout = (int64_t)(depth / 2) * (height / 2) * (width / 2);
  avgpool2_kernel<F32><<<ew_grid(vout, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
      *x, *y, planes, depth, height, width, stats, stats_channels, stats_c0);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_avgpool2(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                            int channels, double* stats, int stats_channels, int stats_c0, void* stream) {
  return avgpool2_launch<false>("vdm_avgpool2", x, y, batch, depth, height, width, channels, stats, stats_channels,
                                stats_c0, stream);
}

extern "C" int vdm_avgpool2_f32(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                                int channels, double* stats, int stats_channels, int stats_c0, void* stream) {
  return avgpool2_launch<true>("vdm_avgpool2_f32", x, y, batch, depth, height, width, channels, stats, stats_channels,
                               stats_c0, stream);
}

// Nearest x2 up-sampling of a bf16 (vdm_upsample2) or fp32 (vdm_upsample2_f32) planar tensor; (depth, height, width) is
// the fine grid.
template <bool F32>
static int upsample2_launch(const char* who, const VdmTensor* coarse, const VdmTensor* y, int batch, int depth, int height,
                            int width, int channels, double* stats, int stats_channels, int stats_c0, void* stream) {
  constexpr int L = Unit<F32>::L;
  VDM_CHECK_ARG(view_ok<L>(coarse, channels) && view_ok<L>(y, channels) && batch >= 1, "%s: bad argument", who);
  VDM_CHECK_PLANES(L, batch, channels, who);
  if (const int rc = check_grid(who, "fine grid", depth, height, width, true)) return rc;
  if (stats_channels <= 0) stats_channels = channels;
  const int planes = channels / L;
  const int64_t vf = (int64_t)depth * height * width;
  upsample2_kernel<F32><<<ew_grid(vf / 2, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
      *coarse, *y, planes, depth, height, width, stats, stats_channels, stats_c0);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_upsample2(const VdmTensor* coarse, const VdmTensor* y, int batch, int depth, int height, int width,
                             int channels, double* stats, int stats_channels, int stats_c0, void* stream) {
  return upsample2_launch<false>("vdm_upsample2", coarse, y, batch, depth, height, width, channels, stats, stats_channels,
                                 stats_c0, stream);
}

extern "C" int vdm_upsample2_f32(const VdmTensor* coarse, const VdmTensor* y, int batch, int depth, int height, int width,
                                 int channels, double* stats, int stats_channels, int stats_c0, void* stream) {
  return upsample2_launch<true>("vdm_upsample2_f32", coarse, y, batch, depth, height, width, channels, stats,
                                stats_channels, stats_c0, stream);
}
