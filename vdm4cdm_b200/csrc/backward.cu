// Backward of the fused elementwise passes (HBM-bound, channel-planar bf16, 16-byte accesses).
//
// Stand in for autograd's native_group_norm_backward / silu_backward / dropout-mask multiply /
// avg_pool3d_backward / upsample_nearest3d_backward launches of LightVDM / LightSFM training_step
// (trainVDM3D128_c_c_from_field_name_thick_lowbatch.py:128-160 drives them through Lightning).
//
// GroupNorm + SiLU (+ dropout) backward, y = keep/(1-p) * silu(u), u = gamma*xhat + beta:
//   du      = dy * keep/(1-p) * silu'(u)                     silu'(u) = s*(1 + u*(1 - s)), s = sigmoid(u)
//   pass 1  : per (sample, channel) S1 = sum_v du, S2 = sum_v du*xhat   (dbeta, dgamma = sums over samples)
//   pass 2  : dx = rstd*(gamma*du - m1 - xhat*m2) [+ add],   m1 = mean_g(gamma*du), m2 = mean_g(gamma*du*xhat)
// The keep-mask is regenerated from (seed, layer_tag, chunk), never stored.  Algorithmic traffic:
// pass 1 reads 4 B/element, pass 2 reads 4 (+2) and writes 2 B/element.
#include "ew_common.cuh"

namespace vdm {

__device__ __forceinline__ float silu_grad(float u) {
  const float s = fast_sigmoid(u);
  return s * fmaf(u, 1.0f - s, 1.0f);
}

constexpr int kGnBwdUnroll = 2;      // chunks per loop trip of the GroupNorm backward kernels

struct GnBwdArgs {
  VdmTensor x, dy, add, dx;
  int planes;
  int64_t voxels;
  int groups;
  const double* stats;
  const float* gamma;
  const float* beta;
  float eps, dropout_p;
  uint64_t seed;
  const int32_t* seed_step;
  uint32_t layer_tag;
  double* sums;         // window of [B][sums_channels][2] at sums_c0: written by reduce, read by apply
  int sums_channels, sums_c0;
  double* out_stats;
  int out_stats_channels, out_stats_c0;
  int has_add;
};

// du = dy * keep/(1-p) * silu'(x*sc + sh) for the 8 channels of one chunk; x is returned unpacked.
__device__ __forceinline__ void chunk_du(const bf16x8& xv, const bf16x8& dyv, const float* __restrict__ sc,
                                         const float* __restrict__ sh, uint32_t keep, float keep_scale,
                                         float (&du)[8], float (&x)[8]) {
  float dy[8];
  unpack8(xv, x);
  unpack8(dyv, dy);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float m = ((keep >> j) & 1u) ? keep_scale : 0.f;
    du[j] = dy[j] * m * silu_grad(x[j] * sc[j] + sh[j]);
  }
}

// Pass 1.  Per thread: sum du and sum du*x (raw); per block: xhat = (x - mean)*rstd is linear in x, so the
// block partial of sum du*xhat is rstd*(sum du*x - mean*sum du), formed once per block before the atomics.
template <bool DROP>
__global__ void __launch_bounds__(kEwThreads, DROP ? 2 : 4)
gn_silu_bwd_reduce_kernel(const GnBwdArgs a) {
  __shared__ float s_scale[8], s_shift[8], s_mean[8], s_rstd[8];
  __shared__ float s_part[kEwThreads / 32][16];
  const int b = blockIdx.y / a.planes, pl = blockIdx.y % a.planes;
  const int C = a.planes * 8;
  plane_scale_shift(a.stats + (int64_t)b * C * 2, C, a.groups, pl, (double)a.voxels, a.gamma, a.beta, a.eps, s_scale,
                    s_shift, s_mean, s_rstd);
  __syncthreads();
  const bf16x8* xp = plane_ptr(a.x, b, pl, a.voxels);
  const bf16x8* gp = plane_ptr(a.dy, b, pl, a.voxels);
  constexpr bool drop = DROP;
  const uint32_t thresh16 = (uint32_t)(a.dropout_p * 65536.0f + 0.5f);
  const float keep_scale = drop ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
  const uint64_t chunk0 = ((uint64_t)b * a.planes + pl) * (uint64_t)a.voxels;
  const uint64_t seed = a.seed + (a.seed_step ? (uint64_t)(uint32_t)(*a.seed_step) : 0ull);
  float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s2[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const int64_t stride = (int64_t)gridDim.x * kEwThreads;
  constexpr int U = kGnBwdUnroll;                   // chunks per trip: 2 * U independent 16-byte loads in flight per thread
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < a.voxels; i += U * stride) {
    bf16x8 xs[U], gs[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t ii = i + k * stride;
      if (ii < a.voxels) { xs[k] = xp[ii]; gs[k] = gp[ii]; }
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t ii = i + k * stride;
      if (ii >= a.voxels) break;
      const uint32_t keep = drop ? dropout_keep8(chunk0 + (uint64_t)ii, a.layer_tag, seed, thresh16) : 0xffu;
      float du[8], x[8];
      chunk_du(xs[k], gs[k], s_scale, s_shift, keep, keep_scale, du, x);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s1[j] += du[j];
        s2[j] += du[j] * x[j];
      }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    s1[j] = warp_sum(s1[j]);
    s2[j] = warp_sum(s2[j]);
  }
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s_part[warp][j] = s1[j];
      s_part[warp][8 + j] = s2[j];
    }
  }
  __syncthreads();
  if (threadIdx.x < 8) {
    float t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int w = 0; w < kEwThreads / 32; ++w) {
      t1 += s_part[w][threadIdx.x];
      t2 += s_part[w][8 + threadIdx.x];
    }
    double* dst = a.sums + ((int64_t)b * a.sums_channels + a.sums_c0 + pl * 8 + threadIdx.x) * 2;
    atomicAdd(dst, (double)t1);
    atomicAdd(dst + 1, (double)(s_rstd[threadIdx.x] * (t2 - s_mean[threadIdx.x] * t1)));
  }
}

// Pass 2.  dx = rstd*(gamma*du - m1 - xhat*m2) [+ add]  ==  A*du + Bc + Cc*x with per-channel
// A = rstd*gamma, Cc = -rstd^2*m2, Bc = -rstd*m1 - Cc*mean.
template <bool DROP>
__global__ void __launch_bounds__(kEwThreads, DROP ? 2 : 3)
gn_silu_bwd_apply_kernel(const GnBwdArgs a) {
  __shared__ float s_scale[8], s_shift[8], s_mean[8], s_rstd[8], s_A[8], s_B[8], s_C[8];
  const int b = blockIdx.y / a.planes, pl = blockIdx.y % a.planes;
  const int C = a.planes * 8;
  plane_scale_shift(a.stats + (int64_t)b * C * 2, C, a.groups, pl, (double)a.voxels, a.gamma, a.beta, a.eps, s_scale,
                    s_shift, s_mean, s_rstd);
  if (threadIdx.x < 8) {
    const int c = pl * 8 + threadIdx.x;
    const int cpg = C / a.groups;
    const int g0 = (c / cpg) * cpg;
    const double* sb = a.sums + ((int64_t)b * a.sums_channels + a.sums_c0) * 2;
    double m1 = 0.0, m2 = 0.0;
    for (int k = 0; k < cpg; ++k) {
      const double gk = (double)a.gamma[g0 + k];
      m1 += gk * sb[2 * (g0 + k)];
      m2 += gk * sb[2 * (g0 + k) + 1];
    }
    const double n = (double)a.voxels * cpg;
    m1 /= n;
    m2 /= n;
    const double rstd = (double)s_rstd[threadIdx.x], mean = (double)s_mean[threadIdx.x];   // written by this thread
    const double Cc = -rstd * rstd * m2;
    s_A[threadIdx.x] = (float)(rstd * (double)a.gamma[c]);
    s_C[threadIdx.x] = (float)Cc;
    s_B[threadIdx.x] = (float)(-rstd * m1 - Cc * mean);
  }
  __syncthreads();
  float cA[8], cB[8], cC[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    cA[j] = s_A[j]; cB[j] = s_B[j]; cC[j] = s_C[j];
  }
  const bf16x8* xp = plane_ptr(a.x, b, pl, a.voxels);
  const bf16x8* gp = plane_ptr(a.dy, b, pl, a.voxels);
  const bf16x8* ap = a.has_add ? plane_ptr(a.add, b, pl, a.voxels) : nullptr;
  bf16x8* op = plane_ptr_mut(a.dx, b, pl, a.voxels);
  constexpr bool drop = DROP;
  const uint32_t thresh16 = (uint32_t)(a.dropout_p * 65536.0f + 0.5f);
  const float keep_scale = drop ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
  const uint64_t chunk0 = ((uint64_t)b * a.planes + pl) * (uint64_t)a.voxels;
  const uint64_t seed = a.seed + (a.seed_step ? (uint64_t)(uint32_t)(*a.seed_step) : 0ull);
  float sum[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const int64_t stride = (int64_t)gridDim.x * kEwThreads;
  constexpr int U = kGnBwdUnroll;
  const bool stream_out = a.voxels * a.planes > ((int64_t)4 << 20);
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < a.voxels; i += U * stride) {
    bf16x8 xs[U], gs[U], rs[U];
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t ii = i + k * stride;
      if (ii < a.voxels) {
        xs[k] = xp[ii]; gs[k] = gp[ii];
        if (ap) rs[k] = ap[ii];
      }
    }
#pragma unroll
    for (int k = 0; k < U; ++k) {
      const int64_t ii = i + k * stride;
      if (ii >= a.voxels) break;
      const uint32_t keep = drop ? dropout_keep8(chunk0 + (uint64_t)ii, a.layer_tag, seed, thresh16) : 0xffu;
      float du[8], x[8], o[8];
      chunk_du(xs[k], gs[k], s_scale, s_shift, keep, keep_scale, du, x);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = cA[j] * du[j] + cB[j] + cC[j] * x[j];
      if (ap) {
        float r[8];
        unpack8(rs[k], r);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] += r[j];
      }
      const bf16x8 packed = pack8(o);
      if (stream_out) st_stream(op + ii, packed);
      else op[ii] = packed;
      if (a.out_stats) {
        float r[8];
        unpack8(packed, r);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          sum[j] += r[j];
          sq[j] += r[j] * r[j];
        }
      }
    }
  }
  if (a.out_stats)
    block_flush_stats(sum, sq, a.out_stats + ((int64_t)b * a.out_stats_channels + a.out_stats_c0 + pl * 8) * 2);
}

// ---- avg-pool backward: fine dx = [dx +] dy(coarse)/8 -----------------------------------------------
// One thread per FINE voxel (coalesced read-modify-write; the coarse gradient is re-read through L1/L2).
__global__ void __launch_bounds__(kEwThreads)
avgpool2_bwd_kernel(VdmTensor dy, VdmTensor dx, int planes, int D, int H, int W, int accumulate,
                    double* __restrict__ stats, int stats_channels, int stats_c0) {
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const int Hc = H >> 1, Wc = W >> 1;
  const int64_t vc = (int64_t)(D >> 1) * Hc * Wc, vf = (int64_t)D * H * W;
  const bf16x8* gp = plane_ptr(dy, b, pl, vc);
  bf16x8* op = plane_ptr_mut(dx, b, pl, vf);
  float sum[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < vf; i += (int64_t)gridDim.x * kEwThreads) {
    unsigned v = (unsigned)i;                       // a plane has < 2^31 voxels (checked on the host): 32-bit divisions
    const int w = (int)(v % (unsigned)W); v /= (unsigned)W;
    const int h = (int)(v % (unsigned)H);
    const int d = (int)(v / (unsigned)H);
    float g[8], o[8];
    unpack8(gp[((int64_t)(d >> 1) * Hc + (h >> 1)) * Wc + (w >> 1)], g);
    if (accumulate) {
      unpack8(op[i], o);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] += 0.125f * g[j];
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = 0.125f * g[j];
    }
    const bf16x8 packed = pack8(o);
    op[i] = packed;
    if (stats) {
      float r[8];
      unpack8(packed, r);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        sum[j] += r[j];
        sq[j] += r[j] * r[j];
      }
    }
  }
  if (stats) block_flush_stats(sum, sq, stats + ((int64_t)b * stats_channels + stats_c0 + pl * 8) * 2);
}

// ---- nearest-upsample backward: coarse = sum of the 8 fine gradients ----------------------------------
__global__ void __launch_bounds__(kEwThreads)
upsample2_bwd_kernel(VdmTensor dy, VdmTensor dc, int planes, int D, int H, int W, double* __restrict__ stats,
                     int stats_channels, int stats_c0) {
  const int b = blockIdx.y / planes, pl = blockIdx.y % planes;
  const int Do = D >> 1, Ho = H >> 1, Wo = W >> 1;
  const int64_t vin = (int64_t)D * H * W, vout = (int64_t)Do * Ho * Wo;
  const bf16x8* gp = plane_ptr(dy, b, pl, vin);
  bf16x8* op = plane_ptr_mut(dc, b, pl, vout);
  float sum[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sq[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t i = (int64_t)blockIdx.x * kEwThreads + threadIdx.x; i < vout; i += (int64_t)gridDim.x * kEwThreads) {
    unsigned v = (unsigned)i;
    const int wo = (int)(v % (unsigned)Wo); v /= (unsigned)Wo;
    const int ho = (int)(v % (unsigned)Ho);
    const int dz = (int)(v / (unsigned)Ho);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int d = 2 * dz + (k >> 2), h = 2 * ho + ((k >> 1) & 1), w = 2 * wo + (k & 1);
      float f[8];
      unpack8(gp[((int64_t)d * H + h) * W + w], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += f[j];
    }
    const bf16x8 packed = pack8(acc);
    op[i] = packed;
    if (stats) {
      float r[8];
      unpack8(packed, r);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        sum[j] += r[j];
        sq[j] += r[j] * r[j];
      }
    }
  }
  if (stats) block_flush_stats(sum, sq, stats + ((int64_t)b * stats_channels + stats_c0 + pl * 8) * 2);
}

// ---- optimizer -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ x, int64_t n, double* __restrict__ out) {
  __shared__ double s_part[8];
  double acc = 0.0;
  const int64_t n4 = n >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n4; i += (int64_t)gridDim.x * 256) {
    const float4 v = x4[i];
    acc += (double)(v.x * v.x + v.y * v.y) + (double)(v.z * v.z + v.w * v.w);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
    const float v = x[(n4 << 2) + threadIdx.x];
    acc += (double)v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += s_part[w];
    atomicAdd(out, t);
  }
}

__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
             float lr, float beta1, float beta2, float eps, float weight_decay, int step,
             const int32_t* __restrict__ step_ptr, const double* __restrict__ grad_sumsq, float max_norm, float grad_scale) {
  const float stepf = (float)(step + (step_ptr ? *step_ptr : 0));
  const float bc1 = 1.0f - powf(beta1, stepf);
  const float bc2_sqrt = sqrtf(1.0f - powf(beta2, stepf));
  float gs = grad_scale;
  if (grad_sumsq != nullptr && max_norm > 0.f) {
    const float norm = grad_scale * (float)sqrt(*grad_sumsq);
    const float coef = max_norm / (norm + 1e-6f);
    if (coef < 1.0f) gs *= coef;
  }
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const float gi = g[i] * gs;
    float pi = p[i];
    pi *= 1.0f - lr * weight_decay;
    const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

}  // namespace vdm

using namespace vdm;

static int gn_bwd_common(const char* who, const VdmTensor* x, const VdmTensor* dy, int batch, int64_t voxels, int channels,
                         int groups, const double* stats, const float* gamma, const float* beta, float dropout_p,
                         const double* sums) {
  VDM_CHECK_ARG(sums, "%s: bad tensor argument", who);
  return check_gn<8>(who, x, dy, batch, voxels, channels, groups, stats, gamma, beta, dropout_p);
}

extern "C" int vdm_gn_silu_bwd_reduce(const VdmTensor* x, const VdmTensor* dy, int batch, int64_t voxels, int channels,
                                      int groups, const double* stats, const float* gamma, const float* beta, float eps,
                                      float dropout_p, uint64_t seed, const int32_t* seed_step, uint32_t layer_tag,
                                      double* sums, int sums_channels, int sums_c0, void* stream) {
  const int rc = gn_bwd_common("vdm_gn_silu_bwd_reduce", x, dy, batch, voxels, channels, groups, stats, gamma, beta,
                               dropout_p, sums);
  if (rc != VDM_OK) return rc;
  GnBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.x = *x; a.dy = *dy; a.planes = channels / 8; a.voxels = voxels; a.groups = groups; a.stats = stats;
  a.gamma = gamma; a.beta = beta; a.eps = eps; a.dropout_p = dropout_p; a.seed = seed; a.layer_tag = layer_tag;
  a.seed_step = seed_step;
  a.sums = sums;
  a.sums_channels = sums_channels > 0 ? sums_channels : channels;
  a.sums_c0 = sums_c0;
  if (dropout_p > 0.f)
    gn_silu_bwd_reduce_kernel<true><<<ew_grid(voxels, batch * a.planes), kEwThreads, 0, (cudaStream_t)stream>>>(a);
  else
    gn_silu_bwd_reduce_kernel<false><<<ew_grid(voxels, batch * a.planes), kEwThreads, 0, (cudaStream_t)stream>>>(a);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_gn_silu_bwd_apply(const VdmTensor* x, const VdmTensor* dy, const VdmTensor* add, const VdmTensor* dx,
                                     int batch, int64_t voxels, int channels, int groups, const double* stats,
                                     const float* gamma, const float* beta, float eps, float dropout_p, uint64_t seed,
                                     const int32_t* seed_step, uint32_t layer_tag, const double* sums, int sums_channels,
                                     int sums_c0, double* out_stats, int out_stats_channels, int out_stats_c0,
                                     void* stream) {
  const int rc = gn_bwd_common("vdm_gn_silu_bwd_apply", x, dy, batch, voxels, channels, groups, stats, gamma, beta,
                               dropout_p, sums);
  if (rc != VDM_OK) return rc;
  VDM_CHECK_ARG(view_ok<8>(dx, channels) && (add == nullptr || view_ok<8>(add, channels)), "vdm_gn_silu_bwd_apply: bad dx/add view");
  GnBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.x = *x; a.dy = *dy; a.dx = *dx; a.planes = channels / 8; a.voxels = voxels; a.groups = groups; a.stats = stats;
  a.gamma = gamma; a.beta = beta; a.eps = eps; a.dropout_p = dropout_p; a.seed = seed; a.layer_tag = layer_tag;
  a.seed_step = seed_step;
  a.sums = const_cast<double*>(sums);
  a.sums_channels = sums_channels > 0 ? sums_channels : channels;
  a.sums_c0 = sums_c0;
  if (add) { a.add = *add; a.has_add = 1; }
  a.out_stats = out_stats;
  a.out_stats_channels = out_stats_channels > 0 ? out_stats_channels : channels;
  a.out_stats_c0 = out_stats_c0;
  if (dropout_p > 0.f)
    gn_silu_bwd_apply_kernel<true><<<ew_grid(voxels, batch * a.planes), kEwThreads, 0, (cudaStream_t)stream>>>(a);
  else
    gn_silu_bwd_apply_kernel<false><<<ew_grid(voxels, batch * a.planes), kEwThreads, 0, (cudaStream_t)stream>>>(a);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_avgpool2_bwd(const VdmTensor* dy, const VdmTensor* dx, int batch, int depth, int height, int width,
                                int channels, int accumulate, double* stats, int stats_channels, int stats_c0,
                                void* stream) {
  VDM_CHECK_ARG(view_ok<8>(dy, channels) && view_ok<8>(dx, channels) && batch >= 1, "vdm_avgpool2_bwd: bad argument");
  VDM_CHECK_PLANES(8, batch, channels, "vdm_avgpool2_bwd");
  if (const int rc = check_grid("vdm_avgpool2_bwd", "fine grid", depth, height, width, true)) return rc;
  if (stats_channels <= 0) stats_channels = channels;
  const int planes = channels / 8;
  const int64_t vf = (int64_t)depth * height * width;
  avgpool2_bwd_kernel<<<ew_grid(vf, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
      *dy, *dx, planes, depth, height, width, accumulate, stats, stats_channels, stats_c0);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_upsample2_bwd(const VdmTensor* dy, const VdmTensor* dcoarse, int batch, int depth, int height,
                                 int width, int channels, double* stats, int stats_channels, int stats_c0, void* stream) {
  VDM_CHECK_ARG(view_ok<8>(dy, channels) && view_ok<8>(dcoarse, channels) && batch >= 1, "vdm_upsample2_bwd: bad argument");
  VDM_CHECK_PLANES(8, batch, channels, "vdm_upsample2_bwd");
  if (const int rc = check_grid("vdm_upsample2_bwd", "fine grid", depth, height, width, true)) return rc;
  if (stats_channels <= 0) stats_channels = channels;
  const int planes = channels / 8;
  const int64_t vout = (int64_t)(depth / 2) * (height / 2) * (width / 2);
  upsample2_bwd_kernel<<<ew_grid(vout, batch * planes), kEwThreads, 0, (cudaStream_t)stream>>>(
      *dy, *dcoarse, planes, depth, height, width, stats, stats_channels, stats_c0);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_sumsq(const float* x, int64_t n, double* out, void* stream) {
  VDM_CHECK_ARG(x && out && n >= 0, "vdm_sumsq: bad argument");
  VDM_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0, "vdm_sumsq: x must be 16-byte aligned");
  if (n == 0) return VDM_OK;
  int64_t blocks = (n / 4 + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  if (blocks < 1) blocks = 1;
  sumsq_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, out);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

static int adamw_launch(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                        float beta1, float beta2, float eps, float weight_decay, int step, const int32_t* step_ptr,
                        const double* grad_sumsq, float max_norm, float grad_scale, void* stream) {
  VDM_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && n >= 0 && (step >= 1 || step_ptr), "vdm_adamw_step: bad argument");
  if (n == 0) return VDM_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  adamw_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                   eps, weight_decay, step, step_ptr, grad_sumsq, max_norm,
                                                                   grad_scale);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_adamw_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                              float beta1, float beta2, float eps, float weight_decay, int step, const double* grad_sumsq,
                              float max_norm, float grad_scale, void* stream) {
  return adamw_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, step, nullptr, grad_sumsq,
                      max_norm, grad_scale, stream);
}

extern "C" int vdm_adamw_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                                  float beta1, float beta2, float eps, float weight_decay, int step, const int32_t* step_ptr,
                                  const double* grad_sumsq, float max_norm, float grad_scale, void* stream) {
  return adamw_launch(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, step, step_ptr, grad_sumsq,
                      max_norm, grad_scale, stream);
}
