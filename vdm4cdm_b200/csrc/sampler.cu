// Fused VDM ancestral-sampler update (HBM-bound, vectorised, Philox noise in registers).
//
// Stands in for the elementwise tail of VDM.sample_zs_given_zt (mltools vdm_model.py:370-378,
// recovered in model_test.ipynb:681):  mean = alpha_s/alpha_t*(zt - c*sigma_t*pred_noise);
// z_s = mean + sigma_s*sqrt(c)*randn.  The reference issues ~6 elementwise launches plus
// torch.randn_like per step; this is one pass: 4 B (z) + 4 B (eps_hat) read, 4 B written per
// voxel, optionally + 16 B for plane 0 of the packed bf16 network input of the next step.
#include "common.cuh"

namespace vdm {

// One thread = 4 consecutive voxels (one Philox call).  coef = (w_z, w_eps, noise_scale, out_scale).
__global__ void __launch_bounds__(256)
sampler_step_kernel(const float* __restrict__ z, const float* __restrict__ eps_hat, float* __restrict__ z_out,
                    int64_t voxels, const float* __restrict__ coef, const int32_t* __restrict__ step_ptr,
                    uint64_t seed, const int32_t* __restrict__ realisation_id, int32_t draw_base,
                    const float* __restrict__ noise_in, const float* __restrict__ cond, int n_cond,
                    bf16x8* __restrict__ packed_out, int packed_planes) {
  const int b = blockIdx.y;
  const int step = step_ptr ? *step_ptr : 0;
  const float4 cf = *reinterpret_cast<const float4*>(coef + 4 * (int64_t)step);
  const uint32_t draw = (uint32_t)(draw_base + step);
  const uint32_t rid = realisation_id ? (uint32_t)realisation_id[b] : (uint32_t)b;
  const int64_t groups = (voxels + 3) >> 2;
  const float* zb = z + (int64_t)b * voxels;
  const float* eb = eps_hat + (int64_t)b * voxels;
  float* ob = z_out + (int64_t)b * voxels;
  const bool vec_ok = (voxels & 3) == 0;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups;
       g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t e0 = g << 2;
    float zi[4], ei[4], ni[4], out[4];
    if (vec_ok) {
      const float4 a = *reinterpret_cast<const float4*>(zb + e0);
      const float4 e = *reinterpret_cast<const float4*>(eb + e0);
      zi[0] = a.x; zi[1] = a.y; zi[2] = a.z; zi[3] = a.w;
      ei[0] = e.x; ei[1] = e.y; ei[2] = e.z; ei[3] = e.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool ok = e0 + i < voxels;
        zi[i] = ok ? zb[e0 + i] : 0.f;
        ei[i] = ok ? eb[e0 + i] : 0.f;
      }
    }
    if (noise_in) {
#pragma unroll
      for (int i = 0; i < 4; ++i) ni[i] = (e0 + i < voxels) ? noise_in[(int64_t)b * voxels + e0 + i] : 0.f;
    } else if (cf.z != 0.f) {
      const float4 n = philox_normal4((uint32_t)g, draw, rid, seed);
      ni[0] = n.x; ni[1] = n.y; ni[2] = n.z; ni[3] = n.w;
    } else {
      ni[0] = ni[1] = ni[2] = ni[3] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) out[i] = cf.w * (cf.x * zi[i] + cf.y * ei[i] + cf.z * ni[i]);
    if (vec_ok) {
      *reinterpret_cast<float4*>(ob + e0) = make_float4(out[0], out[1], out[2], out[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (e0 + i < voxels) ob[e0 + i] = out[i];
    }
    if (packed_out) {
      // plane 0 of the packed network input: (z, cond_1..cond_n, 0...) as 8 bf16 = one 16-byte store per voxel
      bf16x8* plane0 = packed_out + (int64_t)b * packed_planes * voxels;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int64_t v = e0 + i;
        if (v >= voxels) break;
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          f[j] = (j == 0) ? out[i] : (j <= n_cond ? cond[((int64_t)b * n_cond + (j - 1)) * voxels + v] : 0.f);
        plane0[v] = pack8(f);
      }
    }
  }
}

__global__ void __launch_bounds__(256)
philox_normal_kernel(float* __restrict__ out, int64_t voxels, uint64_t seed,
                     const int32_t* __restrict__ realisation_id, int32_t draw) {
  const int b = blockIdx.y;
  const uint32_t rid = realisation_id ? (uint32_t)realisation_id[b] : (uint32_t)b;
  const int64_t groups = (voxels + 3) >> 2;
  float* ob = out + (int64_t)b * voxels;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < groups;
       g += (int64_t)gridDim.x * blockDim.x) {
    const float4 n = philox_normal4((uint32_t)g, (uint32_t)draw, rid, seed);
    const float v[4] = {n.x, n.y, n.z, n.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if ((g << 2) + i < voxels) ob[(g << 2) + i] = v[i];
  }
}

// z fp32 + cond fp32 planes -> channel-planar bf16: plane 0 = (z, cond_1..cond_n, 0...), other planes 0.
// F32: fp32 channel-planar, the same 8 channels in planes 0 and 1.
template <bool F32 = false>
__global__ void __launch_bounds__(256)
pack_input_kernel(const float* __restrict__ z, const float* __restrict__ cond, VdmTensor out, int planes,
                  int64_t voxels, int n_cond) {
  using T = typename Unit<F32>::T;
  constexpr int L = Unit<F32>::L, P = 8 / L;       // planes holding (z, cond_1..cond_7)
  const int b = blockIdx.y;
  T* ob = reinterpret_cast<T*>(out.data) + ((int64_t)b * out.planes + out.plane0) * voxels;
  for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < voxels;
       v += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int q = 0; q < P; ++q) {
      float f[L];
#pragma unroll
      for (int i = 0; i < L; ++i) {
        const int j = q * L + i;
        f[i] = (j == 0) ? z[(int64_t)b * voxels + v]
                        : (j <= n_cond ? cond[((int64_t)b * n_cond + (j - 1)) * voxels + v] : 0.f);
      }
      T u;
      pack_unit(f, u);
      ob[(int64_t)q * voxels + v] = u;
    }
    const float zero[L] = {};
    for (int pl = P; pl < planes; ++pl) {
      T u;
      pack_unit(zero, u);
      ob[(int64_t)pl * voxels + v] = u;
    }
  }
}

static inline dim3 grid_for(int64_t work_items, int batch, int threads) {
  int64_t blocks = (work_items + threads - 1) / threads;
  const int64_t cap = (int64_t)kNumSMs * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return dim3((unsigned)blocks, (unsigned)batch);
}

}  // namespace vdm

extern "C" int vdm_sampler_step(const float* z, const float* eps_hat, float* z_out, int batch, int64_t voxels,
                                const float* coef, const int32_t* step_ptr, uint64_t seed,
                                const int32_t* realisation_id, int32_t draw_base, const float* noise_in,
                                const float* cond, int n_cond, void* packed_out, int packed_planes, void* stream) {
  VDM_CHECK_ARG(z && eps_hat && z_out && coef, "vdm_sampler_step: NULL pointer argument");
  VDM_CHECK_ARG(batch >= 1 && batch <= 65535 && voxels >= 1, "vdm_sampler_step: bad shape (%d, %lld)", batch,
                (long long)voxels);
  VDM_CHECK_ARG(voxels <= ((int64_t)1 << 34), "vdm_sampler_step: field too large for the 32-bit Philox group index");
  if (packed_out) {
    VDM_CHECK_ARG(packed_planes >= 1 && n_cond >= 0 && n_cond + 1 <= 8, "vdm_sampler_step: bad packed_planes %d / n_cond %d",
                  packed_planes, n_cond);
    VDM_CHECK_ARG(n_cond == 0 || cond, "vdm_sampler_step: cond is NULL with n_cond=%d", n_cond);
  }
  const dim3 grid = vdm::grid_for((voxels + 3) / 4, batch, 256);
  vdm::sampler_step_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      z, eps_hat, z_out, voxels, coef, step_ptr, seed, realisation_id, draw_base, noise_in, cond, n_cond,
      static_cast<vdm::bf16x8*>(packed_out), packed_planes);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_philox_normal(float* out, int batch, int64_t voxels, uint64_t seed,
                                 const int32_t* realisation_id, int32_t draw, void* stream) {
  VDM_CHECK_ARG(out && batch >= 1 && batch <= 65535 && voxels >= 1, "vdm_philox_normal: bad argument");
  const dim3 grid = vdm::grid_for((voxels + 3) / 4, batch, 256);
  vdm::philox_normal_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, voxels, seed, realisation_id, draw);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_pack_input(const float* z, const float* cond, const VdmTensor* out, int batch, int64_t voxels,
                              int n_cond, int c_pad, void* stream) {
  VDM_CHECK_ARG(z && out && out->data && batch >= 1 && batch <= 65535 && voxels >= 1, "vdm_pack_input: bad argument");
  VDM_CHECK_ARG(c_pad >= 8 && c_pad % 8 == 0 && n_cond >= 0 && n_cond + 1 <= 8 && out->plane0 >= 0 &&
                    out->planes >= out->plane0 + c_pad / 8,
                "vdm_pack_input: bad c_pad %d / n_cond %d / plane window", c_pad, n_cond);
  VDM_CHECK_ARG(n_cond == 0 || cond, "vdm_pack_input: cond is NULL with n_cond=%d", n_cond);
  const dim3 grid = vdm::grid_for(voxels, batch, 256);
  vdm::pack_input_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(z, cond, *out, c_pad / 8, voxels, n_cond);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_pack_input_f32(const float* z, const float* cond, const VdmTensor* out, int batch, int64_t voxels,
                                  int n_cond, int c_pad, void* stream) {
  VDM_CHECK_ARG(z && out && out->data && batch >= 1 && batch <= 65535 && voxels >= 1 &&
                    (reinterpret_cast<uintptr_t>(out->data) & 15) == 0, "vdm_pack_input_f32: bad argument");
  VDM_CHECK_ARG(c_pad >= 8 && c_pad % 8 == 0 && n_cond >= 0 && n_cond + 1 <= 8 && out->plane0 >= 0 &&
                    out->planes >= out->plane0 + c_pad / 4,
                "vdm_pack_input_f32: bad c_pad %d / n_cond %d / plane window", c_pad, n_cond);
  VDM_CHECK_ARG(n_cond == 0 || cond, "vdm_pack_input_f32: cond is NULL with n_cond=%d", n_cond);
  const dim3 grid = vdm::grid_for(voxels, batch, 256);
  vdm::pack_input_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(z, cond, *out, c_pad / 4, voxels, n_cond);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}
