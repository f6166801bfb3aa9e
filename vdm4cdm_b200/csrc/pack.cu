// fp32 torch Conv3d weights -> the bf16 operand layout of vdm_conv3d, forward and dgrad variants, and the fp32 (TF32-rounded)
// layout of vdm_conv3d_tf32.
//
// Stands in for the per-step host-side glue a mixed-precision PyTorch run does implicitly (autocast's
// weight casts) plus the layout change the tensor-core kernels want.  One thread per 16-byte chunk of the
// packed tensor (8 consecutive K values of one (tap, N row)); trivially HBM-bound and tiny (<= 7 MB per conv).
#include <type_traits>

#include "common.cuh"

namespace vdm {

// Chunk = bf16x8: bf16 [tap][k_pad/8][n_pad][8].  Chunk = uint4: fp32 [tap][k_pad/4][n_pad][4], every value rounded to the
// nearest TF32 number (cvt.rna: the tensor core then multiplies an exact operand whether it rounds or truncates the other).
template <typename Chunk>
__device__ __forceinline__ void pack_conv_weight_body(const float* __restrict__ w, Chunk* __restrict__ out, int c_out, int c_in,
                                                      int k3, int transpose_flip, int ci0, int n_ci, int k_pad, int n_pad) {
  constexpr bool F32 = sizeof(Chunk) == 16 && !std::is_same<Chunk, bf16x8>::value;
  constexpr int L = F32 ? 4 : 8;       // K values per 16-byte chunk
  const int64_t total = (int64_t)k3 * (k_pad / L) * n_pad;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
    int64_t v = i;
    const int n = (int)(v % n_pad); v /= n_pad;
    const int kg = (int)(v % (k_pad / L));
    const int tap = (int)(v / (k_pad / L));
    float f[L];
#pragma unroll
    for (int j = 0; j < L; ++j) {
      const int k = kg * L + j;
      float val = 0.f;
      if (!transpose_flip) {
        // K = conv input channel, N = conv output channel
        if (k < c_in && n < c_out) val = w[((int64_t)n * c_in + k) * k3 + tap];
      } else {
        // dgrad: K = conv output channel, N = conv input channel ci0 + n, taps mirrored
        if (k < c_out && n < n_ci) val = w[((int64_t)k * c_in + ci0 + n) * k3 + (k3 - 1 - tap)];
      }
      f[j] = val;
    }
    if constexpr (F32) {
      uint32_t r[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r[j]) : "f"(f[j]));
      out[i] = make_uint4(r[0], r[1], r[2], r[3]);
    } else {
      out[i] = pack8(f);
    }
  }
}

template <typename Chunk>
__global__ void __launch_bounds__(256)
pack_conv_weight_kernel(const float* __restrict__ w, Chunk* __restrict__ out, int c_out, int c_in, int k3,
                        int transpose_flip, int ci0, int n_ci, int k_pad, int n_pad) {
  pack_conv_weight_body(w, out, c_out, c_in, k3, transpose_flip, ci0, n_ci, k_pad, n_pad);
}

// Every filter of a network in ONE launch (blockIdx.y = job): a training step re-packs ~56 filters (forward + dgrad
// variants) after each optimizer update, and as separate launches they cost 0.24 ms of launch gaps per 17 ms step.
__global__ void __launch_bounds__(256)
pack_conv_weight_batched_kernel(const VdmPackJob* __restrict__ jobs) {
  const VdmPackJob j = jobs[blockIdx.y];
  pack_conv_weight_body(j.w, static_cast<bf16x8*>(j.packed), j.c_out, j.c_in, j.k3, j.transpose_flip, j.ci0, j.n_ci, j.c_in_pad,
                        j.c_out_pad);
}

}  // namespace vdm

using namespace vdm;

extern "C" int vdm_pack_conv_weight(const float* w, void* packed, int c_out, int c_in, int kernel, int transpose_flip,
                                    int ci0, int n_ci, int c_in_pad, int c_out_pad, void* stream) {
  VDM_CHECK_ARG(w && packed && c_out >= 1 && c_in >= 1 && kernel >= 1 && kernel <= 3, "vdm_pack_conv_weight: bad argument");
  VDM_CHECK_ARG(c_in_pad % 16 == 0 && c_out_pad % 16 == 0 && c_in_pad >= 16 && c_out_pad >= 16,
                "vdm_pack_conv_weight: padded sizes (%d, %d) must be multiples of 16", c_in_pad, c_out_pad);
  VDM_CHECK_ARG((reinterpret_cast<uintptr_t>(packed) & 15) == 0, "vdm_pack_conv_weight: packed must be 16-byte aligned");
  if (!transpose_flip) {
    VDM_CHECK_ARG(c_in <= c_in_pad && c_out <= c_out_pad, "vdm_pack_conv_weight: padded sizes smaller than the filter");
  } else {
    VDM_CHECK_ARG(ci0 >= 0 && n_ci >= 1 && ci0 + n_ci <= c_in && c_out <= c_in_pad && n_ci <= c_out_pad,
                  "vdm_pack_conv_weight: dgrad slice [%d, %d) of %d input channels does not fit", ci0, ci0 + n_ci, c_in);
  }
  const int k3 = kernel * kernel * kernel;
  const int64_t total = (int64_t)k3 * (c_in_pad / 8) * c_out_pad;
  int64_t blocks = (total + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  pack_conv_weight_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      w, static_cast<bf16x8*>(packed), c_out, c_in, k3, transpose_flip, ci0, n_ci, c_in_pad, c_out_pad);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_pack_conv_weight_f32(const float* w, void* packed, int c_out, int c_in, int kernel, int c_in_pad,
                                        int c_out_pad, void* stream) {
  VDM_CHECK_ARG(w && packed && c_out >= 1 && c_in >= 1 && kernel >= 1 && kernel <= 3, "vdm_pack_conv_weight_f32: bad argument");
  VDM_CHECK_ARG(c_in_pad % 8 == 0 && c_out_pad % 16 == 0 && c_in_pad >= 8 && c_out_pad >= 16,
                "vdm_pack_conv_weight_f32: padded sizes (%d, %d) must be multiples of 8 and 16", c_in_pad, c_out_pad);
  VDM_CHECK_ARG(c_in <= c_in_pad && c_out <= c_out_pad, "vdm_pack_conv_weight_f32: padded sizes smaller than the filter");
  VDM_CHECK_ARG((reinterpret_cast<uintptr_t>(packed) & 15) == 0, "vdm_pack_conv_weight_f32: packed must be 16-byte aligned");
  const int k3 = kernel * kernel * kernel;
  const int64_t total = (int64_t)k3 * (c_in_pad / 4) * c_out_pad;
  int64_t blocks = (total + 255) / 256;
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  pack_conv_weight_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(w, static_cast<uint4*>(packed), c_out, c_in, k3, 0, 0,
                                                                              c_out, c_in_pad, c_out_pad);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

extern "C" int vdm_pack_conv_weight_batched(const VdmPackJob* jobs_device, int n_jobs, void* stream) {
  VDM_CHECK_ARG(jobs_device && n_jobs >= 1 && n_jobs <= 65535, "vdm_pack_conv_weight_batched: bad argument");
  // (the jobs live in device memory: their fields were validated by the host code that built the table)
  dim3 grid(64, (unsigned)n_jobs);
  pack_conv_weight_batched_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(jobs_device);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}
