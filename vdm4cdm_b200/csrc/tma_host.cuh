// Host-side helpers of the TMA-fed launchers (conv3d.cu, wgrad.cu): the driver queries, the tensor map of a
// channel-planar operand and a kernel launch with the large dynamic shared-memory opt-in.
#pragma once

#include <cudaTypedefs.h>

#include "common.cuh"

namespace vdm {

// cuTensorMapEncodeTiled from the driver (nullptr when the driver does not provide it), looked up once.
inline PFN_cuTensorMapEncodeTiled_v12000 encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = []() -> PFN_cuTensorMapEncodeTiled_v12000 {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  }();
  return fn;
}

// SMs of the current device, queried once (kNumSMs if the query fails).
inline int num_sms() {
  static int n = []() {
    int dev = 0, v = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return kNumSMs;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) return kNumSMs;
    return v;
  }();
  return n;
}

struct PlanarBox {
  uint32_t w, h, d, planes;   // voxels along w, h, d and 8-channel planes
};

// 4-D tensor map over a bf16 channel-planar tensor [batch_planes][D + 2 pad][H + 2 pad][W + 2 pad][8] that exposes the
// W x H x D window starting at `base`: dimensions (W*8 channels-in-plane, H, D, batch_planes), positions outside it read
// zeros.  `pad` only sets the strides (a periodic halo around every plane the map does not show).  Failure is reported
// as "<who>: cuTensorMapEncodeTiled(<operand>) failed with <CUresult>" and VDM_E_DRIVER.
inline int encode_planar(CUtensorMap* map, const void* base, uint64_t W, uint64_t H, uint64_t D, uint64_t batch_planes,
                         int pad, PlanarBox box, const char* who, const char* operand) {
  const uint64_t Wp = W + 2 * pad, Hp = H + 2 * pad, Dp = D + 2 * pad;
  cuuint64_t gdim[4] = {W * 8, H, D, batch_planes};
  cuuint64_t gstr[3] = {Wp * 16, Hp * Wp * 16, Dp * Hp * Wp * 16};
  cuuint32_t bdim[4] = {box.w * 8, box.h, box.d, box.planes};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult r = encode_fn()(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, bdim, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                 CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("%s: cuTensorMapEncodeTiled(%s) failed with %d", who, operand, (int)r);
    return VDM_E_DRIVER;
  }
  return VDM_OK;
}

// Launches `Kernel` with `smem_bytes` of dynamic shared memory; the first launch of each kernel raises its limit to the
// 227 KB an sm_100 block can have.
template <auto Kernel, typename... Args>
int launch_kernel(int grid, int threads, size_t smem_bytes, cudaStream_t stream, const Args&... args) {
  static bool configured = false;
  if (!configured) {
    VDM_CHECK_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    configured = true;
  }
  Kernel<<<grid, threads, smem_bytes, stream>>>(args...);
  VDM_CHECK_LAUNCH();
  return VDM_OK;
}

}  // namespace vdm
