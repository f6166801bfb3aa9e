// Shared helpers for the vdm4cdm_b200 CUDA sources (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/vdm4cdm_b200.h"

namespace vdm {

void set_error(const char* fmt, ...);

#define VDM_CHECK_ARG(cond, ...)                \
  do {                                          \
    if (!(cond)) {                              \
      ::vdm::set_error(__VA_ARGS__);            \
      return VDM_E_BADARG;                      \
    }                                           \
  } while (0)

#define VDM_CHECK_CUDA(expr)                                                            \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      ::vdm::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                       __LINE__);                                                       \
      return VDM_E_CUDA;                                                                \
    }                                                                                   \
  } while (0)

#define VDM_CHECK_LAUNCH() VDM_CHECK_CUDA(cudaGetLastError())

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

static inline int ceil_div(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// ---------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller: the noise definition of oracle/philox_ref.py.
// ---------------------------------------------------------------------------------------
constexpr uint32_t kPhiloxM0 = 0xD2511F53u;
constexpr uint32_t kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u;
constexpr uint32_t kPhiloxW1 = 0xBB67AE85u;
constexpr uint32_t kStreamTagNoise = 0x56444D34u;    // 'VDM4'
constexpr uint32_t kStreamTagDropout = 0x44524F50u;  // 'DROP'

template <int ROUNDS>
__device__ __forceinline__ uint4 philox4x32(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    const uint32_t hi0 = __umulhi(kPhiloxM0, c.x), lo0 = kPhiloxM0 * c.x;
    const uint32_t hi1 = __umulhi(kPhiloxM1, c.z), lo1 = kPhiloxM1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += kPhiloxW0;
    k.y += kPhiloxW1;
  }
  return c;
}
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) { return philox4x32<10>(c, k); }
// Seven rounds (Random123's "Philox4x32-7": the smallest round count that passes BigCrush) for the dropout masks, which are
// regenerated three times per layer and step (forward, backward reduce, backward apply) and made those kernels ALU-bound
// (R4z: 3.0 TB/s with dropout vs 4.8 without).  The sampler noise keeps the ten-round generator of oracle/philox_ref.py.
__device__ __forceinline__ uint4 philox4x32_7(uint4 c, uint2 k) { return philox4x32<7>(c, k); }

__device__ __forceinline__ float philox_unit(uint32_t w) {
  return ((float)(w >> 8) + 0.5f) * 5.9604644775390625e-08f;  // 2^-24
}

// Four N(0,1) values for element group g (elements 4g..4g+3) of (realisation, draw).
__device__ __forceinline__ float4 philox_normal4(uint32_t group, uint32_t draw, uint32_t realisation,
                                                 uint64_t seed) {
  const uint4 w = philox4x32_10(make_uint4(group, draw, realisation, kStreamTagNoise),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float u0 = philox_unit(w.x), u1 = philox_unit(w.y), u2 = philox_unit(w.z), u3 = philox_unit(w.w);
  const float ra = sqrtf(-2.0f * logf(u0));
  const float rb = sqrtf(-2.0f * logf(u2));
  float s1, c1, s3, c3;
  sincosf(6.283185307179586f * u1, &s1, &c1);
  sincosf(6.283185307179586f * u3, &s3, &c3);
  return make_float4(ra * s1, ra * c1, rb * s3, rb * c3);
}

// ---------------------------------------------------------------------------------------
// bf16 <-> fp32 vector helpers (8 bf16 = one 16-byte access)
// ---------------------------------------------------------------------------------------
// One uint4 member so that every copy / load / store of a chunk is a single 128-bit access.  (r01h: with
// four __nv_bfloat162 members nvcc emitted four 32-bit STG/LDG per chunk -- 4x the L2 sector requests in the
// conv epilogue and in every elementwise kernel.)
struct alignas(16) bf16x8 {
  uint4 u;
};

// streaming (evict-first) 128-bit accesses for tensors that are read or written exactly once per kernel
__device__ __forceinline__ bf16x8 ld_stream(const bf16x8* p) {
  bf16x8 r;
  r.u = __ldcs(reinterpret_cast<const uint4*>(p));
  return r;
}
__device__ __forceinline__ void st_stream(bf16x8* p, const bf16x8& v) { __stcs(reinterpret_cast<uint4*>(p), v.u); }
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(float4* p, const float4& v) { __stcs(p, v); }

__device__ __forceinline__ float2 bf16pair_to_float2(uint32_t w) {
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}

__device__ __forceinline__ void unpack8(const bf16x8& p, float (&f)[8]) {
  const uint32_t w[4] = {p.u.x, p.u.y, p.u.z, p.u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = bf16pair_to_float2(w[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

__device__ __forceinline__ uint32_t float2_to_bf16pair(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

__device__ __forceinline__ bf16x8 pack8(const float (&f)[8]) {
  bf16x8 p;
  p.u = make_uint4(float2_to_bf16pair(f[0], f[1]), float2_to_bf16pair(f[2], f[3]), float2_to_bf16pair(f[4], f[5]),
                   float2_to_bf16pair(f[6], f[7]));
  return p;
}

// The 16-byte unit of a channel-planar tensor as fp32 lanes: 8 bf16 channels, or 4 fp32 channels (the fp32 channel-planar
// layout [B][C/4][D][H][W][4] of the TF32 inference mode).  Unit<F32>::T is the type, L its channel count.
template <bool F32> struct Unit { using T = bf16x8; static constexpr int L = 8; };
template <> struct Unit<true> { using T = float4; static constexpr int L = 4; };
__device__ __forceinline__ void unpack_unit(const bf16x8& p, float (&f)[8]) { unpack8(p, f); }
__device__ __forceinline__ void unpack_unit(const float4& p, float (&f)[4]) { f[0] = p.x; f[1] = p.y; f[2] = p.z; f[3] = p.w; }
__device__ __forceinline__ void pack_unit(const float (&f)[8], bf16x8& p) { p = pack8(f); }
__device__ __forceinline__ void pack_unit(const float (&f)[4], float4& p) { p = make_float4(f[0], f[1], f[2], f[3]); }

// sigmoid via the hardware tanh (one MUFU op, ~2^-11 relative error: well inside the bf16 the results are stored in).
// r01m: with exp + full-precision division the GroupNorm/SiLU kernels were issue-bound at 30-50% of the HBM roofline.
__device__ __forceinline__ float fast_sigmoid(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
  return fmaf(0.5f, t, 0.5f);
}
__device__ __forceinline__ float silu(float x) { return x * fast_sigmoid(x); }
// silu(2h) = 2h * sigmoid(2h) = h + h * tanh(h): with the factor 1/2 folded into the GroupNorm scale / shift the
// activation is FFMA, MUFU.TANH, FFMA per element instead of FMUL, MUFU, FFMA, FMUL on top of the affine FFMA (R2: the
// level-0 GroupNorm + SiLU passes spend half of their time issuing ~58 instructions per 16-byte unit).
__device__ __forceinline__ float silu_half(float h) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}

// silu in fp32 for the TF32 inference mode: x * sigmoid(x) with an exp-based sigmoid (a few ulp, where the hardware tanh
// above is ~2^-11 -- the size of a whole TF32 rounding).
__device__ __forceinline__ float silu_f32(float x) { return x / (1.0f + expf(-x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Packed fp32x2 arithmetic (Blackwell FADD2 / FFMA2: two fp32 lanes per instruction, same rounding as the scalar ops).
__device__ __forceinline__ void add2(float& a0, float& a1, float b0, float b1) {
  uint64_t a, b;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a) : "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(a));
}
// (c0, c1) += (a0 * a0, a1 * a1)
__device__ __forceinline__ void fma2_sq(float& c0, float& c1, float a0, float a1) {
  uint64_t a, c;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(c0), "f"(c1));
  asm("fma.rn.f32x2 %0, %1, %1, %0;" : "+l"(c) : "l"(a));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(c0), "=f"(c1) : "l"(c));
}

}  // namespace vdm
