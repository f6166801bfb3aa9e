// Thin inline-PTX wrappers for the sm_100a features used by the conv kernels:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / fences).
#pragma once

#include <cuda.h>
#include <stdint.h>

namespace vdm {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- mbarrier -----------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the waiting warp sleeps in hardware until the phase completes (or ~2 us pass)
// instead of returning after ~100 cycles.  R2b ncu: the 9-instruction polling loops of the MMA / producer warps were
// 20% of all issued instructions of the conv kernel, taken from the schedulers the epilogue warps run on.
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t hint_ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(hint_ns)
      : "memory");
  return ok != 0;
}
// Wait with a watchdog: a pipeline bug must trap (a launch error the host sees) instead of hanging the GPU
// (2^21 suspended retries of up to ~2 us each: seconds).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t spins = 0;
  while (!mbar_try_wait_hint(bar, parity, 2000u)) {
    if (++spins > (1u << 21)) {
      printf("vdm4cdm_b200: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}

// One lane of a fully converged warp (elect.sync): the compiler knows the guarded region is
// executed by a single thread, so warp-uniform operands stay in uniform registers.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// Per-warpgroup register budget (all four warps of the warpgroup execute the same instruction).
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}

// ---- TMA ------------------------------------------------------------------------------------
// 16-byte asynchronous global -> shared copy of the issuing thread (LDGSTS: no destination register, completion is
// tracked per commit group).
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// Wait until at most `pending` (0..3) of this thread's most recent commit groups are still in flight.
__device__ __forceinline__ void cp_async_wait(int pending) {
  switch (pending) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
  }
}

// Pull the cache line holding `p` into L2 (no register, no dependency).
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], "
      "[%2];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::
          "r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// 1-D bulk copy global -> shared (bytes % 16 == 0, both addresses 16-byte aligned), completing on `bar`.
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- tcgen05 ----------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Operand type of a tcgen05.mma: bf16 (kind::f16) or tf32 (kind::tf32).  One K step is 32 bytes of each operand in both
// kinds (K = 16 bf16 or K = 8 tf32), so the shared-memory descriptors of a K step are the same; only the instruction's
// kind and the A / B format fields of the instruction descriptor differ.
enum class MmaKind { kF16, kTF32 };
#define VDM_UMMA_KIND_ASM(K, BODY) \
  if constexpr (K == MmaKind::kTF32) asm volatile(BODY("tf32")); else asm volatile(BODY("f16"))

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 (or tf32) inputs, fp32 accumulate.
#define VDM_UMMA_BODY(KIND)                                                                    \
      "{\n\t"                                                                                  \
      ".reg .pred p;\n\t"                                                                      \
      "setp.ne.b32 p, %4, 0;\n\t"                                                              \
      "tcgen05.mma.cta_group::1.kind::" KIND " [%0], %1, %2, %3, p;\n\t"                       \
      "}" ::"r"(d_tmem),                                                                       \
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)                                    \
      : "memory"
template <MmaKind K = MmaKind::kF16>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  VDM_UMMA_KIND_ASM(K, VDM_UMMA_BODY);
}
#undef VDM_UMMA_BODY
// Same, with the descriptors assembled INSIDE the asm block from warp-uniform bases plus per-MMA offsets:
//   a_desc = {a_lo + a_off, a_hi32}, b_desc = {b_lo + b_off, b_hi32}, d = d_tmem + d_off.
// Keeping the adds next to the (volatile) MMA stops ptxas from pre-computing hundreds of descriptors into vector
// registers and moving them back with R2UR (r01s: ~65 issue cycles per MMA in the unrolled schedule).
#define VDM_UMMA_OFF_BODY(KIND)                                                                \
      "{\n\t"                                                                                  \
      ".reg .pred p;\n\t"                                                                      \
      ".reg .b32 alo, blo, dd;\n\t"                                                            \
      ".reg .b64 da, db;\n\t"                                                                  \
      "add.u32 alo, %1, %2;\n\t"                                                               \
      "add.u32 blo, %4, %5;\n\t"                                                               \
      "add.u32 dd, %0, %9;\n\t"                                                                \
      "mov.b64 da, {alo, %3};\n\t"                                                             \
      "mov.b64 db, {blo, %6};\n\t"                                                             \
      "setp.ne.b32 p, %8, 0;\n\t"                                                              \
      "tcgen05.mma.cta_group::1.kind::" KIND " [dd], da, db, %7, p;\n\t"                       \
      "}" ::"r"(d_tmem),                                                                       \
      "r"(a_lo), "r"(a_off), "r"(a_hi32), "r"(b_lo), "r"(b_off), "r"(b_hi32), "r"(idesc), "r"(accumulate), "r"(d_off) \
      : "memory"
template <MmaKind K = MmaKind::kF16>
__device__ __forceinline__ void umma_bf16_off(uint32_t d_tmem, uint32_t d_off, uint32_t a_lo, uint32_t a_off, uint32_t a_hi32,
                                              uint32_t b_lo, uint32_t b_off, uint32_t b_hi32, uint32_t idesc,
                                              uint32_t accumulate) {
  VDM_UMMA_KIND_ASM(K, VDM_UMMA_OFF_BODY);
}
#undef VDM_UMMA_OFF_BODY
// Same with whole 64-bit descriptors plus per-MMA offsets: ONE UIADD3.64 per descriptor in SASS (the 32-bit form above costs an
// add for the low word and a move for the high word of every descriptor pair: R3e, 6 uniform instructions per MMA from a single
// issuing thread that has ~56 cycles per MMA).  The low words (address >> 4 | LBO << 16) never carry into the high ones.
#define VDM_UMMA_OFF64_BODY(KIND)                                                              \
      "{\n\t"                                                                                  \
      ".reg .pred p;\n\t"                                                                      \
      ".reg .b32 dd;\n\t"                                                                      \
      ".reg .b64 da, db;\n\t"                                                                  \
      "add.u64 da, %1, %2;\n\t"                                                                \
      "add.u64 db, %3, %4;\n\t"                                                                \
      "add.u32 dd, %0, %7;\n\t"                                                                \
      "setp.ne.b32 p, %6, 0;\n\t"                                                              \
      "tcgen05.mma.cta_group::1.kind::" KIND " [dd], da, db, %5, p;\n\t"                       \
      "}" ::"r"(d_tmem),                                                                       \
      "l"(a_desc), "l"((uint64_t)a_off), "l"(b_desc), "l"((uint64_t)b_off), "r"(idesc), "r"(accumulate), "r"(d_off) \
      : "memory"
template <MmaKind K = MmaKind::kF16>
__device__ __forceinline__ void umma_bf16_off64(uint32_t d_tmem, uint32_t d_off, uint64_t a_desc, uint32_t a_off, uint64_t b_desc,
                                                uint32_t b_off, uint32_t idesc, uint32_t accumulate) {
  VDM_UMMA_KIND_ASM(K, VDM_UMMA_OFF64_BODY);
}
#undef VDM_UMMA_OFF64_BODY
#undef VDM_UMMA_KIND_ASM
// Arrive on `bar` when all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp receives lane (base+i).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Same, with the destination registers of the load as (fake) in/out operands: arithmetic on them cannot be scheduled
// above the wait, which matters once a second load is in flight while the first one's values are used.
__device__ __forceinline__ void tmem_ld_wait_dep(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :
               : "memory");
}

// ---- descriptors --------------------------------------------------------------------------------
// K-major shared-memory matrix descriptor for a tile whose rows are `row_bytes` (= swizzle span:
// 32, 64 or 128 bytes) of contiguous K, 8-row swizzle atoms stacked every 8*row_bytes.
// Field layout per cute/arch/mma_sm100_desc.hpp (SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout type [61,64) (SW128=2, SW64=4, SW32=6).
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t smem_addr, uint32_t row_bytes) {
  const uint64_t layout = row_bytes == 128 ? 2ull : (row_bytes == 64 ? 4ull : 6ull);
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;                              // LBO: unused for swizzled K-major
  d |= (uint64_t)((8u * row_bytes) >> 4) << 32;        // SBO: next 8-row atom
  d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
  d |= layout << 61;
  return d;
}
// Instruction descriptor (InstrDescriptor): D=f32 [4,6)=1, A format [7,10), B format [10,13) (kind::f16: bf16 = 1;
// kind::tf32: tf32 = 2), A,B K-major (bits 15,16 = 0), N>>3 [17,23), M>>4 [24,29).
template <MmaKind K = MmaKind::kF16>
__device__ __host__ __forceinline__ uint32_t make_idesc_bf16(uint32_t m, uint32_t n) {
  constexpr uint32_t ab = K == MmaKind::kTF32 ? 2u : 1u;
  return (1u << 4) | (ab << 7) | (ab << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

}  // namespace ptx
}  // namespace vdm
