// Conv3d ("same", stride 1, up to 27 taps) as an implicit GEMM on the 5th-gen tensor cores, fed from
// ONE halo tile per (output tile, channel chunk) instead of one tile per filter tap.
//
// Stands in for the cuDNN conv3d fprop (and, with flipped/transposed weights, dgrad) launched by
// every torch.nn.Conv3d of mltools' CUNet (networks.py:259-265 -> blocks.py:129-132, recovered in
// model_test.ipynb:684-692).
//
// Data layout ("channel-planar", 8 channels = 16 B per voxel and plane):
//     activations  bf16 [B][C/8][D][H][W][8]          weights  bf16 [tap][Cin/8][Cout_pad][8]
// Why: tcgen05.mma's un-swizzled K-major operand is a grid of 8-row x 16-byte core matrices whose
// rows are 16 B apart, 8-row groups SBO apart and K-neighbours LBO apart.  With the planar layout a
// halo box (MT+2, 18, 10) of one channel plane sits in shared memory as [d'][h'][w'][16 B], so
//   * 8 consecutive voxels along w are one core matrix,
//   * the 16 h-rows of a 16x8 output tile are 16 row groups at SBO = 10*16 B,
//   * the second half of K=16 is the next plane at LBO = plane stride,
//   * and a filter tap (dd,dh,dw) is nothing but a START-ADDRESS OFFSET of the descriptor.
// All 27 taps therefore read the same shared-memory bytes: L2->SM traffic per output voxel drops
// from 27x (per-tap im2col loads, what cuDNN/CUTLASS implicit GEMM do) to (MT+2)/MT*18/16*10/8 ~ 2.1x.
// (Descriptor semantics verified on hardware by tools/probe_umma.cu, profiles/r01_probe_umma.txt.)
//
// Pipeline per persistent CTA (16 warps in four warpgroups, setmaxnreg 64 / 176 / 176 / 88 registers):
//   warp 0   A producer : one 4-D TMA load per (tile, channel chunk) -> halo stage (2-4 stages);
//                         out-of-range voxels are zero-filled by the TMA unit == Conv3d zero padding
//   warp 2,3 B producer : weights -> shared memory, once per CTA when they fit (resident), else a ring of
//                         (chunk, 3 taps) stages (warp 3 takes every other stage of a streamed ring)
//   warp 1   MMA issuer : ONE elected lane.  generic path (issue_generic_tiles): chunk, weight stage, tap, sub-tile
//                         s < MT, k16: tcgen05.mma M=128 N=n_cta K=16 into accumulator s (TMEM, fp32), per-tap 64-bit
//                         descriptors + immediate per-MMA offsets, ring positions advanced without divisions.
//                         kd-folded path (narrow layers, NF = Cout_pad in {16, 32, 64}): see issue_fold_tile /
//                         issue_fold_stage; optionally one more channel chunk from a second tensor of which
//                         only the centre tap is multiplied (the block's 1x1x1 skip conv, issue_skip_chunk).
//                         2 accumulator sets: the epilogue of tile i overlaps the main loop of tile i+1
//   warps 4-11 epilogue : tcgen05.ld -> + bias/conditioning row + residual (cp.async ring in shared memory,
//                         optionally read through a nearest x2 up-sampling or a depth-to-space shuffle) -> bf16
//                         planar (or fp32 NCDHW) store, per-channel (sum, sumsq) GroupNorm statistics by warp-shuffle
//                         transpose reduction, kept per CTA in shared memory (fp64) and flushed with fp64
//                         atomics when the CTA moves to another sample.  Two warps per TMEM lane quarter.
//   warps 12-15 input transform (in_norm): GroupNorm + SiLU applied to the landed halo stage in place.
// Narrow 3x3x3 layers whose input channels are one chunk (Cin, Cout_pad <= 32) do not run this kernel but the
// d-marching schedule of conv3d_march.cuh (conv3d_march_kernel): one input slice per stage, a TMEM ring of 16 output
// slices, twelve epilogue warps (or eight + four transform warps).
//
// Roofline: tensor-bound; algorithmic FLOPs = 2 * taps * Cin * Cout * B*D*H*W.
#include "common.cuh"
#include "ptx.cuh"
#include "tma_host.cuh"

// Ablation branches (timing experiments whose results are wrong by construction) exist in bring-up builds only
// (-DVDM_BRINGUP, `make bringup`); in the release library VDM_DBG is a compile-time false and the branches vanish.
#ifdef VDM_BRINGUP
#define VDM_DBG(p, f) (((p).debug_flags & (f)) != 0)
#else
#define VDM_DBG(p, f) (false)
#endif

namespace vdm {

// 16 warps in four warpgroups (setmaxnreg re-balances the register file per warpgroup):
//   WG0  warp 0 A producer, warp 1 MMA issuer, warps 2, 3 B producers                 64 registers
//   WG1-2 warps 4..11  epilogue (two per TMEM lane quarter)                          176 registers
//   WG3  warps 12..15  input transform (GroupNorm + SiLU on the landed halo tile)     88 registers
constexpr int kConvThreads = 512;
constexpr int kEpiThreads = 256;        // warps 4..11
constexpr int kEpiFirst = 128;
constexpr int kXfThreads = 128;         // warps 12..15
constexpr int kXfFirst = 384;
constexpr int kRegsWg0 = 64, kRegsEpi = 176, kRegsXf = 88;
constexpr int kXfGroup = 2;              // units per software-pipeline group of the input transform (2 groups in flight)   // 128*64 + 256*176 + 128*88 = 64512 <= 65536
constexpr int kResSlotBytes = 2 * 16 * kEpiThreads;   // one unit (two 8-channel planes) of residual for every epilogue thread
constexpr int kMaxBStages = 16;
constexpr int kMaxAStages = 4;
constexpr int kTileH = 16, kTileW = 8;

struct ConvKernelParams {
  int B, D, H, W;
  int c_out;                 // real output channels
  int n_cta, n_split;        // UMMA N per CTA, CTAs sharing one spatial tile
  int n_pad;                 // rows per (tap, plane) of the weight tensor
  int n_taps, pad;
  uint16_t tap16[VDM_MAX_TAPS];  // halo offset of every tap in voxels (== 16-byte units)
  int8_t tap_kd[VDM_MAX_TAPS];   // fold path: which filter plane (0..2) a tap belongs to, and its (kh, kw) index
  int8_t tap_khw[VDM_MAX_TAPS];
  int8_t tap_of[3][9];           // fold path: tap index of (kd, khw)
  int fold_streamed;             // fold path with the weights streamed per (chunk, kh, kw) stage instead of resident
  int MT, KC, k_chunks;
  int Hd, Hh, Wh;            // halo box (voxels)
  int tiles_w, tiles_h, tiles_d, n_tiles;
  int fast_div_ok;           // n_tiles < 2^22: tile decoding by float reciprocals
  float inv_n_split, inv_tiles_w, inv_tiles_h, inv_tiles_d;
  int a_stage_bytes, b_stage_bytes, nsb, taps_per_stage;
  int nsa;                   // halo stages in flight (2..kMaxAStages): as many as fit next to the weights
  int b_resident;            // all weights of this CTA's channel slice stay in shared memory (loaded once)
  int plane_bytes;           // Hd*Hh*Wh*16
  int tmem_cols;
  int x_planes, x_plane0, c_in8;
  int x_shift;               // 1 when x carries a one-voxel periodic halo (circular padding)
  // fused 1x1x1 skip-path conv (kd-folded resident layers): extra channel chunks read from a second tensor, centre tap only
  int skip_chunks;           // number of KC-channel chunks of the second tensor (0: none)
  int x2_planes, x2_plane0;
  int skip_w_bytes;          // bytes of its weights in shared memory, right after the main weights
  const __nv_bfloat16* w2;   // packed [1][skip_c_in/8][n_pad][8]
  const __nv_bfloat16* w;
  // epilogue
  void* y;
  int y_planes, y_plane0, out_fp32;
  const float* chan_add;
  const int32_t* step_ptr;
  long long chan_add_step_stride;
  const __nv_bfloat16* residual;
  int r_planes, r_plane0;
  int r_up;                  // residual on the half-resolution grid, read through a nearest x2 up-sampling
  int r_d2s_planes;          // != 0 (with r_up): the half-resolution residual holds 8 parity blocks of this many planes each
                             // (block (d&1)*4 + (h&1)*2 + (w&1)) and is read through a depth-to-space shuffle
  int res_depth;             // units of residual in flight per epilogue thread (cp.async ring), 1..4
  int res_ring_off;          // byte offset of that ring in dynamic shared memory
  double* stats;
  int stats_channels, stats_c0;
  const float* in_norm;      // fused input transform: fp32 [B][c_in][2] (a, b), silu(gn(x)) = h + h tanh(h), h = a x + b
  int c_in;                  // channels of x read (the in_norm row length)
  int xf_coef_off;           // byte offset of the current sample's (a, b) table in dynamic shared memory
  int m_units, m_nseg, m_seglen;   // d-marching schedule (conv3d_march.cuh): units = columns x d-segments of m_seglen slices
  int debug_flags;           // bring-up experiments (results are wrong): 1 = epilogue does no work, 2 = halo loaded for the
                             // first two tiles only, 4 = no TMEM reads, 8 = no output stores, 16 = no statistics
                             // transpose-reduction, 32 = no statistics barrier + fold
};

struct ConvShared {
  uint64_t a_full[kMaxAStages], a_empty[kMaxAStages];
  uint64_t a_ready[kMaxAStages];   // fused input transform: the landed halo stage has been rewritten in place
  uint64_t b_full[kMaxBStages], b_empty[kMaxBStages];
  uint64_t tmem_full[2], tmem_empty[2];
  uint32_t tmem_base;
  // (statistics scratch follows this struct in shared memory, sized by the CTA's channel count: per-tile, per-warp
  //  partials float [2 parities][2][8][n_cta], then the per-CTA running (sum, sumsq) of the current sample,
  //  double [2][n_cta], flushed when the sample changes -- 3.5 KB less than fixed 256-channel arrays, which is what
  //  lets the 96 -> 32 layer keep its weights resident next to MT = 3 halo stages)
  alignas(16) float cadd[2][256];  // bias + conditioning row of this tile's sample, double-buffered by tile parity
};

// Transpose-reduce 16 per-row values over the 32 lanes of a warp: afterwards lane l (even) holds
// the column (l >> 1) total in v[0].
__device__ __forceinline__ void warp_column_sums16(float (&v)[16]) {
  const unsigned full = 0xffffffffu;
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const bool hi = lane & 16;
    const float send = hi ? v[i] : v[i + 8];
    const float keep = hi ? v[i + 8] : v[i];
    v[i] = keep + __shfl_xor_sync(full, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const bool hi = lane & 8;
    const float send = hi ? v[i] : v[i + 4];
    const float keep = hi ? v[i + 4] : v[i];
    v[i] = keep + __shfl_xor_sync(full, send, 8);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const bool hi = lane & 4;
    const float send = hi ? v[i] : v[i + 2];
    const float keep = hi ? v[i + 2] : v[i];
    v[i] = keep + __shfl_xor_sync(full, send, 4);
  }
  {
    const bool hi = lane & 2;
    const float send = hi ? v[0] : v[1];
    const float keep = hi ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(full, send, 2);
  }
  v[0] += __shfl_xor_sync(full, v[0], 1);
}

struct TileCoord {
  int b, d0, h0, w0, ns;
};
// x / d for 0 <= x < 2^22 with inv = 1.0f / d: (x + 0.5) * inv is at least 0.5/d away from an integer, far more than
// the fp32 rounding error, so truncation is exact.  (Every epilogue thread decodes every tile; four integer divisions
// by run-time values were 9% of the epilogue's instructions in r01t.)
__device__ __forceinline__ int fast_div(int x, int d, float inv) {
  (void)d;
  return __float2int_rz(((float)x + 0.5f) * inv);
}
__device__ __forceinline__ TileCoord decode_tile(const ConvKernelParams& p, int tile) {
  TileCoord t;
  int q;
  if (p.fast_div_ok) {
    q = fast_div(tile, p.n_split, p.inv_n_split); t.ns = tile - q * p.n_split; tile = q;
    q = fast_div(tile, p.tiles_w, p.inv_tiles_w); t.w0 = (tile - q * p.tiles_w) * kTileW; tile = q;
    q = fast_div(tile, p.tiles_h, p.inv_tiles_h); t.h0 = (tile - q * p.tiles_h) * kTileH; tile = q;
    q = fast_div(tile, p.tiles_d, p.inv_tiles_d); t.d0 = (tile - q * p.tiles_d) * p.MT;
    t.b = q;
  } else {
    t.ns = tile % p.n_split; tile /= p.n_split;
    t.w0 = (tile % p.tiles_w) * kTileW; tile /= p.tiles_w;
    t.h0 = (tile % p.tiles_h) * kTileH; tile /= p.tiles_h;
    t.d0 = (tile % p.tiles_d) * p.MT;
    t.b = tile / p.tiles_d;
  }
  return t;
}

// Position in a ring of `n` pipeline stages and the mbarrier phase parity of that lap, advanced without divisions.
// (R3w ncu of a 128 -> 128 layer: the issuing thread spent half of every 12-MMA weight stage on `it % nsb`, `it / nsb` with a
// run-time nsb -- an I2F / MUFU.RCP sequence -- and on re-loading loop-invariant kernel parameters from the constant bank;
// the tensor pipe was active 48 % of the time with L2 at 12 %.)  Consumers wait full[s] with parity ph, producers empty[s]
// with parity ph ^ 1.
struct Ring {
  uint32_t s, ph, n;
  __device__ __forceinline__ explicit Ring(uint32_t n_) : s(0u), ph(0u), n(n_) {}
  __device__ __forceinline__ void next() {
    if (++s == n) {
      s = 0u;
      ph ^= 1u;
    }
  }
};
// A copy of a kernel parameter the compiler has to keep in a register (it otherwise re-materialises loop-invariant
// parameters with LDCU inside the issue loops, ~30 cycles of latency each on the single issuing thread).
__device__ __forceinline__ uint32_t hold_u32(uint32_t v) {
  asm volatile("mov.u32 %0, %0;" : "+r"(v));
  return v;
}

// Un-swizzled K-major descriptor: rows 16 B apart inside a core matrix, `sbo` between 8-row groups,
// `lbo` between the two K core matrices of one K=16 MMA (cute::UMMA::SmemDescriptor, version 1).
__device__ __forceinline__ uint64_t make_planar_desc(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}

// ---- kd-folded issue schedule (narrow layers) -----------------------------------------------------------
// With N = Cout_pad = 32 a tcgen05.mma (M=128, K=16) needs 5 KB of operands for 16 tensor-pipe cycles of
// math and runs at the 128 B/clk shared-memory operand rate instead: 41 cycles (tools/probe_mma_rate.cu,
// profiles/r01d_probe_mma_rate.txt) -- 39% of the tensor peak at best.  The fix is to make N wider without
// touching the layer: ONE input slice i of the halo feeds up to THREE output slices (s = i - kd), so
// for a fixed (kh, kw, k16) the A operand (slice i shifted by (kh, kw)) is multiplied by the weights of
// kd = 2, 1, 0 stacked along N (3*NF rows, shared-memory order [khw][plane][2-kd][co]) straight into the
// accumulators of slices s = i-2, i-1, i, which are adjacent TMEM column blocks.  Same MACs, a third of the
// A fetches: N = 96 runs at 56 cycles for 3x the math (86% of peak), the two edge slices of a tile at N = 64 / 32.
// The accumulator of slice s = i is first touched at (kh, kw, k16) = (0, 0, 0) of input slice i, as the LAST block
// of that MMA's span, so that one MMA is split in two (fresh block / accumulating blocks).
// Layers with more input channels than one halo stage holds run the schedule once per channel chunk (FIRST = false
// accumulates everywhere); all chunks' weights stay resident.
// Everything is compile-time: the schedule is a straight line of (MT+2)*9*KJ (+MT) MMAs with immediate
// descriptor offsets, because the per-tap bookkeeping of the generic loop, not the MMAs, bounded these
// layers (r01i: identical time with the epilogue and the halo loads switched off).
template <int MT, int KJ, int NF, bool FIRST>
__device__ __forceinline__ void issue_fold_tile(uint32_t a_lo0, uint32_t b_base16, uint64_t a_hi, uint64_t b_hi,
                                                uint32_t d_tmem0) {
  constexpr int Hh = kTileH + 2, Wh = kTileW + 2, Hd = MT + 2;
  constexpr uint32_t plane16 = (uint32_t)(Hd * Hh * Wh);
  constexpr uint32_t kstep_a16 = 2u * plane16;
  const uint32_t a_hi32 = (uint32_t)(a_hi >> 32), b_hi32 = (uint32_t)(b_hi >> 32);
  // One loop trip per input slice (NOT unrolled: a fully unrolled schedule made ptxas software-pipeline the
  // descriptor arithmetic over dozens of MMAs and spill uniform registers, ~65 issue cycles per MMA); inside a
  // trip the 9*KJ MMAs differ only by immediate offsets from per-slice bases.
#pragma unroll 1
  for (int i = 0; i < MT + 2; ++i) {
    const int kd_lo = (i - MT + 1) > 0 ? (i - MT + 1) : 0;
    const int kd_hi = i < 2 ? i : 2;
    const int s_lo = i - kd_hi;
    const int nblk = kd_hi - kd_lo + 1;
    // accumulator s = i receives its first contribution (kd = 0, the last block) in the first channel chunk
    const bool starts = FIRST && i < MT;
    // low descriptor words: start address (16-byte units) | LBO << 16 (the low word of a_hi / b_hi)
    const uint32_t a_i = a_lo0 + (uint32_t)(i * Hh * Wh) + (uint32_t)a_hi;
    const uint32_t b_i = b_base16 + (uint32_t)((2 - kd_hi) * NF) + (uint32_t)b_hi;
    const uint32_t d_i = d_tmem0 + (uint32_t)(s_lo * NF);
    const uint32_t idesc_i = ptx::make_idesc_bf16(128, (uint32_t)(nblk * NF));
#pragma unroll
    for (int khw = 0; khw < 9; ++khw) {
#pragma unroll
      for (int j = 0; j < KJ; ++j) {
        const uint32_t a_off = (uint32_t)((khw / 3) * Wh + khw % 3) + (uint32_t)j * kstep_a16;
        const uint32_t b_off = (uint32_t)((khw * 2 * KJ + 2 * j) * 3 * NF);
        if (khw == 0 && j == 0) {
          if (starts) {
            if (nblk > 1)
              ptx::umma_bf16_off(d_i, 0u, a_i, a_off, a_hi32, b_i, b_off, b_hi32,
                                 ptx::make_idesc_bf16(128, (uint32_t)((nblk - 1) * NF)), 1u);
            ptx::umma_bf16_off(d_tmem0, (uint32_t)(i * NF), a_i, a_off, a_hi32, b_i, b_off + (uint32_t)((nblk - 1) * NF), b_hi32,
                               ptx::make_idesc_bf16(128, (uint32_t)NF), 0u);
          } else {
            ptx::umma_bf16_off(d_i, 0u, a_i, a_off, a_hi32, b_i, b_off, b_hi32, idesc_i, 1u);
          }
        } else {
          ptx::umma_bf16_off(d_i, 0u, a_i, a_off, a_hi32, b_i, b_off, b_hi32, idesc_i, 1u);
        }
      }
    }
  }
}

// Fused 1x1x1 skip-path conv of a ResNet block (h_out = conv3x3x3(a2) + conv1x1x1(x_skip) + ...): one more channel
// chunk loaded from the skip tensor as a box WITHOUT halo, [plane][MT d][16 h][8 w][16 B] (a 1x1x1 filter needs the
// tile's own voxels only: 32 KB instead of a 69 KB halo box), MT*KJ MMAs of N = NF on top of the (MT+2)*9*KJ of a main
// chunk.  Weights: [plane][co] (LBO = NF*16 bytes).
template <int MT, int KJ, int NF>
__device__ __forceinline__ void issue_skip_chunk(uint32_t a_lo0, uint32_t b_lo16, uint32_t d_tmem0) {
  constexpr uint32_t slice16 = (uint32_t)(kTileH * kTileW);          // one d-slice of a plane, 16-byte units
  constexpr uint32_t plane16 = (uint32_t)MT * slice16;
  constexpr uint32_t kstep_a16 = 2u * plane16;
  // A: K-major, 8 voxels along w = one core matrix, next h row (SBO) 128 B on, next 8 channels (LBO) one plane on
  const uint64_t a_hi = make_planar_desc(0, plane16 * 16u, (uint32_t)kTileW * 16u);
  const uint64_t b_hi = make_planar_desc(0, (uint32_t)NF * 16u, 128u);
  const uint32_t a_hi32 = (uint32_t)(a_hi >> 32), b_hi32 = (uint32_t)(b_hi >> 32);
  const uint32_t idesc = ptx::make_idesc_bf16(128, (uint32_t)NF);
  const uint32_t b_i = b_lo16 + (uint32_t)b_hi;
#pragma unroll
  for (int i = 0; i < MT; ++i) {
    const uint32_t a_i = a_lo0 + (uint32_t)i * slice16 + (uint32_t)a_hi;
#pragma unroll
    for (int j = 0; j < KJ; ++j)
      ptx::umma_bf16_off(d_tmem0, (uint32_t)(i * NF), a_i, (uint32_t)j * kstep_a16, a_hi32, b_i, (uint32_t)(2 * j * NF),
                         b_hi32, idesc, 1u);
  }
}

// Same schedule for layers whose weights do not fit shared memory (Cout_pad = 64): the weights of ONE (chunk, kh, kw)
// for the three kd stacked along N are a ring stage [plane][2 - kd][co]; the stage's MMAs run over all input slices.
// N = 192 is tensor-bound (96 cycles of math for 80 cycles of operand fetch) where N = 64 is fetch-bound (48 for 32).
template <int MT, int KJ, int NF>
__device__ __forceinline__ void issue_fold_stage(uint32_t a_lo, uint32_t b_lo, uint32_t a_hi32, uint32_t b_hi32,
                                                 uint32_t d_tmem0, bool first) {
  constexpr int Hh = kTileH + 2, Wh = kTileW + 2, Hd = MT + 2;
  constexpr uint32_t plane16 = (uint32_t)(Hd * Hh * Wh);
  constexpr uint32_t kstep_a16 = 2u * plane16;
#pragma unroll
  for (int i = 0; i < MT + 2; ++i) {
    const int kd_lo = (i - MT + 1) > 0 ? (i - MT + 1) : 0;
    const int kd_hi = i < 2 ? i : 2;
    const int s_lo = i - kd_hi;
    const int nblk = kd_hi - kd_lo + 1;
#pragma unroll
    for (int j = 0; j < KJ; ++j) {
      const uint32_t a_off = (uint32_t)(i * Hh * Wh) + (uint32_t)j * kstep_a16;
      const uint32_t b_off = (uint32_t)((2 * j * 3 + (2 - kd_hi)) * NF);
      if (j == 0 && i < MT && first) {
        // accumulator s = i receives its first contribution here (kd = 0, the last block of the span)
        if (nblk > 1)
          ptx::umma_bf16_off(d_tmem0, (uint32_t)(s_lo * NF), a_lo, a_off, a_hi32, b_lo, b_off, b_hi32,
                             ptx::make_idesc_bf16(128, (uint32_t)((nblk - 1) * NF)), 1u);
        ptx::umma_bf16_off(d_tmem0, (uint32_t)(i * NF), a_lo, a_off, a_hi32, b_lo, b_off + (uint32_t)((nblk - 1) * NF), b_hi32,
                           ptx::make_idesc_bf16(128, (uint32_t)NF), 0u);
      } else {
        ptx::umma_bf16_off(d_tmem0, (uint32_t)(s_lo * NF), a_lo, a_off, a_hi32, b_lo, b_off, b_hi32,
                           ptx::make_idesc_bf16(128, (uint32_t)(nblk * NF)), 1u);
      }
    }
  }
}

// ---- fused input transform -----------------------------------------------------------------------------------
// The conv reads the RAW tensor (the producer's output before GroupNorm); warps 12..15 rewrite every landed halo stage
// in place, y = silu(a_c x + b'_c) per (sample, channel) = h + h tanh(h) with h = a x + b (vdm_gn_coef), re-zero the
// voxels the TMA unit filled for out-of-range coordinates (Conv3d's zero padding is applied AFTER the non-linearity),
// make the writes visible to the async proxy (tcgen05.mma reads shared memory through it) and hand the stage to the
// MMA issuer.  This removes the separate GroupNorm + SiLU pass: one read and one write of the tensor per conv input.
// Work split: a warp owns whole planes (its 16 coefficients stay in registers for the stage); with fewer than four
// planes per chunk the voxels of a plane are split between warps.  Lanes walk consecutive 16-byte units (conflict-free).
template <int HH, int WH>
__device__ __forceinline__ bool halo_voxel_oob(int v, int dlo, int hlo, int wlo, int D, int H, int W) {
  const int dz = v / (HH * WH);
  const int rem = v - dz * (HH * WH);
  const int hy = rem / WH;
  const int wx = rem - hy * WH;
  return (unsigned)(dlo + dz) >= (unsigned)D || (unsigned)(hlo + hy) >= (unsigned)H || (unsigned)(wlo + wx) >= (unsigned)W;
}

__device__ __forceinline__ uint4 gn_silu8(const uint4 x, const float (&ca)[8], const float (&cb)[8]) {
  bf16x8 in;
  in.u = x;
  float f[8];
  unpack8(in, f);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float h = fmaf(f[j], ca[j], cb[j]);
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    f[j] = fmaf(h, t, h);
  }
  return pack8(f).u;
}

// (a, b) of 8 channels, stored interleaved [channel][a | b], into ca[8], cb[8]: from shared memory, or (LDG) from global
// memory through the read-only path.
template <bool LDG>
__device__ __forceinline__ void load_coef8(const float* src, float (&ca)[8], float (&cb)[8]) {
  const float4* cs = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int j4 = 0; j4 < 4; ++j4) {
    const float4 c4 = LDG ? __ldg(cs + j4) : cs[j4];
    ca[2 * j4] = c4.x; cb[2 * j4] = c4.y; ca[2 * j4 + 1] = c4.z; cb[2 * j4 + 1] = c4.w;
  }
}

template <int MT, int KJ>
__device__ __forceinline__ void transform_tiles(const ConvKernelParams& p, ConvShared* sh, uint8_t* a_smem, float* coef) {
  constexpr int planes = 2 * KJ;
  constexpr int nparts = planes >= 4 ? 1 : 4 / planes;        // warps sharing one plane
  static_assert((MT + 2) * (kTileH + 2) * (kTileW + 2) <= 64 * 32, "zmask: one bit per 16-byte unit of a thread");
  constexpr int pl_step = planes >= 4 ? 4 : planes;
  const int xt = threadIdx.x - kXfFirst, tw = xt >> 5, lane = xt & 31;
  const int pl0 = planes >= 4 ? tw : tw % planes;
  const int part = planes >= 4 ? 0 : tw / planes;
  const int vh = p.Hd * p.Hh * p.Wh;                          // voxels (16-byte units) of one plane of the stage
  const int total_chunks = p.k_chunks + p.skip_chunks;
  int cur_b = -1;
  Ring ra((uint32_t)p.nsa);
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const TileCoord t = decode_tile(p, tile);
    if (t.b != cur_b) {
      // (a, b) table of this sample -> shared memory; the first barrier keeps a slow warp from reading a table that
      // is being replaced
      asm volatile("bar.sync 3, 128;" ::: "memory");
      const float4* src = reinterpret_cast<const float4*>(p.in_norm + (long long)t.b * p.c_in * 2);
      for (int i = xt; i < p.c_in / 2; i += kXfThreads) reinterpret_cast<float4*>(coef)[i] = __ldg(src + i);
      asm volatile("bar.sync 3, 128;" ::: "memory");
      cur_b = t.b;
    }
    const int dlo = t.d0 - p.pad + p.x_shift, hlo = t.h0 - p.pad + p.x_shift, wlo = t.w0 - p.pad + p.x_shift;
    // Units of this thread that lie outside the grid (zero padding applies AFTER the non-linearity): bit k = unit
    // part * 32 + lane + k * step, the same for every plane and chunk of the tile (at most 6 * 18 * 10 / 32 = 34 units per
    // thread).  One mask per tile instead of a branch and two divisions per unit: the loop body below is branch-free, so
    // ptxas interleaves the units of a group (R5g/R5i: the branchy body of the marching schedule ran at ~4.5 cycles per
    // instruction and its four warps were the bound of the fused layers).
    unsigned long long zmask = 0ull;
    if (dlo < 0 || dlo + p.Hd > p.D || hlo < 0 || hlo + p.Hh > p.H || wlo < 0 || wlo + p.Wh > p.W) {
      int k = 0;
      for (int idx = part * 32 + lane; idx < vh; idx += 32 * nparts, ++k) {
        const bool oob = p.pad ? halo_voxel_oob<kTileH + 2, kTileW + 2>(idx, dlo, hlo, wlo, p.D, p.H, p.W)
                               : halo_voxel_oob<kTileH, kTileW>(idx, dlo, hlo, wlo, p.D, p.H, p.W);
        if (oob) zmask |= 1ull << k;
      }
    }
    for (int kc = 0; kc < total_chunks; ++kc, ra.next()) {
      const int s = (int)ra.s;
      ptx::mbar_wait(&sh->a_full[s], ra.ph);
      if (kc < p.k_chunks && !VDM_DBG(p, 64)) {          // (bring-up flag 64: hand-off only, no arithmetic)
        uint8_t* stage = a_smem + (size_t)s * p.a_stage_bytes;
#pragma unroll 1
        for (int pl = pl0; pl < planes; pl += pl_step) {
          float ca[8], cb[8];
          load_coef8<false>(coef + (size_t)((kc * planes + pl) * 8) * 2, ca, cb);
          uint4* base = reinterpret_cast<uint4*>(stage + (size_t)pl * p.plane_bytes);
          // Software pipeline, kXfGroup units per group, the NEXT group's loads in flight while this one is computed:
          // while the tensor core streams its operands out of the same shared memory (the N = 96 MMAs of the narrow layers
          // run at the shared-memory operand rate) an LDS takes several hundred cycles, and with one or two loads in
          // flight per thread the transform of a stage took 9K cycles (R2e ncu) -- longer than the MMAs of a tile.
          constexpr int G = kXfGroup;
          const int step = 32 * nparts;
          int v = part * 32 + lane;
          uint4 cur[G], nxt[G];
#pragma unroll
          for (int g2 = 0; g2 < G; ++g2) {
            const int idx = v + g2 * step;
            cur[g2] = idx < vh ? base[idx] : make_uint4(0u, 0u, 0u, 0u);
          }
          int k = 0;
#pragma unroll 1
          for (; v < vh; v += G * step, k += G) {
            const int vn = v + G * step;
#pragma unroll
            for (int g2 = 0; g2 < G; ++g2) {
              const int idx = vn + g2 * step;
              nxt[g2] = idx < vh ? base[idx] : make_uint4(0u, 0u, 0u, 0u);
            }
            const unsigned zk = (unsigned)(zmask >> k);
#pragma unroll
            for (int g2 = 0; g2 < G; ++g2) {
              const int idx = v + g2 * step;
              uint4 y = VDM_DBG(p, 128) ? cur[g2] : gn_silu8(cur[g2], ca, cb);     // (bring-up 128: copy through)
              if ((zk >> g2) & 1u) y = make_uint4(0u, 0u, 0u, 0u);
              if (idx < vh && !VDM_DBG(p, 256)) base[idx] = y;                       // (bring-up 256: no stores)
            }
#pragma unroll
            for (int g2 = 0; g2 < G; ++g2) cur[g2] = nxt[g2];
          }
        }
      }
      // generic-proxy writes -> visible to the async proxy (UMMA operand fetch), then release the stage to the MMA warp
      ptx::fence_proxy_async();
      ptx::mbar_arrive(&sh->a_ready[s]);
    }
  }
}

// ---- epilogue ---------------------------------------------------------------------------------------------
// 8 warps, two per TMEM lane quarter; thread = one output voxel of the 16 x 8 tile face, unit = (d-slice, 16-channel
// chunk).  The two warps of a quarter split the units by chunk when the CTA has at least two chunks (each warp then owns
// whole channels and reduces their statistics over all MT slices in registers), else by slice.
// The feature set (residual, statistics, fp32 output) is a TEMPLATE parameter chosen once per launch: the r02 epilogue
// tested those run-time flags inside the unit loop and executed 130 (bare) to 325 (bias + residual + statistics)
// instructions per unit, 37 of them branches, from two warps per scheduler -- the level-0 layers were bound by that
// instruction stream, not by the tensor pipe (profiles/R2b_epilogue_sass.txt).  Here a unit is straight-line code: the
// bias row of a chunk lives in registers for the whole tile, the TMEM load of unit i+1 is issued before unit i is
// processed, output pointers advance by adds, and shared memory is addressed as shared memory.
constexpr int kEpiRes = 1, kEpiStats = 2, kEpiFp32 = 4;
// fp32 channel-planar output [B][C/4][D][H][W][4] (the TF32 instances): a 16-channel unit is four 16-byte planes, the
// residual is read in the same layout, and the statistics are those of the stored, un-rounded fp32 values.
constexpr int kEpiF32Planar = 8;

// Bias + conditioning rows of the launch, [B][c_out] (the sampler step's rows when they vary per step), or null.
__device__ __forceinline__ const float* cadd_rows(const ConvKernelParams& p) {
  const long long cadd_step = (p.chan_add && p.step_ptr) ? (long long)(*p.step_ptr) : 0ll;
  return p.chan_add ? p.chan_add + cadd_step * p.chan_add_step_stride : nullptr;
}

__device__ __forceinline__ void load_row16(const float* src, float (&v)[16]) {
  const float4* cs = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int j4 = 0; j4 < 4; ++j4) {
    const float4 cv = cs[j4];
    v[4 * j4] = cv.x; v[4 * j4 + 1] = cv.y; v[4 * j4 + 2] = cv.z; v[4 * j4 + 3] = cv.w;
  }
}

// The pieces below are macros, not functions: nvcc optimises a __forceinline__ function on its own before it inlines it, and
// written as functions they changed the code of most conv kernels (address arithmetic, loop bounds and branches moved).
// Expanded in place, every expression stays where the caller's code had it and both schedules compile as before.

// Bias + conditioning rows of every sample (cadd_g: cadd_rows) -> shared-memory table dst[rows][cols], zeros past c_out and
// without rows, so that the unit code has no "is there a bias" branch; filled by the kThreads epilogue threads (et = 0 ..
// kThreads - 1), which then meet at named barrier 1.
#define VDM_CADD_TABLE_FILL(dst, cadd_g, rows, cols, c_out, et, kThreads)                                                    \
  {                                                                                                                         \
    for (int i_ = (et); i_ < (rows) * (cols); i_ += (kThreads)) {                                                          \
      const int bb_ = i_ / (cols), c_ = i_ - bb_ * (cols);                                                                  \
      (dst)[i_] = ((cadd_g) && c_ < (c_out)) ? __ldg((cadd_g) + (long long)bb_ * (c_out) + c_) : 0.f;                      \
    }                                                                                                                       \
    asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory");                                                           \
  }

// fp32 NCDHW output (conv_out): the first c_left channels of the 16-channel unit f, V (one channel) apart from yp on.
#define VDM_STORE_FP32_NCDHW(yp, f, c_left, V)                                                                              \
  {                                                                                                                         \
    float* yp_ = (yp);                                                                                                      \
    _Pragma("unroll") for (int j_ = 0; j_ < 16; ++j_) if (j_ < (c_left)) yp_[(long long)j_ * (V)] = (f)[j_];                \
  }

// Half h (channels 8h .. 8h + 7) of the 16-channel unit f of planar output: + residual, store, per-lane statistics
// s1[8h + j] += y, s2[8h + j] += y^2 of the STORED values (for bf16 output: after rounding).  bf16 planes: residual r0, one
// store at y_out[off].  fp32 planes: residual r0, r1, stores at y_out[off0], y_out[off1].  RES, STATS: compile-time flags.
#define VDM_HALF_STATS(g, h, s1, s2)                                                                                        \
  {                                                                                                                         \
    _Pragma("unroll") for (int j_ = 0; j_ < 8; j_ += 2) {                                                                   \
      add2((s1)[(h) * 8 + j_], (s1)[(h) * 8 + j_ + 1], (g)[j_], (g)[j_ + 1]);                                               \
      fma2_sq((s2)[(h) * 8 + j_], (s2)[(h) * 8 + j_ + 1], (g)[j_], (g)[j_ + 1]);                                            \
    }                                                                                                                       \
  }
#define VDM_STORE_HALF_BF16(RES, STATS, f, h, r0, y_out, off, s1, s2)                                                       \
  {                                                                                                                         \
    float g_[8];                                                                                                            \
    _Pragma("unroll") for (int j_ = 0; j_ < 8; ++j_) g_[j_] = (f)[(h) * 8 + j_];                                            \
    if (RES) {                                                                                                              \
      float rr_[8];                                                                                                         \
      bf16x8 rv_;                                                                                                           \
      rv_.u = (r0);                                                                                                         \
      unpack8(rv_, rr_);                                                                                                    \
      _Pragma("unroll") for (int j_ = 0; j_ < 8; j_ += 2) add2(g_[j_], g_[j_ + 1], rr_[j_], rr_[j_ + 1]);                   \
    }                                                                                                                       \
    const bf16x8 packed_ = pack8(g_);                                                                                       \
    (y_out)[off] = packed_;                                                                                                 \
    if (STATS) {                                                                                                            \
      unpack8(packed_, g_);                                                                                                 \
      VDM_HALF_STATS(g_, h, s1, s2);                                                                                        \
    }                                                                                                                       \
  }
#define VDM_STORE_HALF_F32P(RES, STATS, f, h, r0, r1, y_out, off0, off1, s1, s2)                                            \
  {                                                                                                                         \
    float g_[8];                                                                                                            \
    _Pragma("unroll") for (int j_ = 0; j_ < 8; ++j_) g_[j_] = (f)[(h) * 8 + j_];                                            \
    if (RES) {                                                                                                              \
      const uint4 ra_ = (r0), rb_ = (r1);                                                                                   \
      add2(g_[0], g_[1], __uint_as_float(ra_.x), __uint_as_float(ra_.y));                                                   \
      add2(g_[2], g_[3], __uint_as_float(ra_.z), __uint_as_float(ra_.w));                                                   \
      add2(g_[4], g_[5], __uint_as_float(rb_.x), __uint_as_float(rb_.y));                                                   \
      add2(g_[6], g_[7], __uint_as_float(rb_.z), __uint_as_float(rb_.w));                                                   \
    }                                                                                                                       \
    (y_out)[off0] = make_float4(g_[0], g_[1], g_[2], g_[3]);                                                                \
    (y_out)[off1] = make_float4(g_[4], g_[5], g_[6], g_[7]);                                                                \
    if (STATS) VDM_HALF_STATS(g_, h, s1, s2);                                                                               \
  }

// Per-lane statistics s1, s2 of a 16-channel chunk (channels c0 .. c0 + 15 of the CTA) -> this warp's slots: one transpose
// reduction, then part[ew][c] = sum, part[kSlotWarps + ew][c] = sum of squares (rows of `cols` channels).
#define VDM_STATS_TO_SLOTS(s1, s2, part, ew, cols, c0, kSlotWarps, lane)                                                     \
  {                                                                                                                         \
    warp_column_sums16(s1);                                                                                                 \
    warp_column_sums16(s2);                                                                                                 \
    if (((lane) & 1) == 0) {                                                                                                \
      const int c_ = (c0) + ((lane) >> 1);                                                                                  \
      (part)[(ew) * (cols) + c_] = (s1)[0];                                                                                 \
      (part)[((kSlotWarps) + (ew)) * (cols) + c_] = (s2)[0];                                                                \
    }                                                                                                                       \
  }

// Channel c of the CTA: the slots of its kWarps warps, summed in a fixed order (statistics do not depend on timing), into the
// fp64 running sums acc[c], acc[cols + c]; on `flush` (the CTA moves on to another sample or channel slice, or ends) those go
// to the (sum, sumsq) of (sample b, channel cbase + c) with fp64 atomics -- never for padded channels -- and restart.
// kZeroSlots: the slots are cleared as they are read, for a caller whose warps do not write every slot of every round.
#define VDM_FOLD_STATS(p, part, acc, cols, c, kWarps, kSlotWarps, kZeroSlots, flush, b, cbase)                              \
  {                                                                                                                         \
    const int c_ = (c);                                                                                                     \
    float t1_ = 0.f, t2_ = 0.f;                                                                                             \
    _Pragma("unroll") for (int wv_ = 0; wv_ < (kWarps); ++wv_) {                                                            \
      t1_ += (part)[wv_ * (cols) + c_];                                                                                     \
      t2_ += (part)[((kSlotWarps) + wv_) * (cols) + c_];                                                                    \
      if (kZeroSlots) {                                                                                                     \
        (part)[wv_ * (cols) + c_] = 0.f;                                                                                    \
        (part)[((kSlotWarps) + wv_) * (cols) + c_] = 0.f;                                                                   \
      }                                                                                                                     \
    }                                                                                                                       \
    const double a1_ = (acc)[c_] + (double)t1_;                                                                             \
    const double a2_ = (acc)[(cols) + c_] + (double)t2_;                                                                    \
    if (flush) {                                                                                                            \
      if ((cbase) + c_ < (p).c_out) {                                                                                       \
        double* dst_ = (p).stats + ((long long)(b) * (p).stats_channels + (p).stats_c0 + (cbase) + c_) * 2;                 \
        atomicAdd(dst_, a1_);                                                                                               \
        atomicAdd(dst_ + 1, a2_);                                                                                           \
      }                                                                                                                     \
      (acc)[c_] = 0.0;                                                                                                      \
      (acc)[(cols) + c_] = 0.0;                                                                                             \
    } else {                                                                                                                \
      (acc)[c_] = a1_;                                                                                                      \
      (acc)[(cols) + c_] = a2_;                                                                                             \
    }                                                                                                                       \
  }

template <int MT, int MODE>
__device__ __forceinline__ void epilogue_tiles(const ConvKernelParams& p, ConvShared* sh, uint8_t* smem, float* stat_part,
                                               double* stat_acc, const uint32_t tmem_base) {
  constexpr bool RES = (MODE & kEpiRes) != 0, STATS = (MODE & kEpiStats) != 0, FP32 = (MODE & kEpiFp32) != 0;
  constexpr bool F32P = (MODE & kEpiF32Planar) != 0;
  constexpr int kUnitPlanes = F32P ? 4 : 2;     // 16-byte planes of one 16-channel unit of the planar output / residual
  constexpr int kPlaneShift = F32P ? 2 : 3;     // log2(channels per plane)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = warp & 3;                       // TMEM lane quarter this warp may read
  const int ew = warp - (kEpiFirst >> 5);       // 0..7
  const int half = ew >> 2;                     // which of the two warps of that quarter
  const int et = threadIdx.x - kEpiFirst;       // 0..255
  const int r = q * 32 + lane;                  // tile row == TMEM lane
  const int lh = r >> 3, lw = r & 7;
  const int n_cta = p.n_cta;
  const int n_chunks = n_cta >> 4;
  const bool split_ch = n_chunks >= 2;
  const int ch0 = split_ch ? half : 0, ch_step = split_ch ? 2 : 1;
  const int s0 = split_ch ? 0 : half, s_step = split_ch ? 1 : 2;
  const long long HW = (long long)p.H * p.W, V = (long long)p.D * HW;
  // Bias + conditioning rows: when the [B][n_pad] table fits the 512-float buffer it is loaded ONCE per CTA
  // (r01r: a per-tile global load + barrier in front of every tile cost ~1 us on the epilogue-bound layers).
  // A launch without rows gets zeros, so that the unit code has no "is there a bias" branch.
  float* cadd_tab = &sh->cadd[0][0];
  const bool cadd_table = p.B * p.n_pad <= 512;
  const float* cadd_g = cadd_rows(p);
  if (cadd_table) VDM_CADD_TABLE_FILL(cadd_tab, cadd_g, p.B, p.n_pad, p.c_out, et, kEpiThreads);
  // Residual prefetch ring in SHARED memory.  The residual does not depend on the accumulator, and a dependent
  // 16-byte global load per (unit, half) cost ~700 cycles each (r01f: 0.44 -> 0.76 ms on the 32->32 level-0 conv).
  // This warp consumes its units in a fixed order; p.res_depth of them are always in flight as cp.async copies
  // (one commit group per unit) into per-thread slots, and the prefetch cursor runs AHEAD ACROSS TILE BOUNDARIES.
  // cp.async has no destination register; the only wait is cp.async.wait_group on the oldest group.
  constexpr int kResPrefetchTiles = 3;
  const int r_depth = p.res_depth;
  uint4* r_ring = reinterpret_cast<uint4*>(smem + p.res_ring_off) + et;   // slot i, plane k: r_ring[(kUnitPlanes*i + k) * kEpiThreads]
  int r_slot = 0;                                  // oldest slot == the one refilled next (the ring is always full)
  const uint4* res_base = reinterpret_cast<const uint4*>(p.residual);
  // residual grid: the output grid, or (r_up) its half-resolution parent (coordinates shifted right by one)
  const int r_sh = p.r_up;
  const int r_H = p.H >> r_sh, r_W = p.W >> r_sh;
  const long long r_HW = (long long)r_H * r_W, r_V = (long long)(p.D >> r_sh) * r_HW;
  int r_tile = blockIdx.x - (int)gridDim.x;        // tile the prefetch cursor is in (advanced before first use)
  int ru_s = 0, ru_ch = n_chunks;                  // (slice, chunk) of the next unit to prefetch; "tile exhausted"
  const uint4* r_ptr = nullptr;
  int r_d0 = 0, r_cbase = 0;
  bool r_hw_ok = false;
  auto res_issue = [&](int slot) __attribute__((always_inline)) {
    bool live = true;
    if (ru_ch >= n_chunks) {                       // move the cursor to this CTA's next tile
      r_tile += (int)gridDim.x;
      if (r_tile < p.n_tiles) {
        const TileCoord tr = decode_tile(p, r_tile);
        const int hr = tr.h0 + lh, wr = tr.w0 + lw;
        r_hw_ok = (hr < p.H) && (wr < p.W);
        r_d0 = tr.d0;
        r_cbase = tr.ns * n_cta;
        r_ptr = res_base + ((long long)tr.b * p.r_planes + p.r_plane0 + (r_cbase >> kPlaneShift) +
                            (((hr & 1) << 1) | (wr & 1)) * p.r_d2s_planes) * r_V +
                (long long)(hr >> r_sh) * r_W + (wr >> r_sh);
        ru_s = s0; ru_ch = ch0;
      } else {
        live = false;
      }
    }
    if (live) {
      const int su = ru_s, chu = ru_ch;
      ru_s += s_step;
      if (ru_s >= MT) { ru_s = s0; ru_ch += ch_step; }
      if (r_hw_ok && r_d0 + su < p.D) {
        const uint4* src = r_ptr + (long long)(chu * kUnitPlanes + (((r_d0 + su) & 1) << 2) * p.r_d2s_planes) * r_V +
                           (long long)((r_d0 + su) >> r_sh) * r_HW;
        const int cu = r_cbase + chu * 16;
        uint4* dst = r_ring + (kUnitPlanes * slot) * kEpiThreads;
        if constexpr (F32P) {
#pragma unroll
          for (int k = 0; k < 4; ++k)
            if (cu + 4 * k < p.c_out) ptx::cp_async16(dst + k * kEpiThreads, src + k * r_V);
        } else {
          if (cu < p.c_out) ptx::cp_async16(dst, src);
          if (cu + 8 < p.c_out) ptx::cp_async16(dst + kEpiThreads, src + r_V);
        }
      }
    }
    ptx::cp_async_commit();                        // one group per unit, also when nothing was copied
  };
  if (RES) {
    for (int i = 0; i < r_depth; ++i) res_issue(i);
  }
  uint32_t ti = 0;
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++ti) {
    const TileCoord t = decode_tile(p, tile);
    const int h = t.h0 + lh, w = t.w0 + lw;
    const bool hw_ok = (h < p.H) && (w < p.W);
    const int cbase = t.ns * n_cta;
    const uint32_t acc = ti & 1;
    if (RES && p.r_d2s_planes == 0) {
      // The ring runs about one tile ahead, which covers an L2 hit but not an HBM miss (r02g).  Pull the residual rows
      // of the tile this CTA processes kResPrefetchTiles from now into L2: one 128-byte row per thread.
      const int pt = tile + kResPrefetchTiles * (int)gridDim.x;
      if (pt < p.n_tiles) {
        const TileCoord tp = decode_tile(p, pt);
        const int pc0 = tp.ns * n_cta;
        const int n_rows = (n_cta >> kPlaneShift) * MT * 16;
        const uint4* pbase = res_base + ((long long)tp.b * p.r_planes + p.r_plane0 + (pc0 >> kPlaneShift)) * r_V + (tp.w0 >> r_sh);
        for (int idx = et; idx < n_rows; idx += kEpiThreads) {
          const int hh = tp.h0 + (idx & 15);
          const int sp_ = idx >> 4;
          const int pp = sp_ / MT;
          const int dd = tp.d0 + (sp_ - pp * MT);
          if (hh < p.H && dd < p.D && pc0 + (pp << kPlaneShift) < p.c_out && !(r_sh && ((hh | dd) & 1)))
            ptx::prefetch_l2(pbase + (long long)pp * r_V + ((long long)(dd >> r_sh) * r_H + (hh >> r_sh)) * r_W);
        }
      }
    }
    const int buf = ti & 1;
    if (!cadd_table) {
      // bias + conditioning row of this sample -> shared memory, double-buffered by tile parity
      if (et < n_cta)
        sh->cadd[buf][et] = (cadd_g && cbase + et < p.c_out) ? __ldg(cadd_g + (long long)t.b * p.c_out + cbase + et) : 0.f;
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
    const float* cadd_row = cadd_tab + (cadd_table ? t.b * p.n_pad + cbase : buf * 256);
    // per-tile bases (64-bit once per tile; per unit only adds): voxel of slice 0 of this thread
    const long long vox0 = ((long long)t.d0 * p.H + h) * p.W + w;
    float* sp = stat_part + (ti & 1) * (16 * n_cta);   // this tile's partials (double-buffered by tile parity)
    ptx::mbar_wait(&sh->tmem_full[acc], (ti >> 1) & 1);
    ptx::tc_fence_after();
    const uint32_t trow0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * MT * n_cta);
    bool released = false;
    for (int ch = ch0; ch < n_chunks; ch += ch_step) {
      const int c0 = cbase + ch * 16;
      const bool last_chunk = ch + ch_step >= n_chunks;
      // valid 8-channel planes of this chunk (bf16 output: c_out % 8 == 0) / valid channels (fp32 output); warp-uniform
      const int c_left = p.c_out - c0;
      const int nhf = c_left >= 16 ? 2 : (c_left >= 8 ? 1 : 0);
      float cb[16];                              // bias + conditioning row of this chunk, for all slices of the tile
      load_row16(cadd_row + ch * 16, cb);
      float s1[16], s2[16];                      // per-lane statistics of this chunk over the warp's slices
      if (STATS) {
#pragma unroll
        for (int j = 0; j < 16; ++j) s1[j] = s2[j] = 0.f;
      }
      typename Unit<F32P>::T* y_ch = reinterpret_cast<typename Unit<F32P>::T*>(p.y) +
                                     ((long long)t.b * p.y_planes + p.y_plane0 + (c0 >> kPlaneShift)) * V + vox0;
      float* y32_ch = static_cast<float*>(p.y) + ((long long)t.b * p.c_out + c0) * V + vox0;
      auto process = [&](uint32_t (&raw)[16], int s) __attribute__((always_inline)) {
        const bool valid = hw_ok && (t.d0 + s < p.D);
        uint4 rcur0 = make_uint4(0, 0, 0, 0), rcur1 = make_uint4(0, 0, 0, 0);
        uint4 rcur2 = make_uint4(0, 0, 0, 0), rcur3 = make_uint4(0, 0, 0, 0);   // (fp32 planar: planes 2, 3 of the unit)
        if (RES) {
          // the oldest slot is this unit's residual; refill it for the unit r_depth ahead
          ptx::cp_async_wait(r_depth - 1);
          const uint4* slot = r_ring + (kUnitPlanes * r_slot) * kEpiThreads;
          rcur0 = slot[0]; rcur1 = slot[kEpiThreads];
          if (F32P) { rcur2 = slot[2 * kEpiThreads]; rcur3 = slot[3 * kEpiThreads]; }
          res_issue(r_slot);
          r_slot = (r_slot + 1 == r_depth) ? 0 : r_slot + 1;
        }
        float f[16];
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          f[j] = __uint_as_float(raw[j]); f[j + 1] = __uint_as_float(raw[j + 1]);
          add2(f[j], f[j + 1], cb[j], cb[j + 1]);
        }
        if (FP32) {
          if (valid) VDM_STORE_FP32_NCDHW(y32_ch + (long long)s * HW, f, c_left, V);
          return;
        }
        if (nhf == 0 || !valid) return;          // padded output channels (warp-uniform) / voxels beyond the grid
        typename Unit<F32P>::T* yp = y_ch + (long long)s * HW;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          if (hf == 1 && nhf < 2) break;
          if constexpr (F32P) {
            VDM_STORE_HALF_F32P(RES, STATS, f, hf, hf == 0 ? rcur0 : rcur2, hf == 0 ? rcur1 : rcur3, yp, (long long)(2 * hf) * V,
                                (long long)(2 * hf + 1) * V, s1, s2);
          } else {
            VDM_STORE_HALF_BF16(RES, STATS, f, hf, hf == 0 ? rcur0 : rcur1, yp, hf == 0 ? 0 : V, s1, s2);
          }
        }
      };
      // unit pipeline of this chunk: the TMEM load of the next slice is in flight while this one is processed
      const uint32_t tcol = trow0 + (uint32_t)(ch * 16);
      uint32_t raw_a[16], raw_b[16];
      int s = s0;
      if (s < MT) ptx::tmem_ld16(tcol + (uint32_t)(s * n_cta), raw_a);
#pragma unroll
      for (int i = 0; i < MT; ++i) {
        if (s >= MT) break;
        const int sn = s + s_step;
        if ((i & 1) == 0) {
          ptx::tmem_ld_wait_dep(raw_a);
          if (sn < MT) ptx::tmem_ld16(tcol + (uint32_t)(sn * n_cta), raw_b);
        } else {
          ptx::tmem_ld_wait_dep(raw_b);
          if (sn < MT) ptx::tmem_ld16(tcol + (uint32_t)(sn * n_cta), raw_a);
        }
        if (last_chunk && sn >= MT) {
          // every TMEM read of this accumulator set has completed (wait::ld above): hand it back before the arithmetic
          ptx::tc_fence_before();
          ptx::mbar_arrive(&sh->tmem_empty[acc]);
          released = true;
        }
        if ((i & 1) == 0) process(raw_a, s);
        else process(raw_b, s);
        s = sn;
      }
      // one transpose-reduction per chunk and tile (r01j: per (slice, chunk) it cost 0.22 -> 0.30 ms on 32->32)
      if (STATS && nhf > 0) VDM_STATS_TO_SLOTS(s1, s2, sp, ew, n_cta, ch * 16, 8, lane);
    }
    if (!released) {
      ptx::tc_fence_before();
      ptx::mbar_arrive(&sh->tmem_empty[acc]);
    }
    if (STATS) {
      // Fold this tile's per-warp fp32 partials into the CTA's fp64 running sums (fixed order: the result is
      // reproducible run to run up to the order of the final fp64 atomics); global atomics happen only when
      // this CTA moves on to another (sample, channel slice) or finishes.
      // ONE barrier per tile: the partials are double-buffered by tile parity, and the fold of tile i is ordered
      // before the writes of tile i+2 by the barrier of tile i+1 (r02i: 14% of the samples sat in two barriers).
      asm volatile("bar.sync 2, 256;" ::: "memory");
      if (et < n_cta) {
        const int next_tile = tile + (int)gridDim.x;
        bool flush = next_tile >= p.n_tiles;
        if (!flush) {
          const TileCoord tn = decode_tile(p, next_tile);
          flush = (tn.b != t.b) || (tn.ns != t.ns);
        }
        // a warp writes the slots of its own chunks only (split by chunk, padded chunks skipped): clear them as they are read
        VDM_FOLD_STATS(p, sp, stat_acc, n_cta, et, 8, 8, true, flush, t.b, cbase);
      }
    }
  }
}

// ---- generic issue schedule (wide layers, tap subsets, 1x1x1) ----------------------------------------------------------
// chunk -> weight stage (one (kd, kh) row of taps, or one tap) -> tap -> sub-tile s < MT -> k16, N = n_cta.  The issuing
// thread has ~64 cycles per MMA at N = 128: the r02 loop built every descriptor from run-time loop indices in vector
// registers (12 instructions per MMA, two of them R2UR: ~84 cycles, R3 SASS) and the wide layers sat at 66 % of the tensor
// rate while L2 ran at 8 %.  Here the run-time part is per TAP (its halo offset from the tap table, its weight block: one
// 64-bit descriptor for A and KJ for B), and the MT x KJ MMAs of a tap differ by IMMEDIATE offsets (PAD fixes the halo
// geometry at compile time): one UIADD3.64 and the UTCHMMA per MMA.
template <int MT, int KJ, int PAD, int TPS, bool RESIDENT, ptx::MmaKind KIND>
__device__ __forceinline__ void issue_generic_tiles(const ConvKernelParams& p, ConvShared* sh, uint64_t* a_rdy, uint32_t a_base16,
                                                    uint32_t b_base16, uint32_t tmem_u, bool leader) {
  constexpr uint32_t Hh = kTileH + 2 * PAD, Wh = kTileW + 2 * PAD, Hd = MT + 2 * PAD;
  constexpr uint32_t slice16 = Hh * Wh;                      // one d-slice of a plane, 16-byte units
  constexpr uint32_t kstep_a16 = 2u * Hd * Hh * Wh;          // two planes (K = 16)
  const uint32_t n_cta = hold_u32((uint32_t)p.n_cta);
  const uint32_t idesc = ptx::make_idesc_bf16<KIND>(128, n_cta);
  const uint64_t a_hi = make_planar_desc(0, Hd * Hh * Wh * 16u, Wh * 16u);
  const uint64_t b_hi = make_planar_desc(0, n_cta * 16u, 128u);
  const uint32_t a_stage16 = hold_u32((uint32_t)p.a_stage_bytes >> 4), b_stage16 = hold_u32((uint32_t)p.b_stage_bytes >> 4);
  const uint32_t kstep_b16 = 2u * n_cta;
  const uint32_t btap16 = (uint32_t)(2 * KJ) * n_cta;          // one tap inside a B stage
  constexpr int tps = TPS;                                     // taps per weight stage: one (kd, kh) row of three, or one
  constexpr bool resident = RESIDENT;                          // all weights stay in shared memory (loaded once)
  const int n_taps = (int)hold_u32((uint32_t)p.n_taps);
  const int k_chunks = (int)hold_u32((uint32_t)p.k_chunks);
  Ring ra(hold_u32((uint32_t)p.nsa)), rb(hold_u32((uint32_t)p.nsb));   // rb is advanced by the issuing lane only
  uint32_t ti = 0;
  bool first_chunk = true;
  for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++ti) {
    const uint32_t acc = ti & 1;
    ptx::mbar_wait(&sh->tmem_empty[acc], ((ti >> 1) & 1) ^ 1);
    ptx::tc_fence_after();
    const uint32_t d_tmem0 = tmem_u + acc * (uint32_t)MT * n_cta;
    for (int kc = 0; kc < k_chunks; ++kc, ra.next()) {
      const uint32_t sa = ra.s;
      ptx::mbar_wait(&a_rdy[sa], ra.ph);
      if (resident && first_chunk) ptx::mbar_wait(&sh->b_full[0], 0);
      first_chunk = false;
      ptx::tc_fence_after();
      const uint32_t a_lo0 = a_base16 + sa * a_stage16;
      // ONE elected lane runs the whole chunk, weight-stage waits included (R2k: the per-stage warp-wide wait / fence / elect /
      // __syncwarp sequence cost ~500 cycles per step)
      if (leader) {
        for (int tap0 = 0; tap0 < n_taps; tap0 += tps) {
          uint32_t b_lo0;
          if (resident) {
            b_lo0 = b_base16 + (uint32_t)(kc * n_taps + tap0) * btap16;
          } else {
            ptx::mbar_wait(&sh->b_full[rb.s], rb.ph);
            ptx::tc_fence_after();
            b_lo0 = b_base16 + rb.s * b_stage16;
          }
#pragma unroll
          for (int q = 0; q < tps; ++q) {
            const uint64_t a_tap = a_hi | (uint64_t)(a_lo0 + (uint32_t)p.tap16[tap0 + q]);
            const uint32_t first = (kc | tap0 | q) != 0 ? 1u : 0u;
            uint64_t b_tap[KJ];
#pragma unroll
            for (int j = 0; j < KJ; ++j) b_tap[j] = b_hi | (uint64_t)(b_lo0 + (uint32_t)q * btap16 + (uint32_t)j * kstep_b16);
#pragma unroll
            for (int s = 0; s < MT; ++s) {
#pragma unroll
              for (int j = 0; j < KJ; ++j)
                ptx::umma_bf16_off64<KIND>(d_tmem0, (uint32_t)s * n_cta, a_tap, (uint32_t)s * slice16 + (uint32_t)j * kstep_a16, b_tap[j],
                                           0u, idesc, j == 0 ? first : 1u);
            }
          }
          if (!resident) {
            ptx::umma_commit(&sh->b_empty[rb.s]);
            rb.next();
          }
        }
        ptx::umma_commit(&sh->a_empty[sa]);
        if (kc == k_chunks - 1) ptx::umma_commit(&sh->tmem_full[acc]);
      }
      __syncwarp();
    }
  }
}

// The dynamic shared-memory window of a conv kernel, rounded up to 1024 bytes by POINTER ARITHMETIC on the __shared__ array:
// a round trip through uintptr_t made nvcc lose the address space, and every access through the shared structures and the
// residual ring compiled to generic LD / ST (R2b ncu: LD.E.128 for the bias rows and the ring slots in the epilogue's inner loop).
__device__ __forceinline__ uint8_t* smem_window_1024(uint8_t* smem_raw) {
  return smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
}

// MT = d-slices (accumulators) per tile, KJ = K=16 MMAs per channel chunk (KC = 16*KJ), NF = 0 for the generic
// path or Cout_pad for the kd-folded path: compile-time so that the MMA issue loops are straight lines of
// tcgen05.mma with immediate offsets (r01a: a generic loop cost ~240 issue cycles per MMA).
// TF32: fp32 channel-planar activations [B][C/4][D][H][W][4] and fp32 weights [tap][Cin/4][Cout_pad][4], tcgen05.mma
// kind::tf32.  A plane is 16 bytes and a K step 32 bytes in both element types, so everything up to the accumulator
// (TMA boxes, weight copies, descriptors, the issue schedule) is that of the bf16 layer with twice the input channels;
// only the MMA kind and the epilogue's output element differ.  Generic schedule only, no fused input transform.
template <int MT, int KJ, int NF, bool TF32 = false>
__global__ void __launch_bounds__(kConvThreads, 1)
conv3d_planar_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_x2,
                     const __grid_constant__ ConvKernelParams p) {
  static_assert(!TF32 || NF == 0, "the TF32 instances run the generic schedule only");
  constexpr ptx::MmaKind kKind = TF32 ? ptx::MmaKind::kTF32 : ptx::MmaKind::kF16;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_window_1024(smem_raw);
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + (size_t)p.nsa * p.a_stage_bytes;
  ConvShared* sh = reinterpret_cast<ConvShared*>(b_smem + (size_t)p.nsb * p.b_stage_bytes + p.skip_w_bytes);
  constexpr bool kFold = NF > 0;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmap_x);
    for (int s = 0; s < kMaxAStages; ++s) {
      ptx::mbar_init(&sh->a_full[s], 1);
      ptx::mbar_init(&sh->a_empty[s], 1);
      ptx::mbar_init(&sh->a_ready[s], kXfThreads);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&sh->tmem_full[s], 1);
      ptx::mbar_init(&sh->tmem_empty[s], kEpiThreads);
    }
    for (int s = 0; s < p.nsb && s < kMaxBStages; ++s) {
      ptx::mbar_init(&sh->b_full[s], 1);
      ptx::mbar_init(&sh->b_empty[s], 1);
    }
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&sh->tmem_base, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish();
  }
  float* stat_part = reinterpret_cast<float*>(sh + 1);     // [tile parity][sum | sumsq][epilogue warp][channel of this CTA]
  double* stat_acc = reinterpret_cast<double*>(stat_part + 2 * 2 * 8 * p.n_cta);   // [sum | sumsq][channel of this CTA]
  if (warp >= 4 && warp < 12) {
    for (int i = threadIdx.x - kEpiFirst; i < 2 * p.n_cta; i += kEpiThreads) stat_acc[i] = 0.0;
    for (int i = threadIdx.x - kEpiFirst; i < 2 * 2 * 8 * p.n_cta; i += kEpiThreads) stat_part[i] = 0.f;
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = sh->tmem_base;
  constexpr int planes_per_chunk = KJ * 2;
  // the barrier the MMA issuer waits on before it reads a halo stage
  uint64_t* const a_rdy = p.in_norm ? sh->a_ready : sh->a_full;
  // Per-warpgroup register budgets (the launch gives every thread 65536 / 512 = 128): setmaxnreg is the FIRST statement
  // of each warpgroup's branch, with no control-flow merge before the role code, so that ptxas allocates each role
  // against its own budget (with the three instructions in front of a merged if-chain it compiled everything for 128
  // registers and spilled 7 KB in the epilogue).
  if (warp < 4) {
  ptx::setmaxnreg_dec<kRegsWg0>();

  if (warp == 0) {
    // ===================== A producer: halo tiles =====================
    if (lane == 0) {
      uint32_t it = 0;
      Ring ra((uint32_t)p.nsa);
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const TileCoord t = decode_tile(p, tile);
        for (int kc = 0; kc < p.k_chunks + p.skip_chunks; ++kc, ++it, ra.next()) {
          const int s = (int)ra.s;
          ptx::mbar_wait(&sh->a_empty[s], ra.ph ^ 1u);
          if (VDM_DBG(p, 2) && it >= 2) {       // experiment: no halo traffic after the pipeline fill
            ptx::mbar_arrive(&sh->a_full[s]);
            continue;
          }
          if (kc < p.k_chunks) {
            ptx::mbar_arrive_expect_tx(&sh->a_full[s], (uint32_t)(planes_per_chunk * p.plane_bytes));
            ptx::tma_load_4d(a_smem + (size_t)s * p.a_stage_bytes, &tmap_x, &sh->a_full[s], (t.w0 - p.pad + p.x_shift) * 8,
                             t.h0 - p.pad + p.x_shift, t.d0 - p.pad + p.x_shift,
                             t.b * p.x_planes + p.x_plane0 + kc * planes_per_chunk);
          } else {   // skip-path tensor (never halo-padded): the tile's own voxels, box (8 w, 16 h, MT d, planes)
            ptx::mbar_arrive_expect_tx(&sh->a_full[s], (uint32_t)(planes_per_chunk * MT * kTileH * kTileW * 16));
            ptx::tma_load_4d(a_smem + (size_t)s * p.a_stage_bytes, &tmap_x2, &sh->a_full[s], t.w0 * 8, t.h0, t.d0,
                             t.b * p.x2_planes + p.x2_plane0 + (kc - p.k_chunks) * planes_per_chunk);
          }
        }
      }
    }
  } else if (warp == 2 || warp == 3) {
    // ===================== B producer(s) =====================
    // Streamed weights: warps 2 AND 3 issue the copies, alternating stages (one thread needed ~900 cycles for the twelve
    // 1-2 KB copies of a stage the tensor core consumes in 770-1150: R4r ncu, the issuer waited for b_full 29 % of its time
    // on the 64 -> 64 layers).  Resident weights: warp 2 loads them once.
    const uint32_t pj = (uint32_t)(warp - 2);
    const bool streamed = kFold ? p.fold_streamed != 0 : p.b_resident == 0;
    if (lane == 0 && blockIdx.x < (unsigned)p.n_tiles && (pj == 0 || streamed)) {
      const uint32_t plane_copy_bytes = (uint32_t)p.n_cta * 16u;
      const int tps = p.taps_per_stage, nsb = p.nsb, n_taps = p.n_taps, k_chunks = p.k_chunks;
      const size_t tap_stride = (size_t)p.c_in8 * p.n_pad * 8, plane_stride = (size_t)p.n_pad * 8;
      if constexpr (kFold) {
       if (p.fold_streamed) {
        // one ring stage per (tile, chunk, kh, kw): [plane][2 - kd][co] (see issue_fold_stage); n_split == 1
        Ring rb((uint32_t)nsb);
        uint32_t n_st = 0;
        for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x)
          for (int kc = 0; kc < k_chunks; ++kc)
            for (int khw = 0; khw < 9; ++khw, rb.next(), ++n_st) {
              if ((n_st & 1u) != pj) continue;
              const int s = (int)rb.s;
              ptx::mbar_wait(&sh->b_empty[s], rb.ph ^ 1u);
              ptx::mbar_arrive_expect_tx(&sh->b_full[s], plane_copy_bytes * planes_per_chunk * 3u);
              uint8_t* dst = b_smem + (size_t)s * p.b_stage_bytes;
#pragma unroll
              for (int kd = 0; kd < 3; ++kd) {
                const __nv_bfloat16* src = p.w + (size_t)p.tap_of[kd][khw] * tap_stride + (size_t)kc * planes_per_chunk * plane_stride;
#pragma unroll
                for (int pl = 0; pl < planes_per_chunk; ++pl)
                  ptx::bulk_load(dst + (size_t)(pl * 3 + (2 - kd)) * plane_copy_bytes, src + (size_t)pl * plane_stride,
                                 plane_copy_bytes, &sh->b_full[s]);
              }
            }
       } else {
        // resident, kd-folded order: [chunk][khw][plane][2 - kd][co] (see issue_fold_tile); n_split == 1
        ptx::mbar_arrive_expect_tx(&sh->b_full[0], plane_copy_bytes * planes_per_chunk * (uint32_t)(n_taps * k_chunks) +
                                                       (uint32_t)p.skip_w_bytes);
        for (int kc = 0; kc < k_chunks; ++kc)
          for (int tap = 0; tap < n_taps; ++tap) {
            const int kd = p.tap_kd[tap], khw = p.tap_khw[tap];
#pragma unroll
            for (int pl = 0; pl < planes_per_chunk; ++pl)
              ptx::bulk_load(b_smem + (size_t)(((kc * 9 + khw) * planes_per_chunk + pl) * 3 + (2 - kd)) * plane_copy_bytes,
                             p.w + (size_t)tap * tap_stride + (size_t)(kc * planes_per_chunk + pl) * plane_stride,
                             plane_copy_bytes, &sh->b_full[0]);
          }
        // 1x1x1 skip-path weights: [plane][co] right after the main weights
        for (int pl = 0; pl < p.skip_chunks * planes_per_chunk; ++pl)
          ptx::bulk_load(b_smem + (size_t)p.b_stage_bytes + (size_t)pl * plane_copy_bytes, p.w2 + (size_t)pl * plane_stride,
                         plane_copy_bytes, &sh->b_full[0]);
       }
      } else if (p.b_resident) {
        // Weights fit next to the halo stages: load every (chunk, tap) once.  Per-tile weight streaming was a
        // fixed cost per tile (r01h: 0.454 -> 0.410 ms on the 32->32 layer); n_split == 1 on this path.
        const uint32_t total = plane_copy_bytes * planes_per_chunk * (uint32_t)(n_taps * k_chunks);
        ptx::mbar_arrive_expect_tx(&sh->b_full[0], total);
        for (int kc = 0; kc < k_chunks; ++kc)
          for (int tap = 0; tap < n_taps; ++tap) {
            uint8_t* dst = b_smem + (size_t)(kc * n_taps + tap) * planes_per_chunk * plane_copy_bytes;
            const __nv_bfloat16* src = p.w + (size_t)tap * tap_stride + (size_t)kc * planes_per_chunk * p.n_pad * 8;
#pragma unroll
            for (int pl = 0; pl < planes_per_chunk; ++pl)
              ptx::bulk_load(dst + (size_t)pl * plane_copy_bytes, src + (size_t)pl * plane_stride, plane_copy_bytes,
                             &sh->b_full[0]);
          }
      } else {
        // This thread has ~768 cycles per weight stage (12 MMAs of N = 128): with twelve 2 KB copies per stage and their address
        // arithmetic it took longer, and the issuer waited for b_full 27 % of its time (R4p ncu, 128 -> 128).  When the CTA
        // takes all output channels (n_split == 1) the planes of a channel chunk are contiguous for a tap, in global and in
        // shared memory alike: ONE copy per tap (three per stage); sizes and strides are loop invariants.
        Ring rb((uint32_t)nsb);
        const bool whole_rows = p.n_split == 1;
        const uint32_t stage_tx = plane_copy_bytes * (uint32_t)planes_per_chunk * (uint32_t)tps;
        const uint32_t tap_bytes = plane_copy_bytes * (uint32_t)planes_per_chunk;
        const size_t chunk_stride = (size_t)planes_per_chunk * plane_stride;         // elements between channel chunks
        const uint32_t b_stage_bytes = (uint32_t)p.b_stage_bytes;
        uint32_t n_st = 0;
        for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
          const TileCoord t = decode_tile(p, tile);
          const __nv_bfloat16* src_c = p.w + (size_t)t.ns * p.n_cta * 8;
          for (int kc = 0; kc < k_chunks; ++kc, src_c += chunk_stride) {
            const __nv_bfloat16* src = src_c;
            for (int tap0 = 0; tap0 < n_taps; tap0 += tps, rb.next(), ++n_st) {
              if ((n_st & 1u) != pj) {
                src += (size_t)tps * tap_stride;
                continue;
              }
              const uint32_t s = rb.s;
              ptx::mbar_wait(&sh->b_empty[s], rb.ph ^ 1u);
              ptx::mbar_arrive_expect_tx(&sh->b_full[s], stage_tx);
              uint8_t* dst = b_smem + (size_t)s * b_stage_bytes;
              if (whole_rows) {
                for (int q = 0; q < tps; ++q, src += tap_stride, dst += tap_bytes) ptx::bulk_load(dst, src, tap_bytes, &sh->b_full[s]);
              } else {
                for (int q = 0; q < tps; ++q, src += tap_stride)
#pragma unroll
                  for (int pl = 0; pl < planes_per_chunk; ++pl, dst += plane_copy_bytes)
                    ptx::bulk_load(dst, src + (size_t)pl * plane_stride, plane_copy_bytes, &sh->b_full[s]);
              }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // Everything the issue loops touch is warp-uniform (kernel parameters, the shared-memory window,
    // tmem_base broadcast by a shuffle) and the issuing lane is chosen with elect.sync, so ptxas keeps the
    // descriptors in uniform registers and emits back-to-back UTCHMMA.  (r01c: `if (lane == 0)` on
    // per-thread registers compiled to an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall around every MMA.)
    const uint32_t n_cta = (uint32_t)p.n_cta;
    const uint32_t a_base16 = ptx::smem_u32(a_smem) >> 4, a_stage16 = (uint32_t)p.a_stage_bytes >> 4;
    const uint32_t nsa_u = (uint32_t)p.nsa;
    const uint32_t b_base16 = ptx::smem_u32(b_smem) >> 4, b_stage16 = (uint32_t)p.b_stage_bytes >> 4;
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const bool leader = ptx::elect_one();
    // descriptor high words (LBO = plane stride = K direction, SBO = 8-row group pitch)
    const uint64_t a_hi = make_planar_desc(0, (uint32_t)p.plane_bytes, (uint32_t)p.Wh * 16u);
    if constexpr (kFold) {
      const uint64_t b_hi = make_planar_desc(0, 3u * (uint32_t)NF * 16u, 128u);
      constexpr uint32_t chunk_b16 = 9u * 2u * KJ * 3u * NF;       // one channel chunk of the folded weights, 16-byte units
      const int k_chunks = p.k_chunks;
      uint32_t ti = 0;
      if (p.fold_streamed) {
        const uint32_t a_hi32 = (uint32_t)(a_hi >> 32), b_hi32 = (uint32_t)(b_hi >> 32);
        const uint32_t a_lbo = (uint32_t)a_hi, b_lbo = (uint32_t)b_hi;       // LBO << 16: low descriptor words
        const uint32_t b_stage16 = hold_u32((uint32_t)p.b_stage_bytes >> 4);
        Ring ra(nsa_u), rb((uint32_t)p.nsb);                 // rb is advanced by the issuing lane only
        for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++ti) {
          const uint32_t acc = ti & 1;
          ptx::mbar_wait(&sh->tmem_empty[acc], ((ti >> 1) & 1) ^ 1);
          const uint32_t d_tmem0 = tmem_u + acc * (uint32_t)(MT * NF);
          for (int kc = 0; kc < k_chunks; ++kc, ra.next()) {
            const uint32_t sa = ra.s;
            ptx::mbar_wait(&a_rdy[sa], ra.ph);
            ptx::tc_fence_after();
            const uint32_t a_st = a_base16 + sa * a_stage16 + a_lbo;
            if (leader) {                      // one elected lane per chunk, weight-stage waits included (see the generic path)
              for (int khw = 0; khw < 9; ++khw, rb.next()) {
                const uint32_t sb = rb.s;
                ptx::mbar_wait(&sh->b_full[sb], rb.ph);
                ptx::tc_fence_after();
                const uint32_t kh = (uint32_t)khw / 3u, kw = (uint32_t)khw - 3u * kh;
                issue_fold_stage<MT, KJ, NF>(a_st + kh * (uint32_t)(kTileW + 2) + kw, b_base16 + sb * b_stage16 + b_lbo, a_hi32,
                                             b_hi32, d_tmem0, kc == 0 && khw == 0);
                ptx::umma_commit(&sh->b_empty[sb]);
              }
              ptx::umma_commit(&sh->a_empty[sa]);
              if (kc == k_chunks - 1) ptx::umma_commit(&sh->tmem_full[acc]);
            }
            __syncwarp();
          }
        }
      } else {
      Ring ra(nsa_u);
      for (int tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x, ++ti) {
        const uint32_t acc = ti & 1;
        ptx::mbar_wait(&sh->tmem_empty[acc], ((ti >> 1) & 1) ^ 1);
        if (ti == 0) ptx::mbar_wait(&sh->b_full[0], 0);
        const uint32_t d_tmem0 = tmem_u + acc * (uint32_t)(MT * NF);
        const int total_chunks = k_chunks + p.skip_chunks;
        for (int kc = 0; kc < total_chunks; ++kc, ra.next()) {
          const uint32_t sa = ra.s;
          ptx::mbar_wait(&a_rdy[sa], ra.ph);
          ptx::tc_fence_after();
          if (leader) {
            if (kc == 0)
              issue_fold_tile<MT, KJ, NF, true>(a_base16 + sa * a_stage16, b_base16, a_hi, b_hi, d_tmem0);
            else if (kc < k_chunks)
              issue_fold_tile<MT, KJ, NF, false>(a_base16 + sa * a_stage16, b_base16 + (uint32_t)kc * chunk_b16, a_hi, b_hi,
                                                 d_tmem0);
            else
              issue_skip_chunk<MT, KJ, NF>(a_base16 + sa * a_stage16,
                                           b_base16 + ((uint32_t)p.b_stage_bytes >> 4) + (uint32_t)(kc - k_chunks) * (2u * KJ * NF),
                                           d_tmem0);
            ptx::umma_commit(&sh->a_empty[sa]);
            if (kc == total_chunks - 1) ptx::umma_commit(&sh->tmem_full[acc]);
          }
          __syncwarp();
        }
      }
      }
    } else {
      // (pad == 0 is the 1x1x1 conv: one tap per stage; tap subsets whose count is not a multiple of three too)
      const bool res = p.b_resident != 0;
      if (!p.pad) {
        if (res) issue_generic_tiles<MT, KJ, 0, 1, true, kKind>(p, sh, a_rdy, a_base16, b_base16, tmem_u, leader);
        else issue_generic_tiles<MT, KJ, 0, 1, false, kKind>(p, sh, a_rdy, a_base16, b_base16, tmem_u, leader);
      } else if (p.taps_per_stage == 3) {
        if (res) issue_generic_tiles<MT, KJ, 1, 3, true, kKind>(p, sh, a_rdy, a_base16, b_base16, tmem_u, leader);
        else issue_generic_tiles<MT, KJ, 1, 3, false, kKind>(p, sh, a_rdy, a_base16, b_base16, tmem_u, leader);
      } else {
        if (res) issue_generic_tiles<MT, KJ, 1, 1, true, kKind>(p, sh, a_rdy, a_base16, b_base16, tmem_u, leader);
        else issue_generic_tiles<MT, KJ, 1, 1, false, kKind>(p, sh, a_rdy, a_base16, b_base16, tmem_u, leader);
      }
    }
  }
  } else if (warp >= 12) {
    // ===================== input transform (4 warps): see transform_tiles =====================
    ptx::setmaxnreg_dec<kRegsXf>();
    if constexpr (!TF32)
      if (p.in_norm) transform_tiles<MT, KJ>(p, sh, a_smem, reinterpret_cast<float*>(smem + p.xf_coef_off));
  } else {
    // ===================== epilogue (8 warps; two per TMEM lane quarter): see epilogue_tiles =====================
    ptx::setmaxnreg_inc<kRegsEpi>();
    constexpr int P = TF32 ? kEpiF32Planar : 0;     // planar output element: fp32 (TF32) or bf16
    if (p.out_fp32) epilogue_tiles<MT, kEpiFp32>(p, sh, smem, stat_part, stat_acc, tmem_base);
    else if (p.residual && p.stats) epilogue_tiles<MT, P | kEpiRes | kEpiStats>(p, sh, smem, stat_part, stat_acc, tmem_base);
    else if (p.residual) epilogue_tiles<MT, P | kEpiRes>(p, sh, smem, stat_part, stat_acc, tmem_base);
    else if (p.stats) epilogue_tiles<MT, P | kEpiStats>(p, sh, smem, stat_part, stat_acc, tmem_base);
    else epilogue_tiles<MT, P>(p, sh, smem, stat_part, stat_acc, tmem_base);
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

#include "conv3d_march.cuh"

// ---- host side ------------------------------------------------------------------------------
// Bring-up overrides of the planner, set by vdm_debug_set in `make bringup` builds.  In the release library they are a
// compile-time all-zero constant and their branches vanish.
struct ConvOverrides {
  int debug_flags;                       // ConvKernelParams::debug_flags (ablation experiments: results are wrong)
  int force_mt, force_kc, force_nsplit;  // > 0: replaces the planned value (force_mt / force_nsplit also rule out kd-folding)
  int no_resident;                       // generic schedule: stream the weights even where they fit shared memory
  int no_fold;                           // no kd-folded (nor marching) schedule
  int no_march;                          // the tile kernel's kd-folded schedule instead of the marching one
};
#ifdef VDM_BRINGUP
static ConvOverrides g_overrides = {};
#else
constexpr ConvOverrides g_overrides = {};
#endif

enum class ConvSchedule {
  kTile,           // conv3d_planar_kernel<MT, KJ, 0>: generic tap loop
  kFoldResident,   // conv3d_planar_kernel<MT, KJ, NF>: kd folded into N, all weights resident in shared memory
  kFoldStreamed,   // conv3d_planar_kernel<4, 2, 64>: kd folded into N, weights streamed per (chunk, kh, kw)
  kMarch,          // conv3d_march_kernel (conv3d_march.cuh): kd-folded resident layers whose input channels are one chunk
};

struct ConvPlan {
  ConvSchedule schedule;
  int pad;                        // 1 when a tap reads a neighbour voxel (one-voxel halo), else 0
  int mt, kc, n_split, n_cta;     // d-slices per tile, channels per chunk, CTAs per spatial tile and their UMMA N
  int n_tiles, grid;
  int nsa, nsb, taps_per_stage;   // halo stages, weight stages, filter taps per weight stage
  int a_stage_bytes, b_stage_bytes, b_resident;
  int res_depth, res_ring_off;    // residual units in flight per epilogue thread, byte offset of their ring
  int xf_coef_off;                // byte offset of the fused input transform's (a, b) table
  size_t smem_bytes;              // dynamic shared memory of the launch
  int m_units, m_nseg, m_seglen;  // marching schedule: units = columns x d-segments of m_seglen slices
  int debug_flags;
};

// Cell kd * 9 + kh * 3 + kw of tap t in the 3x3x3 stencil.
static int tap_cell(const VdmConvDesc& d, int t) {
  return (d.tap_offset[t][0] + 1) * 9 + (d.tap_offset[t][1] + 1) * 3 + d.tap_offset[t][2] + 1;
}

// Launch plan of one conv layer: schedule, tiling, pipeline depths and shared-memory layout.  Host arithmetic only (the
// descriptor's ranges are checked by the caller); returns VDM_OK, or the code and message the layer is refused with.
// A TF32 layer is planned as the byte-identical bf16 layer (`d` with twice its input channels) on the generic schedule;
// its residual units are twice as large.
static int plan_conv(const VdmConvDesc& d, bool has_residual, bool has_skip, bool has_xf, int skip_c_in, int sms, bool tf32,
                     ConvPlan& pl) {
  const ConvOverrides& ov = g_overrides;
  pl = ConvPlan{};
  pl.debug_flags = ov.debug_flags;
  int pad = 0;
  for (int t = 0; t < d.n_taps; ++t)
    if (d.tap_offset[t][0] != 0 || d.tap_offset[t][1] != 0 || d.tap_offset[t][2] != 0) pad = 1;
  if (has_xf && d.circular) {
    set_error("vdm_conv3d: the fused input transform is not available with circular padding");
    return VDM_E_UNSUPPORTED;
  }
  if (has_skip && (skip_c_in > 64 || d.out_fp32)) {
    set_error("vdm_conv3d: the fused skip conv supports bf16 layers with skip_c_in <= 64 only (got %d)", skip_c_in);
    return VDM_E_UNSUPPORTED;
  }
  const int xf_bytes = has_xf ? ((d.c_in * 8 + 15) & ~15) : 0;      // (a, b) table of one sample
  const int res_slot = tf32 ? 2 * kResSlotBytes : kResSlotBytes;     // one residual unit for every epilogue thread
  const int skip_w_bytes = has_skip ? skip_c_in * d.c_out_pad * 2 : 0;

  // ---- schedule ----
  // kd-folded schedules (issue_fold_tile): the full 3x3x3 stencil on a narrow layer
  bool fold = !tf32 && d.n_taps == 27 && pad == 1 && (d.c_out_pad == 16 || d.c_out_pad == 32 || d.c_out_pad == 64) && d.depth >= 3 &&
              ov.no_fold == 0 && ov.force_mt == 0 && ov.force_nsplit == 0;
  const bool streamed = d.c_out_pad == 64;
  int fold_mt = 0, fold_kc = 0;
  if (fold && streamed) {
    // N = 3*64: weights streamed per (chunk, kh, kw); MT = 4 (2 x 4 x 64 = all 512 TMEM columns), 32-channel chunks
    fold = d.c_in % 32 == 0 && d.depth >= 4;
    fold_mt = 4; fold_kc = 32;
  } else if (fold) {
    // all weights resident + two halo stages must fit; prefer tall tiles (halo efficiency), then wide chunks
    const int budget = 227 * 1024 - 1024 - (int)sizeof(ConvShared) - (2 * 2 * 8 * d.c_out_pad * 4 + 2 * d.c_out_pad * 8) - 256 -
                       (has_residual ? 2 * res_slot : 0) - xf_bytes;      // room for at least two residual slots
    const int w_bytes = 27 * d.c_in * d.c_out_pad * 2 + skip_w_bytes;
    for (int m = 4; m >= 2 && !fold_mt; --m)
      for (int c = 32; c >= 16 && !fold_mt; c -= 16) {
        if (d.c_in % c != 0 || (has_skip && skip_c_in % c != 0)) continue;
        const int a_stage = (((c / 8) * (m + 2) * (kTileH + 2) * (kTileW + 2) * 16) + 127) & ~127;
        if (2 * a_stage + w_bytes <= budget) { fold_mt = m; fold_kc = c; }
      }
    // (r02j: re-streaming the weights per tile so that a 96 -> 32 layer could use MT = 4 tiles instead of MT = 2 was
    // slower, 4.42 vs 3.05 ms at 128^3 x 8: the 6 KB (chunk, kh, kw) stages are dominated by their hand-off cost.)
    fold = fold_mt != 0;
  }
  if (fold) {   // every cell of the stencil exactly once
    unsigned seen = 0;
    for (int t = 0; t < 27; ++t) seen |= 1u << tap_cell(d, t);
    fold = seen == (1u << 27) - 1u;
  }
  pl.schedule = !fold ? ConvSchedule::kTile : streamed ? ConvSchedule::kFoldStreamed
              : d.c_in == fold_kc && ov.no_march == 0 ? ConvSchedule::kMarch : ConvSchedule::kFoldResident;
  const bool resident_fold = pl.schedule == ConvSchedule::kFoldResident || pl.schedule == ConvSchedule::kMarch;

  // ---- tiling ----
  const int tiles_w = ceil_div(d.width, kTileW), tiles_h = ceil_div(d.height, kTileH);
  int n_split = 1, mt = fold_mt;
  if (!fold) {
    // Pick (n_split, MT) with a small cost model: a CTA tile costs max(tensor time, L2->SM time) and the
    // grid runs in ceil(tiles / SMs) waves.  n_split shares one spatial tile between CTAs that each
    // compute c_out_pad / n_split output channels (more CTAs for the coarse levels); MT d-slices
    // per tile amortise the halo and the weight stream (fewer, fatter tiles).
    double best = -1.0;
    for (int ns = 1; ns <= 8; ns *= 2) {
      if (d.c_out_pad % (ns * 16) != 0) break;
      const int ncta = d.c_out_pad / ns;
      if (ns > 1 && ncta < 32) break;
      int mt_max = 256 / ncta;
      if (mt_max > 4) mt_max = 4;
      if (mt_max > d.depth) mt_max = d.depth;
      for (int m = 1; m <= mt_max; ++m) {
        const long long tiles = (long long)tiles_w * tiles_h * ceil_div(d.depth, m) * d.batch * ns;
        const long long waves = (tiles + sms - 1) / sms;
        const double active = (double)(tiles < sms ? tiles : sms);
        // one MMA (M = 128, K = 16): max(tensor time N/2, shared-memory operand fetch (4 KB of A + 32 B per row of B) at
        // 128 B/clk): N = 32 / 64 are fetch-bound (40 / 48 cycles), N >= 128 tensor-bound (R2r sweep: with the old
        // max(N/2, 24) the model preferred N = 64, MT = 4 over N = 128, MT = 2 and lost ~15% on every wide layer)
        const double fetch_cyc = 32.0 + ncta / 4.0;
        const double mma_cyc = (double)d.n_taps * (d.c_in / 16) * m * (ncta / 2.0 > fetch_cyc ? ncta / 2.0 : fetch_cyc);
        const double bytes = (double)(m + 2 * pad) * (kTileH + 2 * pad) * (kTileW + 2 * pad) * d.c_in * 2.0 +
                             (double)d.n_taps * d.c_in * ncta * 2.0;
        double bw = 5500.0 / active;  // L2 -> SM bytes per cycle per SM when `active` SMs pull at once
        if (bw > 64.0) bw = 64.0;
        const double cyc = (mma_cyc > bytes / bw ? mma_cyc : bytes / bw) + 2000.0;  // + per-tile fixed cost
        const double total = (double)waves * cyc;
        if (best < 0.0 || total < best * 0.999) {
          best = total;
          n_split = ns;
          mt = m;
        }
      }
    }
  }
  if (ov.force_nsplit > 0) n_split = ov.force_nsplit;
  VDM_CHECK_ARG(d.c_out_pad % (n_split * 16) == 0, "vdm_conv3d: n_split=%d does not divide c_out_pad=%d", n_split,
                d.c_out_pad);
  const int n_cta = d.c_out_pad / n_split;
  if (ov.force_mt > 0) mt = ov.force_mt;
  VDM_CHECK_ARG(mt >= 1 && 2 * mt * n_cta <= 512, "vdm_conv3d: MT=%d does not fit TMEM with N=%d", mt, n_cta);
  const long long n_tiles = (long long)tiles_w * tiles_h * ceil_div(d.depth, mt) * d.batch * n_split;
  VDM_CHECK_ARG(n_tiles < (1ll << 31), "vdm_conv3d: too many tiles");
  if (has_skip && !resident_fold) {
    set_error("vdm_conv3d: the fused skip conv needs the kd-folded schedule with resident weights "
              "(3x3x3, c_out_pad 16 or 32, weights + skip weights fit shared memory); c_in=%d c_out=%d", d.c_in, d.c_out);
    return VDM_E_UNSUPPORTED;
  }
  pl.pad = pad; pl.mt = mt; pl.n_split = n_split; pl.n_cta = n_cta; pl.n_tiles = (int)n_tiles;
  pl.taps_per_stage = (d.n_taps % 3 == 0) ? 3 : 1;   // one (kd, kh) row of filter taps per weight stage

  if (pl.schedule == ConvSchedule::kMarch) {
    // Segment length: static round-robin over equal units, so the launch takes ceil(units / SMs) rounds of (seglen + 2) slices
    // (+1: per-unit fixed costs); short segments balance the SMs, long ones amortise the two halo slices.
    const long long cols = (long long)d.batch * tiles_h * tiles_w;
    int nseg_best = 1;
    double best = -1.0;
    for (int nseg = 1; nseg <= ceil_div(d.depth, 4); ++nseg) {
      const int seglen = ceil_div(d.depth, nseg);
      if (ceil_div(d.depth, seglen) != nseg) continue;
      const long long rounds = (cols * nseg + sms - 1) / sms;
      const double cost = (double)rounds * (seglen + 3);
      if (best < 0.0 || cost < best * 0.999) { best = cost; nseg_best = nseg; }
    }
    const long long units = cols * nseg_best;
    VDM_CHECK_ARG(units < (1ll << 31), "vdm_conv3d: too many units");
    pl.kc = fold_kc;
    pl.m_nseg = nseg_best;
    pl.m_seglen = ceil_div(d.depth, nseg_best);
    pl.m_units = (int)units;
    const int stage_bytes = (fold_kc / 8) * (kTileH + 2) * (kTileW + 2) * 16;
    int off = kMarchStages * stage_bytes + 27 * (fold_kc / 8) * n_cta * 16 + skip_w_bytes + (int)sizeof(MarchShared) +
              2 * kMEpiWarps * n_cta * 4 + 2 * n_cta * 8 + kMarchCaddMax * 4;
    off = (off + 15) & ~15;
    if (has_residual) {
      pl.res_ring_off = off;
      pl.res_depth = kMarchResDepth;
      off += kMarchResDepth * (n_cta / 8) * kMEpiThreads * 16;
    }
    pl.smem_bytes = (size_t)off + 1024;
    VDM_CHECK_ARG(pl.smem_bytes <= 227 * 1024, "vdm_conv3d: marching layer does not fit shared memory");
    pl.grid = pl.m_units < sms ? pl.m_units : sms;
    return VDM_OK;
  }

  // ---- shared memory plan: halo stages + weights (resident, or a ring of stages) + residual ring ----
  const int plane_bytes = (mt + 2 * pad) * (kTileH + 2 * pad) * (kTileW + 2 * pad) * 16;
  const int stat_part_bytes = 2 * 2 * 8 * n_cta * 4 + 2 * n_cta * 8;    // partials + running sums
  const int smem_total = 227 * 1024 - 1024 /*alignment slack*/ - (int)sizeof(ConvShared) - stat_part_bytes - 256 - xf_bytes;
  // layers with a residual keep a cp.async ring of it in shared memory: 4 units deep where the weights are streamed
  // anyway, at least 2 where they are resident (the fold search above left room)
  const int smem_budget = smem_total - (has_residual ? (resident_fold ? 2 : 4) * res_slot : 0);
  if (fold) {
    pl.kc = fold_kc;
    pl.a_stage_bytes = ((fold_kc / 8) * plane_bytes + 127) & ~127;
  }
  if (pl.schedule == ConvSchedule::kFoldStreamed) {
    pl.b_stage_bytes = 3 * fold_kc * n_cta * 2;
    pl.nsb = (smem_budget - 2 * pl.a_stage_bytes) / pl.b_stage_bytes;
    if (pl.nsb > kMaxBStages) pl.nsb = kMaxBStages;
    VDM_CHECK_ARG(pl.nsb >= 2, "vdm_conv3d: folded streamed layer does not fit shared memory");
  } else if (pl.schedule == ConvSchedule::kFoldResident) {
    pl.b_stage_bytes = d.n_taps * d.c_in * n_cta * 2;
    pl.nsb = 1;
    pl.b_resident = 1;
    VDM_CHECK_ARG(2 * pl.a_stage_bytes + pl.b_stage_bytes + skip_w_bytes <= smem_budget,
                  "vdm_conv3d: folded layer does not fit shared memory");
  } else {
    for (int c : {64, 32, 16}) {   // the widest channel chunk for which two halo and two weight stages fit
      if ((ov.force_kc > 0 && c != ov.force_kc) || d.c_in % c != 0) continue;
      const int a_stage = ((c / 8) * plane_bytes + 127) & ~127;
      const int b_stage = pl.taps_per_stage * c * n_cta * 2;
      const int room = smem_budget - 2 * a_stage;
      if (room < 2 * b_stage) continue;
      const long long all_b = (long long)d.n_taps * d.c_in * n_cta * 2;
      pl.kc = c;
      pl.a_stage_bytes = a_stage;
      pl.b_stage_bytes = b_stage;
      pl.b_resident = (n_split == 1 && all_b <= room && ov.no_resident == 0) ? 1 : 0;
      pl.nsb = pl.b_resident ? (int)((all_b + b_stage - 1) / b_stage) : (room / b_stage > kMaxBStages ? kMaxBStages : room / b_stage);
      break;
    }
    VDM_CHECK_ARG(pl.kc > 0, "vdm_conv3d: no channel-chunk size fits shared memory (c_in=%d, N=%d, MT=%d)", d.c_in, n_cta, mt);
  }
  VDM_CHECK_ARG(plane_bytes <= 0x3FFF * 16, "vdm_conv3d: halo plane too large for the descriptor stride field");

  // Halo stages: two are planned above; layers whose weights leave room get up to kMaxAStages.  A TMA box takes
  // several thousand cycles to arrive from L2 / HBM, and where a chunk's MMAs are shorter than that (conv_in: 54 MMAs per
  // tile, the 1x1x1 convs) two stages left the tensor core waiting for loads.
  const int fixed = pl.nsb * pl.b_stage_bytes + skip_w_bytes + (has_residual ? 4 * res_slot : 0);
  pl.nsa = 2;
  while (pl.nsa < kMaxAStages && (pl.nsa + 1) * pl.a_stage_bytes + fixed <= smem_total) ++pl.nsa;
  const int used = pl.nsa * pl.a_stage_bytes + pl.nsb * pl.b_stage_bytes + skip_w_bytes;
  if (has_residual) {
    const int depth = (smem_total - used) / res_slot;
    pl.res_depth = depth > 4 ? 4 : depth;
    VDM_CHECK_ARG(pl.res_depth >= 1, "vdm_conv3d: no shared memory left for the residual ring");
    pl.res_ring_off = (used + (int)sizeof(ConvShared) + stat_part_bytes + 15) & ~15;
  }
  pl.xf_coef_off = (used + (int)sizeof(ConvShared) + stat_part_bytes + 16 + pl.res_depth * res_slot + 15) & ~15;
  pl.smem_bytes = (size_t)pl.xf_coef_off + xf_bytes + 1024;
  pl.grid = pl.n_tiles < sms ? pl.n_tiles : sms;
  return VDM_OK;
}

// The kernel instance of a plan.  Every instance compiled into the library is listed here.
static int launch_conv(const ConvPlan& pl, const CUtensorMap& tmx, const CUtensorMap& tmx2, const ConvKernelParams& p,
                       bool tf32, cudaStream_t stream) {
  if (pl.schedule == ConvSchedule::kMarch) {
    const bool sk = p.skip_chunks > 0, xf = p.in_norm != nullptr;
#define VDM_MARCH(KJv, NFv, SKv, XFv)                                                                          \
    if (pl.kc == 16 * KJv && pl.n_cta == NFv && sk == SKv && xf == XFv)                                        \
      return launch_kernel<conv3d_march_kernel<KJv, NFv, SKv, XFv>>(pl.grid, kConvThreads, pl.smem_bytes, stream, tmx, tmx2, p);
#define VDM_MARCH4(SKv, XFv) VDM_MARCH(1, 16, SKv, XFv) VDM_MARCH(1, 32, SKv, XFv) VDM_MARCH(2, 16, SKv, XFv) VDM_MARCH(2, 32, SKv, XFv)
    VDM_MARCH4(false, false) VDM_MARCH4(true, false) VDM_MARCH4(false, true) VDM_MARCH4(true, true)
#undef VDM_MARCH4
#undef VDM_MARCH
    set_error("vdm_conv3d: no marching kernel instance for KC=%d N=%d", pl.kc, pl.n_cta);
    return VDM_E_UNSUPPORTED;
  }
  const int nf = pl.schedule == ConvSchedule::kTile ? 0 : pl.n_cta;
  if (tf32) {
#define VDM_TILE_TF32(MTv, KJv)                                                                                \
    if (pl.mt == MTv && pl.kc == 16 * KJv && nf == 0)                                                          \
      return launch_kernel<conv3d_planar_kernel<MTv, KJv, 0, true>>(pl.grid, kConvThreads, pl.smem_bytes, stream, tmx, tmx2, p);
    VDM_TILE_TF32(1, 1) VDM_TILE_TF32(1, 2) VDM_TILE_TF32(1, 4)
    VDM_TILE_TF32(2, 1) VDM_TILE_TF32(2, 2) VDM_TILE_TF32(2, 4)
    VDM_TILE_TF32(3, 1) VDM_TILE_TF32(3, 2) VDM_TILE_TF32(3, 4)
    VDM_TILE_TF32(4, 1) VDM_TILE_TF32(4, 2) VDM_TILE_TF32(4, 4)
#undef VDM_TILE_TF32
    set_error("vdm_conv3d_tf32: no kernel instance for MT=%d KC=%d", pl.mt, pl.kc / 2);
    return VDM_E_UNSUPPORTED;
  }
#define VDM_TILE(MTv, KJv, NFv)                                                                                \
  if (pl.mt == MTv && pl.kc == 16 * KJv && nf == NFv)                                                          \
    return launch_kernel<conv3d_planar_kernel<MTv, KJv, NFv>>(pl.grid, kConvThreads, pl.smem_bytes, stream, tmx, tmx2, p);
  VDM_TILE(1, 1, 0) VDM_TILE(1, 2, 0) VDM_TILE(1, 4, 0)
  VDM_TILE(2, 1, 0) VDM_TILE(2, 2, 0) VDM_TILE(2, 4, 0)
  VDM_TILE(3, 1, 0) VDM_TILE(3, 2, 0) VDM_TILE(3, 4, 0)
  VDM_TILE(4, 1, 0) VDM_TILE(4, 2, 0) VDM_TILE(4, 4, 0)
  VDM_TILE(4, 1, 16) VDM_TILE(4, 1, 32) VDM_TILE(4, 2, 16) VDM_TILE(4, 2, 32) VDM_TILE(4, 2, 64)
  VDM_TILE(3, 1, 16) VDM_TILE(3, 1, 32) VDM_TILE(3, 2, 16) VDM_TILE(3, 2, 32)
  VDM_TILE(2, 1, 16) VDM_TILE(2, 1, 32) VDM_TILE(2, 2, 16) VDM_TILE(2, 2, 32)
#undef VDM_TILE
  set_error("vdm_conv3d: no kernel instance for MT=%d KC=%d", pl.mt, pl.kc);
  return VDM_E_UNSUPPORTED;
}

}  // namespace vdm

using namespace vdm;

#ifdef VDM_BRINGUP
extern "C" int vdm_debug_set(int key, int value) {
  switch (key) {
    case 0: return VDM_OK;   /* retired knob (LBO/SBO swap) */
    case 1: g_overrides.force_mt = value; return VDM_OK;
    case 2: g_overrides.force_kc = value; return VDM_OK;
    case 3: g_overrides.force_nsplit = value; return VDM_OK;
    case 4: g_overrides.no_resident = value; return VDM_OK;
    case 5: g_overrides.debug_flags = value; return VDM_OK;
    case 6: g_overrides.no_fold = value; return VDM_OK;
    case 7: g_overrides.no_march = value; return VDM_OK;
    default: set_error("vdm_debug_set: unknown key %d", key); return VDM_E_BADARG;
  }
}
#endif

// vdm_conv3d, and vdm_conv3d_tf32 with `d` describing the byte-identical bf16 layer (see plan_conv).
static int conv3d_run(const VdmConvDesc& d, const void* x, const void* w, void* y, const VdmConvEpilogue* epi, bool tf32,
                      cudaStream_t stream) {
  VDM_CHECK_ARG(d.batch >= 1 && d.depth >= 1 && d.height >= 1 && d.width >= 1, "vdm_conv3d: bad grid");
  VDM_CHECK_ARG(d.c_in >= 16 && d.c_in % 16 == 0, "vdm_conv3d: c_in=%d must be a multiple of 16", d.c_in);
  VDM_CHECK_ARG(d.c_out_pad >= 16 && d.c_out_pad % 16 == 0 && d.c_out_pad <= 256,
                "vdm_conv3d: c_out_pad=%d must be a multiple of 16 in [16,256]", d.c_out_pad);
  VDM_CHECK_ARG(d.c_out >= 1 && d.c_out <= d.c_out_pad, "vdm_conv3d: c_out=%d vs c_out_pad=%d", d.c_out, d.c_out_pad);
  VDM_CHECK_ARG(d.out_fp32 || d.c_out % 8 == 0, "vdm_conv3d: bf16 planar output needs c_out %% 8 == 0 (got %d)", d.c_out);
  VDM_CHECK_ARG(d.n_taps >= 1 && d.n_taps <= VDM_MAX_TAPS, "vdm_conv3d: n_taps=%d", d.n_taps);
  const int halo = d.circular ? 1 : 0;      // x carries a one-voxel periodic halo: padded dims, coordinates shifted by one
  const int x_planes = d.x_planes > 0 ? d.x_planes : d.c_in / 8;
  const int y_planes = d.y_planes > 0 ? d.y_planes : (d.c_out + 7) / 8;
  VDM_CHECK_ARG(d.x_plane0 >= 0 && d.x_plane0 + d.c_in / 8 <= x_planes, "vdm_conv3d: x plane window out of range");
  VDM_CHECK_ARG(d.out_fp32 || (d.y_plane0 >= 0 && d.y_plane0 + d.c_out / 8 <= y_planes),
                "vdm_conv3d: y plane window out of range");
  VDM_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(w) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(y) & 15) == 0,
                "vdm_conv3d: pointers must be 16-byte aligned");
  VDM_CHECK_ARG((long long)d.batch * x_planes < (1ll << 31), "vdm_conv3d: too many planes");
  for (int t = 0; t < d.n_taps; ++t)
    for (int k = 0; k < 3; ++k)
      VDM_CHECK_ARG(d.tap_offset[t][k] >= -1 && d.tap_offset[t][k] <= 1, "vdm_conv3d: tap offset out of range");
  const bool has_residual = epi && epi->residual;
  const bool has_skip = epi && epi->skip_x;
  const bool has_xf = epi && epi->in_norm;
  VDM_CHECK_ARG(!has_skip || (epi->skip_w && epi->skip_c_in >= 16 && epi->skip_c_in % 16 == 0),
                "vdm_conv3d: fused skip conv needs packed weights and skip_c_in a multiple of 16, got %d", epi->skip_c_in);
  if (!encode_fn()) {
    set_error("vdm_conv3d: cuTensorMapEncodeTiled is not available from the driver");
    return VDM_E_DRIVER;
  }

  ConvPlan pl;
  const int rc = plan_conv(d, has_residual, has_skip, has_xf, has_skip ? epi->skip_c_in : 0, num_sms(), tf32, pl);
  if (rc != VDM_OK) return rc;
  // (checked after planning: a layer the planner refuses reports VDM_E_UNSUPPORTED, which callers answer with a fallback)
  const int x2_planes = !has_skip ? 0 : epi->skip_planes > 0 ? epi->skip_planes : epi->skip_c_in / 8;
  VDM_CHECK_ARG(!has_skip || (epi->skip_plane0 >= 0 && epi->skip_plane0 + epi->skip_c_in / 8 <= x2_planes),
                "vdm_conv3d: skip plane window out of range");
  VDM_CHECK_ARG(!(epi && epi->stats && d.out_fp32), "vdm_conv3d: stats are only produced for bf16 outputs");
  VDM_CHECK_ARG(!(has_residual && d.out_fp32), "vdm_conv3d: residual is only supported for bf16 outputs");
  VDM_CHECK_ARG(!(has_residual && epi->residual_upsample) || (d.depth % 2 == 0 && d.height % 2 == 0 && d.width % 2 == 0),
                "vdm_conv3d: an up-sampled residual needs an even grid, got (%d,%d,%d)", d.depth, d.height, d.width);
  const bool march = pl.schedule == ConvSchedule::kMarch;

  ConvKernelParams p;
  memset(&p, 0, sizeof(p));
  p.B = d.batch; p.D = d.depth; p.H = d.height; p.W = d.width;
  p.c_out = d.c_out; p.n_pad = d.c_out_pad; p.n_taps = d.n_taps; p.pad = pl.pad;
  p.n_split = pl.n_split; p.n_cta = pl.n_cta;
  p.MT = pl.mt; p.KC = pl.kc; p.k_chunks = d.c_in / pl.kc;
  p.tiles_w = ceil_div(d.width, kTileW); p.tiles_h = ceil_div(d.height, kTileH); p.tiles_d = ceil_div(d.depth, pl.mt);
  p.n_tiles = pl.n_tiles;
  p.fast_div_ok = pl.n_tiles < (1 << 22) ? 1 : 0;
  p.inv_n_split = 1.0f / (float)pl.n_split; p.inv_tiles_w = 1.0f / (float)p.tiles_w;
  p.inv_tiles_h = 1.0f / (float)p.tiles_h; p.inv_tiles_d = 1.0f / (float)p.tiles_d;
  p.Hd = pl.mt + 2 * pl.pad; p.Hh = kTileH + 2 * pl.pad; p.Wh = kTileW + 2 * pl.pad;
  p.plane_bytes = p.Hd * p.Hh * p.Wh * 16;
  for (int t = 0; t < d.n_taps; ++t)
    p.tap16[t] = (uint16_t)(((d.tap_offset[t][0] + pl.pad) * p.Hh + (d.tap_offset[t][1] + pl.pad)) * p.Wh + d.tap_offset[t][2] + pl.pad);
  if (pl.schedule != ConvSchedule::kTile)
    for (int t = 0; t < 27; ++t) {
      const int c = tap_cell(d, t);
      p.tap_kd[t] = (int8_t)(c / 9);
      p.tap_khw[t] = (int8_t)(c % 9);
      p.tap_of[c / 9][c % 9] = (int8_t)t;
    }
  p.fold_streamed = pl.schedule == ConvSchedule::kFoldStreamed ? 1 : 0;
  p.nsa = pl.nsa; p.nsb = pl.nsb; p.taps_per_stage = pl.taps_per_stage;
  p.a_stage_bytes = pl.a_stage_bytes; p.b_stage_bytes = pl.b_stage_bytes; p.b_resident = pl.b_resident;
  int cols = 32;
  while (cols < 2 * pl.mt * pl.n_cta) cols <<= 1;
  p.tmem_cols = cols;
  p.c_in = d.c_in; p.c_in8 = d.c_in / 8;
  p.x_planes = x_planes; p.x_plane0 = d.x_plane0;
  p.x_shift = halo;
  if (has_skip) {
    p.skip_chunks = epi->skip_c_in / pl.kc;
    p.skip_w_bytes = epi->skip_c_in * d.c_out_pad * 2;
    p.w2 = static_cast<const __nv_bfloat16*>(epi->skip_w);
    p.x2_planes = x2_planes;
    p.x2_plane0 = epi->skip_plane0;
  }
  p.w = static_cast<const __nv_bfloat16*>(w);
  p.y = y; p.y_planes = y_planes; p.y_plane0 = d.y_plane0; p.out_fp32 = d.out_fp32;
  if (epi) {
    p.chan_add = epi->chan_add;
    p.step_ptr = epi->step_ptr;
    p.chan_add_step_stride = epi->chan_add_step_stride;
    p.residual = static_cast<const __nv_bfloat16*>(epi->residual);
    p.r_planes = d.r_planes > 0 ? d.r_planes : d.c_out / 8;
    p.r_plane0 = d.r_plane0;
    p.r_up = (epi->residual && epi->residual_upsample) ? 1 : 0;
    p.r_d2s_planes = (epi->residual && epi->residual_upsample == 2) ? d.c_out / 8 : 0;
    p.stats = epi->stats;
    p.stats_channels = epi->stats_channels > 0 ? epi->stats_channels : d.c_out;
    p.stats_c0 = epi->stats_c0;
    p.in_norm = epi->in_norm;   // fused GroupNorm + SiLU of the input (warps 12..15)
  }
  p.res_depth = pl.res_depth; p.res_ring_off = pl.res_ring_off; p.xf_coef_off = pl.xf_coef_off;
  p.m_units = pl.m_units; p.m_nseg = pl.m_nseg; p.m_seglen = pl.m_seglen;
  p.debug_flags = pl.debug_flags;

  // activations: 4-D (W*8 channels-in-plane, H, D, B*planes), box (Wh*8, Hh, Hd, KC/8); out-of-bounds -> zeros.
  // The (w, 8ch) pair is ONE tensor-map dimension on purpose: the TMA unit issues requests per
  // innermost box row, and a 16-byte row (8 channels as their own dimension) capped the r01 kernel at
  // one 32-byte sector per ~9 cycles per SM (profiles/r01_conv_ncu.txt).  Rows are Wh*16 = 160 bytes now.
  // The marching kernel loads one d-slice per stage.
  const uint32_t box_d = march ? 1u : (uint32_t)p.Hd, planes = (uint32_t)(pl.kc / 8);
  CUtensorMap tmx, tmx2;
  int e = encode_planar(&tmx, x, d.width + 2 * halo, d.height + 2 * halo, d.depth + 2 * halo, (uint64_t)d.batch * x_planes,
                        0, {(uint32_t)p.Wh, (uint32_t)p.Hh, box_d, planes}, "vdm_conv3d", march ? "x, marching" : "x");
  if (e != VDM_OK) return e;
  tmx2 = tmx;
  if (has_skip) {   // fused 1x1x1 skip conv: the tile's own voxels, no halo
    e = encode_planar(&tmx2, epi->skip_x, d.width, d.height, d.depth, (uint64_t)d.batch * x2_planes, 0,
                      {(uint32_t)kTileW, (uint32_t)kTileH, march ? 1u : (uint32_t)pl.mt, planes}, "vdm_conv3d",
                      march ? "skip_x, marching" : "skip_x");
    if (e != VDM_OK) return e;
  }
  return launch_conv(pl, tmx, tmx2, p, tf32, stream);
}

extern "C" int vdm_conv3d(const VdmConvDesc* desc, const void* x, const void* w, void* y,
                          const VdmConvEpilogue* epi, void* stream) {
  VDM_CHECK_ARG(desc && x && w && y, "vdm_conv3d: NULL pointer argument");
  return conv3d_run(*desc, x, w, y, epi, false, (cudaStream_t)stream);
}

extern "C" int vdm_conv3d_tf32(const VdmConvDesc* desc, const void* x, const void* w, void* y,
                               const VdmConvEpilogue* epi, void* stream) {
  VDM_CHECK_ARG(desc && x && w && y, "vdm_conv3d_tf32: NULL pointer argument");
  const VdmConvDesc& d = *desc;
  VDM_CHECK_ARG(d.c_in >= 8 && d.c_in % 8 == 0 && d.c_in <= 4096, "vdm_conv3d_tf32: c_in=%d must be a multiple of 8", d.c_in);
  if (epi && (epi->in_norm || epi->skip_x || (epi->residual && epi->residual_upsample))) {
    set_error("vdm_conv3d_tf32: the fused input transform, the fused skip conv and the up-sampled residual are bf16-only");
    return VDM_E_UNSUPPORTED;
  }
  // Planes are 4 fp32 channels: the layer is the bf16 layer of 2 c_in channels; output and residual windows are counted
  // in 4-channel planes here, so they are resolved before the bf16 checks see them.
  VdmConvDesc d2 = d;
  d2.c_in = 2 * d.c_in;
  if (!d.out_fp32) {
    d2.y_planes = d.y_planes > 0 ? d.y_planes : (d.c_out + 3) / 4;
    VDM_CHECK_ARG(d.y_plane0 >= 0 && d.y_plane0 + d.c_out / 4 <= d2.y_planes, "vdm_conv3d_tf32: y plane window out of range");
  }
  d2.r_planes = d.r_planes > 0 ? d.r_planes : d.c_out / 4;
  return conv3d_run(d2, x, w, y, epi, true, (cudaStream_t)stream);
}
