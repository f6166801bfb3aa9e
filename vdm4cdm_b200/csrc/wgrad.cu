// Conv3d weight gradient on the 5th-gen tensor cores:
//     dW[tap][ci][co] += sum over (b, d, h, w) of  a[b][ci][d+kd][h+kh][w+kw] * g[b][co][d][h][w]
// Stands in for the cuDNN conv3d backward-filter launched by autograd for every torch.nn.Conv3d of
// mltools' CUNet during LightVDM / LightSFM training_step (trainVDM3D128_..._lowbatch.py:128-132).
//
// GEMM view: M = input channels, N = output channels, K = voxels.  Both operands are read from the
// same channel-planar bf16 tensors the forward uses, as MN-major un-swizzled UMMA operands (8 channels
// = 16 B contiguous, 8 voxels along w = one core matrix, the next 8 voxels = the next h row = LBO, the
// next 8 channels = the next plane = SBO; verified by tools/probe_umma.cu test T4).  A filter tap is a
// start-address offset into the halo tile of `a`, exactly as in the forward kernel.
//
// tcgen05 wants M = 128.  Narrow layers fold d-slices into M: with cpb = channels per block (16, 32,
// 64 or 128, the largest that divides Cin) one operand block is S = 128 / cpb consecutive halo slices
// x cpb channels, laid out [slice][plane][h'][w'][8] in shared memory so that the 16 groups of 8 rows
// are equally spaced.  Against ONE slice of g, row block s of the accumulator is then filter plane
// kd = s - 1 (+ S per further block); rows with kd > 1 are computed and dropped.  Accumulators (one per
// (block, kh, kw) "job", N fp32 columns each) stay in TMEM over all tiles a CTA visits and are added to
// dW with fp32 atomics once at the end, so split-K over CTAs costs one pass over dW per CTA.
//
// Pipeline per CTA (6 warps): warp 0 TMA producer (halo slices of a + one tile of g per stage),
// warp 1 MMA issuer (jobs x 8 K-steps of 16 voxels per tile), warps 2-5 final TMEM -> atomics.
// Roofline: tensor-bound, algorithmic FLOPs = 2 * taps * Cin * Cout * B*D*H*W (same as the forward).
#include "common.cuh"
#include "ptx.cuh"
#include "tma_host.cuh"

namespace vdm {

constexpr int kWgThreads = 192;
constexpr int kWgTileH = 16, kWgTileW = 8;
constexpr int kWgMaxStages = 4;

struct WgradParams {
  int B, D, H, W;
  int c_in, c_out;
  int n;                 // UMMA N per CTA (c_out padded to 16, or its n-split share)
  int n_split;
  int cpb, S;            // channels per M block, slices folded into M
  int n_cblocks;         // Cin / cpb
  int n_sblocks;         // operand blocks along d: ceil(kd_count / S)
  int kd_count, pad;     // 3 / 1 for 3x3x3, 1 / 0 for 1x1x1
  int Hh, Wh;            // halo tile (voxels)
  int n_jobs_total;      // n_sblocks * n_khw
  int jobs_per_cta, n_jgroups;
  int n_khw;             // (kh, kw) pairs: 9 or 1
  int tiles_w, tiles_h, n_tiles;   // n_tiles = B * tiles_h * tiles_w * D
  int n_splits;          // CTAs sharing one (cblock, jgroup, nsplit)
  int stages, a_stage_bytes, g_stage_bytes;
  int slice_bytes;       // (cpb/8) * Hh * Wh * 16
  int x_planes, x_plane0, g_planes, g_plane0;
  int a_shift;           // 1 when `a` carries a one-voxel periodic halo
  int g_shift;           // same for g
  int tmem_cols;
  float* dw;             // fp32, element (tap, ci, co) at tap*st_tap + ci*st_ci + co*st_co
  long long st_tap, st_ci, st_co;
  int c_in_real;
};

struct WgradShared {
  uint64_t full[kWgMaxStages], empty[kWgMaxStages];
  uint64_t done;
  uint32_t tmem_base;
  uint32_t job_off[32];      // per job of this CTA: offset of its A operand inside a stage (16-byte units), computed once
};

__global__ void __launch_bounds__(kWgThreads, 1)
conv3d_wgrad_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_g,
                    const __grid_constant__ WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int stage_bytes = p.a_stage_bytes + p.g_stage_bytes;
  WgradShared* sh = reinterpret_cast<WgradShared*>(smem + (size_t)p.stages * stage_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // work unit of this CTA
  int u = blockIdx.x;
  const int split = u % p.n_splits; u /= p.n_splits;
  const int ns = u % p.n_split; u /= p.n_split;
  const int jg = u % p.n_jgroups;
  const int cb = u / p.n_jgroups;
  const int job0 = jg * p.jobs_per_cta;
  const int n_jobs = min(p.jobs_per_cta, p.n_jobs_total - job0);
  const int tile_begin = (int)((long long)p.n_tiles * split / p.n_splits);
  const int tile_end = (int)((long long)p.n_tiles * (split + 1) / p.n_splits);

  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmap_a);
    ptx::prefetch_tensormap(&tmap_g);
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&sh->full[s], 1);
      ptx::mbar_init(&sh->empty[s], 1);
    }
    ptx::mbar_init(&sh->done, 1);
    ptx::fence_barrier_init();
    // (the issue loop used to divide job by n_khw and khw by 3 for every job of every 128-voxel tile)
    const int sb0 = job0 / p.n_khw;
    for (int j = 0; j < n_jobs && j < 32; ++j) {
      const int job = job0 + j;
      const int sb = job / p.n_khw, khw = job % p.n_khw;
      const int kh = p.n_khw == 9 ? khw / 3 : 0, kw = p.n_khw == 9 ? khw % 3 : 0;
      sh->job_off[j] = (uint32_t)(sb - sb0) * 16u * (uint32_t)(p.Hh * p.Wh) + (uint32_t)(kh * p.Wh + kw);
    }
  }
  if (warp == 1) {
    ptx::tmem_alloc(&sh->tmem_base, (uint32_t)p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = sh->tmem_base;
  // A CTA's jobs (job = operand block sb along d x (kh, kw)) touch only the halo slices of blocks sb_lo..sb_hi: wide
  // layers (cpb = 128, S = 1, two or four jobs per CTA) mostly need ONE of the three slices, and loading all three
  // made them TMA-bound (202 KB per tile for 16 MMAs of N = 256; r02t).
  const int sb_lo = job0 / p.n_khw, sb_hi = (job0 + n_jobs - 1) / p.n_khw;
  const int sl_lo = sb_lo * p.S;
  const int n_slices = (sb_hi - sb_lo + 1) * p.S;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      // tile -> (b, h0, w0, d), d fastest: decoded once, then advanced (four run-time divisions per 128-voxel tile before)
      int t = tile_begin;
      int d = t % p.D; t /= p.D;
      int tw = t % p.tiles_w; t /= p.tiles_w;
      int th = t % p.tiles_h;
      int b = t / p.tiles_h;
      uint32_t s = 0, ph = 0;
      const uint32_t stages = (uint32_t)p.stages;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        const int w0 = tw * kWgTileW, h0 = th * kWgTileH;
        ptx::mbar_wait(&sh->empty[s], ph ^ 1u);
        ptx::mbar_arrive_expect_tx(&sh->full[s], (uint32_t)(n_slices * p.slice_bytes + p.g_stage_bytes));
        uint8_t* a_dst = smem + (size_t)s * stage_bytes;
        for (int sl = 0; sl < n_slices; ++sl)
          ptx::tma_load_4d(a_dst + (size_t)sl * p.slice_bytes, &tmap_a, &sh->full[s], (w0 - p.pad + p.a_shift) * 8,
                           h0 - p.pad + p.a_shift, d - p.pad + sl_lo + sl + p.a_shift,
                           b * p.x_planes + p.x_plane0 + cb * (p.cpb >> 3));
        ptx::tma_load_4d(a_dst + p.a_stage_bytes, &tmap_g, &sh->full[s], w0 * 8, h0, d,
                         b * p.g_planes + p.g_plane0 + ns * (p.n >> 3));
        if (++s == stages) { s = 0; ph ^= 1u; }
        if (++d == p.D) {
          d = 0;
          if (++tw == p.tiles_w) {
            tw = 0;
            if (++th == p.tiles_h) { th = 0; ++b; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (uniform datapath, see conv3d.cu) =====================
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const bool leader = ptx::elect_one();
    const uint32_t n = (uint32_t)p.n;
    // instruction descriptor: bf16 x bf16 -> f32, A and B MN-major (bits 15, 16)
    const uint32_t idesc = ptx::make_idesc_bf16(128, n) | (1u << 15) | (1u << 16);
    // LBO = stride between 8-voxel groups (next h row), SBO = stride between 8-channel groups
    const uint32_t plane16 = (uint32_t)(p.Hh * p.Wh);      // one plane of one halo slice, 16-byte units
    const uint64_t a_hi = ((uint64_t)((uint32_t)p.Wh & 0x3FFFu) << 16) | ((uint64_t)(plane16 & 0x3FFFu) << 32) | ((uint64_t)1 << 46);
    const uint64_t b_hi = ((uint64_t)8u << 16) | ((uint64_t)128u << 32) | ((uint64_t)1 << 46);
    const uint32_t smem16 = ptx::smem_u32(smem) >> 4;
    const uint32_t stage16 = (uint32_t)stage_bytes >> 4, a_stage16 = (uint32_t)p.a_stage_bytes >> 4;
    const uint32_t block16 = 16u * plane16;                 // one 128-row operand block
    const uint32_t Wh2 = 2u * (uint32_t)p.Wh;
    const uint32_t stages = (uint32_t)p.stages;
    uint32_t s = 0, ph = 0;
    bool first = true;
    for (int tile = tile_begin; tile < tile_end; ++tile) {
      ptx::mbar_wait(&sh->full[s], ph);
      ptx::tc_fence_after();
      if (leader) {
        const uint32_t a0 = smem16 + s * stage16, g0 = a0 + a_stage16;
        const uint32_t acc = first ? 0u : 1u;
        for (int j = 0; j < n_jobs; ++j) {
          const uint32_t a_job = a0 + sh->job_off[j];
          const uint32_t d_tmem = tmem_u + (uint32_t)j * n;
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const uint64_t a_desc = a_hi | (uint64_t)((a_job + (uint32_t)k * Wh2) & 0x3FFFu);
            const uint64_t b_desc = b_hi | (uint64_t)((g0 + (uint32_t)(16 * k)) & 0x3FFFu);
            ptx::umma_bf16(d_tmem, a_desc, b_desc, idesc, k == 0 ? acc : 1u);
          }
        }
        ptx::umma_commit(&sh->empty[s]);
        if (tile == tile_end - 1) ptx::umma_commit(&sh->done);
      }
      __syncwarp();
      first = false;
      if (++s == stages) { s = 0; ph ^= 1u; }
    }
  } else if (tile_end > tile_begin) {
    // ===================== final epilogue: TMEM -> fp32 atomics into dW =====================
    const int q = warp & 3;                 // TMEM lane quarter this warp may read
    const int m = q * 32 + lane;            // accumulator row
    ptx::mbar_wait(&sh->done, 0);
    ptx::tc_fence_after();
    const int s_in_block = m / p.cpb, ci = cb * p.cpb + m % p.cpb;
    for (int j = 0; j < n_jobs; ++j) {
      const int job = job0 + j;
      const int sb = job / p.n_khw, khw = job % p.n_khw;
      const int kd = sb * p.S + s_in_block;               // 0..kd_count-1 are real filter planes
      const bool row_ok = kd < p.kd_count && ci < p.c_in_real;
      const int tap = kd * p.n_khw + khw;
      for (int c0 = 0; c0 < p.n; c0 += 16) {
        uint32_t raw[16];
        ptx::tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(j * p.n + c0), raw);
        ptx::tmem_ld_wait();
        if (row_ok) {
          float* dst = p.dw + (long long)tap * p.st_tap + (long long)ci * p.st_ci + (long long)(ns * p.n + c0) * p.st_co;
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (ns * p.n + c0 + i < p.c_out) atomicAdd(dst + (long long)i * p.st_co, __uint_as_float(raw[i]));
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ---- narrow layers (c_out <= 32, 3x3x3): kw folded into N, halo slices streamed along d -----------------------
// With N = c_out = 32 the MMAs of the kernel above run at the shared-memory operand rate (41 cycles for 16 cycles of
// math), every tile re-loads S halo slices of `a` for ONE slice of g, and 9 (kh, kw) jobs share nothing.  Here
//   dW[kd,kh,kw][ci][co] = sum_u a[u + (kd-1, kh-1, 0)][ci] * g[u - (0, 0, kw-1)][co]
// so for a fixed kh the three kw taps are ONE MMA against three w-shifted copies of the g tile stacked along N
// (3*n rows; the copies are three TMA loads of the same tile at shifted coordinates, zero-filled at the borders):
// 3 jobs x 8 K-steps of N = 96 per output slice instead of 9 x 8 of N = 32.  A CTA marches along d: segments of LEN
// output slices at a fixed (b, h0, w0); halo slice k of a segment lives in slot k of a window of LEN + S - 1 slots,
// output j reads slots j..j+S-1 (rows of filter planes > 2 are garbage and dropped), and slot k is handed back to
// the producer as soon as output k's MMAs completed, so the next segment's loads overlap this segment's MMAs and
// every halo slice is loaded (LEN+2)/LEN times instead of S times.
constexpr int kWnLen = 8;          // output slices per segment
constexpr int kWnMaxSlots = kWnLen + 8;
constexpr int kWnGStages = 3;
constexpr int kWnThreads = 224;    // halo producer, MMA issuer, g producer, 4 epilogue warps (one per TMEM lane quarter)

struct WgradNarrowParams {
  int B, D, H, W;
  int c_in, c_out, c_in_real;
  int n;                 // c_out rounded up to 16 (16 or 32): UMMA N = 3*n
  int cpb, S, n_cblocks;
  int n_slots;           // kWnLen + S - 1
  int tiles_w, tiles_h, segs_d, n_segs;
  int n_splits;          // CTAs per channel block
  int slice_bytes, g_tile_bytes, g_stage_bytes;
  int x_planes, x_plane0, g_planes, g_plane0;
  int a_shift, g_shift;
  float* dw;
  long long st_tap, st_ci, st_co;
};

struct WgradNarrowShared {
  uint64_t slot_full[kWnMaxSlots], slot_empty[kWnMaxSlots];
  uint64_t g_full[kWnGStages], g_empty[kWnGStages];
  uint64_t done;
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kWnThreads, 1)
conv3d_wgrad_narrow_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_g0,
                           const __grid_constant__ CUtensorMap tmap_g1, const __grid_constant__ CUtensorMap tmap_g2,
                           const __grid_constant__ WgradNarrowParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_smem = smem;                                              // n_slots halo slices
  uint8_t* g_smem = smem + (size_t)p.n_slots * p.slice_bytes;          // kWnGStages x 3 shifted g tiles
  WgradNarrowShared* sh = reinterpret_cast<WgradNarrowShared*>(g_smem + (size_t)kWnGStages * p.g_stage_bytes);
  constexpr int Hh = kWgTileH + 2, Wh = kWgTileW + 2;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int split = blockIdx.x % p.n_splits;
  const int cb = blockIdx.x / p.n_splits;
  const int n_my = (p.n_segs - split + p.n_splits - 1) / p.n_splits;   // segments split, split + n_splits, ...

  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmap_a);
    ptx::prefetch_tensormap(&tmap_g0);
    ptx::prefetch_tensormap(&tmap_g1);
    ptx::prefetch_tensormap(&tmap_g2);
    for (int s = 0; s < p.n_slots; ++s) {
      ptx::mbar_init(&sh->slot_full[s], 1);
      ptx::mbar_init(&sh->slot_empty[s], 1);
    }
    for (int s = 0; s < kWnGStages; ++s) {
      ptx::mbar_init(&sh->g_full[s], 1);
      ptx::mbar_init(&sh->g_empty[s], 1);
    }
    ptx::mbar_init(&sh->done, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&sh->tmem_base, 512u);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = sh->tmem_base;

  auto seg_coord = [&](int i, int& b, int& d0, int& h0, int& w0) {
    int t = split + i * p.n_splits;
    d0 = (t % p.segs_d) * kWnLen; t /= p.segs_d;
    w0 = (t % p.tiles_w) * kWgTileW; t /= p.tiles_w;
    h0 = (t % p.tiles_h) * kWgTileH;
    b = t / p.tiles_h;
  };

  if (warp == 0) {
    // ===================== halo-slice producer =====================
    if (lane == 0) {
      for (int i = 0; i < n_my; ++i) {
        int b, d0, h0, w0;
        seg_coord(i, b, d0, h0, w0);
        for (int k = 0; k < kWnLen + 2; ++k) {
          ptx::mbar_wait(&sh->slot_empty[k], (i & 1) ^ 1);
          ptx::mbar_arrive_expect_tx(&sh->slot_full[k], (uint32_t)p.slice_bytes);
          ptx::tma_load_4d(a_smem + (size_t)k * p.slice_bytes, &tmap_a, &sh->slot_full[k], (w0 - 1 + p.a_shift) * 8,
                           h0 - 1 + p.a_shift, d0 - 1 + k + p.a_shift,
                           b * p.x_planes + p.x_plane0 + cb * (p.cpb >> 3));
        }
      }
    }
  } else if (warp == 2) {
    // ===================== g producer: three w-shifted copies of one tile per stage =====================
    if (lane == 0) {
      uint32_t it = 0;
      for (int i = 0; i < n_my; ++i) {
        int b, d0, h0, w0;
        seg_coord(i, b, d0, h0, w0);
        for (int j = 0; j < kWnLen; ++j, ++it) {
          const int s = it % kWnGStages;
          ptx::mbar_wait(&sh->g_empty[s], ((it / kWnGStages) & 1) ^ 1);
          ptx::mbar_arrive_expect_tx(&sh->g_full[s], (uint32_t)p.g_stage_bytes);
          uint8_t* dst = g_smem + (size_t)s * p.g_stage_bytes;
          // copy kw holds g(u - (kw - 1)) along w.  Zero padding: one map, shifted coordinates, out-of-range zero-filled.
          // Circular padding (g with a periodic halo): map kw is a (W, H, D) window of the padded tensor that starts
          // (2 - kw) voxels into a row, so the shift wraps periodically while positions u >= W still read zeros.
          const int sh_w = p.g_shift ? 0 : 1;
          ptx::tma_load_4d(dst, &tmap_g0, &sh->g_full[s], (w0 + sh_w) * 8, h0, d0 + j, b * p.g_planes + p.g_plane0);
          ptx::tma_load_4d(dst + (size_t)p.g_tile_bytes, &tmap_g1, &sh->g_full[s], w0 * 8, h0, d0 + j,
                           b * p.g_planes + p.g_plane0);
          ptx::tma_load_4d(dst + (size_t)2 * p.g_tile_bytes, &tmap_g2, &sh->g_full[s], (w0 - sh_w) * 8, h0, d0 + j,
                           b * p.g_planes + p.g_plane0);
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const bool leader = ptx::elect_one();
    const uint32_t n3 = 3u * (uint32_t)p.n;
    const uint32_t idesc = ptx::make_idesc_bf16(128, n3) | (1u << 15) | (1u << 16);     // A and B MN-major
    const uint32_t plane16 = (uint32_t)(Hh * Wh);
    // A: LBO = next 8 voxels (next h row), SBO = next 8 channels (next plane; slices are contiguous planes)
    const uint64_t a_hi = ((uint64_t)(uint32_t)Wh << 16) | ((uint64_t)plane16 << 32) | ((uint64_t)1 << 46);
    // B: LBO = next h row of the dense 16x8 tile, SBO = next 8 output channels (planes, then the next shifted copy)
    const uint64_t b_hi = ((uint64_t)8u << 16) | ((uint64_t)128u << 32) | ((uint64_t)1 << 46);
    const uint32_t a_base16 = ptx::smem_u32(a_smem) >> 4, g_base16 = ptx::smem_u32(g_smem) >> 4;
    const uint32_t slice16 = (uint32_t)p.slice_bytes >> 4, gstage16 = (uint32_t)p.g_stage_bytes >> 4;
    // ONE elected lane runs the whole schedule, barrier waits included, with 64-bit descriptors and immediate per-MMA
    // offsets (the lessons of conv3d.cu section "issuing thread": a warp-wide wait / fence / elect / __syncwarp per
    // output slice and ~8 instructions per MMA kept this kernel at 815 TFLOP/s where its N = 96 MMAs allow ~1250)
    if (leader) {
      const uint64_t a_desc0 = a_hi | (uint64_t)(a_base16 + 1u);         // + 1: centre column of the halo
      const uint64_t b_desc0 = b_hi | (uint64_t)g_base16;
      uint32_t gs = 0, gph = 0;
      bool first = true;
      for (int i = 0; i < n_my; ++i) {
        const int seg = split + i * p.n_splits;
        const int d0 = (seg % p.segs_d) * kWnLen;
        const int len_eff = min(kWnLen, p.D - d0);
        const uint32_t par = (uint32_t)(i & 1);
        ptx::mbar_wait(&sh->slot_full[0], par);
        ptx::mbar_wait(&sh->slot_full[1], par);
#pragma unroll 1
        for (int j = 0; j < kWnLen; ++j) {
          ptx::mbar_wait(&sh->slot_full[j + 2], par);
          ptx::mbar_wait(&sh->g_full[gs], gph);
          ptx::tc_fence_after();
          if (j < len_eff) {
            const uint64_t a_j = a_desc0 + (uint64_t)((uint32_t)j * slice16);
            const uint64_t b_j = b_desc0 + (uint64_t)(gs * gstage16);
            const uint32_t acc = first ? 0u : 1u;
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
#pragma unroll
              for (int k = 0; k < 8; ++k)
                ptx::umma_bf16_off64(tmem_u, (uint32_t)kh * n3, a_j, (uint32_t)((kh + 2 * k) * Wh), b_j, (uint32_t)(16 * k), idesc,
                                     k == 0 ? acc : 1u);
            }
            first = false;
          }
          ptx::umma_commit(&sh->slot_empty[j]);
          ptx::umma_commit(&sh->g_empty[gs]);
          if (j == kWnLen - 1) {
            ptx::umma_commit(&sh->slot_empty[kWnLen]);
            ptx::umma_commit(&sh->slot_empty[kWnLen + 1]);
            if (i == n_my - 1) ptx::umma_commit(&sh->done);
          }
          if (++gs == (uint32_t)kWnGStages) { gs = 0; gph ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (n_my > 0) {
    // ===================== final epilogue: TMEM -> fp32 atomics into dW =====================
    const int q = warp & 3;
    const int m = q * 32 + lane;            // accumulator row = (slice block, channel)
    ptx::mbar_wait(&sh->done, 0);
    ptx::tc_fence_after();
    const int kd = m / p.cpb, ci = cb * p.cpb + m % p.cpb;
    const bool row_ok = kd < 3 && ci < p.c_in_real;
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) {
        const int tap = (kd * 3 + kh) * 3 + kw;
        for (int c0 = 0; c0 < p.n; c0 += 16) {
          uint32_t raw[16];
          ptx::tmem_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((kh * 3 + kw) * p.n + c0), raw);
          ptx::tmem_ld_wait();
          if (row_ok) {
            float* dst = p.dw + (long long)tap * p.st_tap + (long long)ci * p.st_ci + (long long)c0 * p.st_co;
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (c0 + i < p.c_out) atomicAdd(dst + (long long)i * p.st_co, __uint_as_float(raw[i]));
          }
        }
      }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512u);
  }
}

// Launch plan of one weight-gradient layer: which kernel, its blocking, pipeline depth, grid and shared memory, written
// into the kernel's parameters (the caller adds the operands).  Host arithmetic only.
struct WgradPlan {
  bool narrow;            // conv3d_wgrad_narrow_kernel (3x3x3, c_out <= 32) with `np`, else conv3d_wgrad_kernel with `gp`
  WgradNarrowParams np;
  WgradParams gp;
  int grid;
  size_t smem_bytes;
};

static int plan_wgrad(const VdmWgradDesc& d, int c_out16, int sms, WgradPlan& pl) {
  pl = WgradPlan{};
  pl.narrow = d.kernel == 3 && c_out16 <= 32 && d.depth >= 2;
  if (pl.narrow) {
    WgradNarrowParams& p = pl.np;
    p.n = c_out16;
    int cpb = 32;
    while (d.c_in % cpb != 0) cpb >>= 1;          // 32 or 16 (c_in is a multiple of 16)
    p.cpb = cpb; p.S = 128 / cpb; p.n_cblocks = d.c_in / cpb;
    p.n_slots = kWnLen + p.S - 1;
    p.tiles_w = ceil_div(d.width, kWgTileW);
    p.tiles_h = ceil_div(d.height, kWgTileH);
    p.segs_d = ceil_div(d.depth, kWnLen);
    const long long n_segs = (long long)d.batch * p.tiles_h * p.tiles_w * p.segs_d;
    VDM_CHECK_ARG(n_segs < (1ll << 31), "vdm_conv3d_wgrad: too many segments");
    p.n_segs = (int)n_segs;
    int n_splits = sms / p.n_cblocks;
    if (n_splits < 1) n_splits = 1;
    if (n_splits > p.n_segs) n_splits = p.n_segs;
    p.n_splits = n_splits;
    p.slice_bytes = (cpb / 8) * (kWgTileH + 2) * (kWgTileW + 2) * 16;
    p.g_tile_bytes = p.n * kWgTileH * kWgTileW * 2;
    p.g_stage_bytes = 3 * p.g_tile_bytes;
    pl.smem_bytes = (size_t)p.n_slots * p.slice_bytes + (size_t)kWnGStages * p.g_stage_bytes + sizeof(WgradNarrowShared) + 1024;
    VDM_CHECK_ARG(pl.smem_bytes <= 227 * 1024, "vdm_conv3d_wgrad: narrow-layer plan needs %zu bytes of shared memory",
                  pl.smem_bytes);
    pl.grid = p.n_cblocks * p.n_splits;
    return VDM_OK;
  }

  WgradParams& p = pl.gp;
  p.kd_count = d.kernel; p.pad = d.kernel == 3 ? 1 : 0;
  p.n_khw = d.kernel * d.kernel;
  p.Hh = kWgTileH + 2 * p.pad; p.Wh = kWgTileW + 2 * p.pad;
  int cpb = 128;
  while (d.c_in % cpb != 0) cpb >>= 1;
  p.S = 128 / cpb;
  int over_read = 0;
  if (d.kernel == 1) {
    // 1x1x1: there is no filter plane to fold into M, and the layer is HBM-bound: load each `a` slice ONCE.  One block
    // = the widest multiple of 16 channels <= 128 dividing c_in; accumulator rows beyond it are garbage (the operand
    // descriptor walks 16 plane-strides into whatever follows in shared memory) and are dropped in the epilogue.
    // (r01r: 0.38 ms for the 96->32 skip conv with S = 4 slices loaded per tile, 4x its HBM floor.)
    cpb = 128;
    while (d.c_in % cpb != 0) cpb -= 16;
    p.S = 1;
    over_read = 16 * kWgTileH * kWgTileW * 16;
  }
  p.cpb = cpb; p.n_cblocks = d.c_in / cpb;
  p.n_sblocks = (p.kd_count + p.S - 1) / p.S;
  p.n_jobs_total = p.n_sblocks * p.n_khw;
  p.n_split = c_out16 > 128 ? 2 : 1;
  VDM_CHECK_ARG(c_out16 % (16 * p.n_split) == 0, "vdm_conv3d_wgrad: c_out=%d cannot be split", d.c_out);
  p.n = c_out16 / p.n_split;
  p.jobs_per_cta = 512 / p.n;
  if (p.jobs_per_cta > p.n_jobs_total) p.jobs_per_cta = p.n_jobs_total;
  p.n_jgroups = (p.n_jobs_total + p.jobs_per_cta - 1) / p.jobs_per_cta;
  p.jobs_per_cta = (p.n_jobs_total + p.n_jgroups - 1) / p.n_jgroups;   // balance the groups
  int cols = 32;
  while (cols < p.jobs_per_cta * p.n) cols <<= 1;
  p.tmem_cols = cols;
  p.tiles_w = ceil_div(d.width, kWgTileW);
  p.tiles_h = ceil_div(d.height, kWgTileH);
  const long long n_tiles = (long long)d.batch * p.tiles_h * p.tiles_w * d.depth;
  VDM_CHECK_ARG(n_tiles < (1ll << 31), "vdm_conv3d_wgrad: too many tiles");
  p.n_tiles = (int)n_tiles;
  p.slice_bytes = (cpb / 8) * p.Hh * p.Wh * 16;
  p.a_stage_bytes = (p.n_sblocks * p.S * p.slice_bytes + 127) & ~127;
  p.g_stage_bytes = p.n * kWgTileH * kWgTileW * 2;
  const int budget = 227 * 1024 - 1024 - (int)sizeof(WgradShared) - 256 - over_read;
  int stages = budget / (p.a_stage_bytes + p.g_stage_bytes);
  if (stages > kWgMaxStages) stages = kWgMaxStages;
  VDM_CHECK_ARG(stages >= 1, "vdm_conv3d_wgrad: one stage (%d bytes) does not fit shared memory",
                p.a_stage_bytes + p.g_stage_bytes);
  p.stages = stages;
  VDM_CHECK_ARG(16 * p.Hh * p.Wh <= 0x3FFF, "vdm_conv3d_wgrad: operand block too large for the descriptor");
  const int units = p.n_cblocks * p.n_jgroups * p.n_split;
  int n_splits = (2 * sms) / units;          // about two CTAs' worth of work units per SM ...
  if (n_splits < 1) n_splits = 1;
  if (n_splits > p.n_tiles) n_splits = p.n_tiles;     // ... but at least one tile each
  if (units * n_splits > sms && n_splits > 1) {
    // prefer exactly one wave when that keeps >= 8 tiles per CTA
    const int one_wave = sms / units;
    if (one_wave >= 1 && p.n_tiles / one_wave >= 8) n_splits = one_wave;
  }
  p.n_splits = n_splits;
  pl.smem_bytes = (size_t)p.stages * (p.a_stage_bytes + p.g_stage_bytes) + sizeof(WgradShared) + 1024 + over_read;
  pl.grid = units * n_splits;
  return VDM_OK;
}

}  // namespace vdm

using namespace vdm;

extern "C" int vdm_conv3d_wgrad(const VdmWgradDesc* desc, const void* a, const void* g, float* dw, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  VDM_CHECK_ARG(desc && a && g && dw, "vdm_conv3d_wgrad: NULL pointer argument");
  const VdmWgradDesc& d = *desc;
  VDM_CHECK_ARG(d.batch >= 1 && d.depth >= 1 && d.height >= 1 && d.width >= 1, "vdm_conv3d_wgrad: bad grid");
  VDM_CHECK_ARG(d.c_in >= 16 && d.c_in % 16 == 0, "vdm_conv3d_wgrad: c_in=%d must be a multiple of 16", d.c_in);
  VDM_CHECK_ARG(d.c_out >= 1 && d.c_out <= 256, "vdm_conv3d_wgrad: c_out=%d out of [1,256]", d.c_out);
  VDM_CHECK_ARG(d.kernel == 3 || d.kernel == 1, "vdm_conv3d_wgrad: kernel size %d (3 or 1 supported)", d.kernel);
  VDM_CHECK_ARG(!(d.kernel == 3 && d.a_padded && !d.g_padded), "vdm_conv3d_wgrad: a periodic `a` needs a periodic g (g_padded)");
  const int x_planes = d.a_planes > 0 ? d.a_planes : d.c_in / 8;
  const int c_out16 = (d.c_out + 15) / 16 * 16;
  const int g_planes = d.g_planes > 0 ? d.g_planes : c_out16 / 8;
  VDM_CHECK_ARG(d.a_plane0 >= 0 && d.a_plane0 + d.c_in / 8 <= x_planes, "vdm_conv3d_wgrad: a plane window out of range");
  VDM_CHECK_ARG(d.g_plane0 >= 0 && d.g_plane0 + c_out16 / 8 <= g_planes,
                "vdm_conv3d_wgrad: g plane window out of range (g must hold c_out rounded up to 16 channels)");
  VDM_CHECK_ARG((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0,
                "vdm_conv3d_wgrad: pointers must be 16-byte aligned");
  const bool dense_dw = d.dw_stride_tap == 0 && d.dw_stride_ci == 0 && d.dw_stride_co == 0;
  VDM_CHECK_ARG(dense_dw || (d.c_in_real >= 1 && d.c_in_real <= d.c_in), "vdm_conv3d_wgrad: c_in_real=%d out of [1, c_in]",
                d.c_in_real);
  if (!encode_fn()) {
    set_error("vdm_conv3d_wgrad: cuTensorMapEncodeTiled is not available from the driver");
    return VDM_E_DRIVER;
  }

  WgradPlan pl;
  int e = plan_wgrad(d, c_out16, num_sms(), pl);
  if (e != VDM_OK) return e;
  auto set_operands = [&](auto& p) {   // the fields both kernels' parameters share
    p.B = d.batch; p.D = d.depth; p.H = d.height; p.W = d.width;
    p.c_in = d.c_in; p.c_out = d.c_out;
    p.x_planes = x_planes; p.x_plane0 = d.a_plane0;
    p.a_shift = d.a_padded ? 1 : 0;
    p.g_shift = d.g_padded ? 1 : 0;
    p.g_planes = g_planes; p.g_plane0 = d.g_plane0;
    p.dw = dw;
    if (dense_dw) {
      p.st_tap = (long long)d.c_in * d.c_out; p.st_ci = d.c_out; p.st_co = 1; p.c_in_real = d.c_in;
    } else {
      p.st_tap = d.dw_stride_tap; p.st_ci = d.dw_stride_ci; p.st_co = d.dw_stride_co; p.c_in_real = d.c_in_real;
    }
  };
  if (pl.narrow) set_operands(pl.np);
  else set_operands(pl.gp);

  // `a` with a one-voxel periodic halo: the padded dims; one d-slice per box
  const int ah = d.a_padded ? 1 : 0, pad = pl.narrow ? 1 : pl.gp.pad, cpb = pl.narrow ? pl.np.cpb : pl.gp.cpb;
  CUtensorMap tma, tmg[3];
  e = encode_planar(&tma, a, d.width + 2 * ah, d.height + 2 * ah, d.depth + 2 * ah, (uint64_t)d.batch * x_planes, 0,
                    {(uint32_t)(kWgTileW + 2 * pad), (uint32_t)(kWgTileH + 2 * pad), 1u, (uint32_t)(cpb / 8)},
                    "vdm_conv3d_wgrad", "a");
  if (e != VDM_OK) return e;
  // g: logical dims (W, H, D) always (positions beyond the grid read zeros).  With a periodic halo the window starts in
  // the interior of the padded tensor; the narrow kernel reads three copies, copy kw starting (2 - kw) voxels into the
  // padded row (see the kernel).  Without one, all three maps are the same.
  const int gh = d.g_padded ? 1 : 0, n = pl.narrow ? pl.np.n : pl.gp.n;
  const uint64_t Wg = d.width + 2 * gh, Hg = d.height + 2 * gh;
  for (int kw = 0; kw < (pl.narrow ? 3 : 1); ++kw) {
    const char* base = static_cast<const char*>(g) + (gh ? ((Hg + 1) * Wg + (pl.narrow ? 2 - kw : 1)) * 16 : 0);
    e = encode_planar(&tmg[kw], base, d.width, d.height, d.depth, (uint64_t)d.batch * g_planes, gh,
                      {(uint32_t)kWgTileW, (uint32_t)kWgTileH, 1u, (uint32_t)(n / 8)}, "vdm_conv3d_wgrad", "g");
    if (e != VDM_OK) return e;
  }
  if (pl.narrow)
    return launch_kernel<conv3d_wgrad_narrow_kernel>(pl.grid, kWnThreads, pl.smem_bytes, stream, tma, tmg[0], tmg[1], tmg[2],
                                                     pl.np);
  return launch_kernel<conv3d_wgrad_kernel>(pl.grid, kWgThreads, pl.smem_bytes, stream, tma, tmg[0], pl.gp);
}
