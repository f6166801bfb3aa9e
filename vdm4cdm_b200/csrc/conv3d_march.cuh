// d-marching schedule of the kd-folded conv for the narrow 3x3x3 layers (Cin in {16, 32}, Cout_pad in {16, 32}: conv_in,
// the level-0 32->32 convs, conv_out and their dgrads).  Included by conv3d.cu (uses its helpers and ConvKernelParams).
//
// The tile schedule (conv3d_planar_kernel, issue_fold_tile) loads MT + 2 input slices per MT-slice tile and multiplies input
// slice i by the weights of the kd it can serve: N = 32, 64, 96, 96, 64, 32 for MT = 4.  Every MMA fetches 4 KB of A from
// shared memory whatever its N, so the edge slices run at 40 / 48 cycles for 16 / 32 cycles of math: 288 cycles per (kh, kw,
// k16) for 192 cycles of math, and the d-halo is loaded 1.5 times.  Here a CTA owns a COLUMN (sample, 16 x 8 face, d-segment)
// and marches through it: input slice i arrives ONCE, one N = 96 MMA per (kh, kw, k16) adds it to output slices i-2, i-1, i
// (kd = 2, 1, 0: adjacent column blocks of a TMEM ring of kMarchBlocks accumulators), output slice i-2 is complete right
// after and goes to the epilogue while the tensor core continues with slice i+1.  All MMAs but the two at each end of a
// segment are N = 96 (56 cycles for 48 of math), the halo is loaded (18/16)(10/8) = 1.4 times instead of 2.1, and an input
// stage is one slice (11.5 KB), so eight of them are in flight.
//
// Epilogue: TWELVE warps (warps 4..15, three per TMEM lane quarter; the tile schedule has eight and its input-transform
// warps idle on these layers).  R3a: with eight warps that each read their 16-channel chunk of EVERY slice the schedule was
// slower than the tile kernel (1.13 vs 0.84 ms on 32->32 at 128^3 x 8): wait -> tcgen05.ld -> arithmetic -> store is a
// ~1100-cycle dependent chain per slice and warp, longer than the 1008 cycles of the slice's MMAs.  Here the three warps of
// a quarter take the slices of a column round-robin (all channels of a slice), so a warp's chain may last three slices.
#pragma once
// (included by conv3d.cu INSIDE namespace vdm, after conv3d_planar_kernel)

constexpr int kMarchStages = 8;     // input slices in flight
constexpr int kMarchBlocks = 16;    // accumulator blocks (output slices) in the TMEM ring
constexpr int kMEpiWarps = 12, kMEpiThreads = 384;   // warps 4..15
constexpr int kRegsMEpi = 144;      // 128*64 + 384*144 = 63488 <= 65536
constexpr int kMarchResDepth = 2;   // residual slices in flight per epilogue warp (each warp owns every third slice)
constexpr int kMarchCaddMax = 1024; // floats of the bias + conditioning table kept in shared memory ([B][NF])

struct MarchShared {
  uint64_t a_full[kMarchStages], a_empty[kMarchStages];
  uint64_t a_ready[kMarchStages];     // fused input transform: the landed slice has been rewritten in place
  uint64_t b_full;
  uint64_t t_full[kMarchBlocks], t_empty[kMarchBlocks];
  uint32_t tmem_base;
};

struct MarchUnit {
  int b, h0, w0, d0, len;
};
__device__ __forceinline__ MarchUnit decode_unit(const ConvKernelParams& p, int u) {
  MarchUnit m;
  const int seg = u % p.m_nseg; u /= p.m_nseg;
  m.w0 = (u % p.tiles_w) * kTileW; u /= p.tiles_w;
  m.h0 = (u % p.tiles_h) * kTileH;
  m.b = u / p.tiles_h;
  m.d0 = seg * p.m_seglen;
  m.len = p.D - m.d0 < p.m_seglen ? p.D - m.d0 : p.m_seglen;
  return m;
}

// The MMAs of one input slice into ONE contiguous span of `nblk` accumulator blocks (output slices): for every (kh, kw, k16)
// the slice (shifted by (kh, kw)) times the stacked weights of the kd it serves.  FRESH: the last block of the span is an
// output slice that starts here (kd = 0) and is written without accumulation by the first MMA, which is therefore split.
// a_st / b_lo: low descriptor words (start address in 16-byte units | LBO << 16); b_lo already points at the first weight
// row block of the span; d_col: TMEM column of the span's first block.
template <int KJ, int NF, bool FRESH, int K0, int K1, int NBLK = 0>
__device__ __forceinline__ void issue_march_span(uint64_t a_desc, uint64_t b_desc, uint32_t d_col, int nblk_rt) {
  const int nblk = NBLK > 0 ? NBLK : nblk_rt;     // compile-time on the steady-state path (three blocks, immediate descriptors)
  constexpr int Wh = kTileW + 2;
  constexpr uint32_t kstep_a16 = 2u * (uint32_t)((kTileH + 2) * Wh);
  const uint32_t idesc = ptx::make_idesc_bf16(128, (uint32_t)(nblk * NF));
#pragma unroll
  for (int khw = K0; khw < K1; ++khw) {
#pragma unroll
    for (int j = 0; j < KJ; ++j) {
      const uint32_t a_off = (uint32_t)((khw / 3) * Wh + khw % 3) + (uint32_t)j * kstep_a16;
      const uint32_t b_off = (uint32_t)((khw * 2 * KJ + 2 * j) * 3 * NF);
      if (FRESH && khw == 0 && j == 0) {
        if (nblk > 1)
          ptx::umma_bf16_off64(d_col, 0u, a_desc, a_off, b_desc, b_off, ptx::make_idesc_bf16(128, (uint32_t)((nblk - 1) * NF)), 1u);
        ptx::umma_bf16_off64(d_col, (uint32_t)((nblk - 1) * NF), a_desc, a_off, b_desc, b_off + (uint32_t)((nblk - 1) * NF),
                             ptx::make_idesc_bf16(128, (uint32_t)NF), 0u);
      } else {
        ptx::umma_bf16_off64(d_col, 0u, a_desc, a_off, b_desc, b_off, idesc, 1u);
      }
    }
  }
}

// One input slice's MMAs for (kh, kw) in [K0, K1): output slices s_lo..s_hi = accumulator blocks g_lo.. (mod R) = weight row
// blocks starting at b_desc; the span is split in two where the ring wraps (2 of every 16 slices).
template <int KJ, int NF, int K0, int K1>
__device__ __forceinline__ void issue_march_slice(uint64_t a_desc, uint64_t b_desc, uint32_t tmem_u, uint32_t g_lo, int n, int n1,
                                                  bool fresh) {
  if (n1 == n) {
    if (fresh) issue_march_span<KJ, NF, true, K0, K1>(a_desc, b_desc, tmem_u + g_lo * (uint32_t)NF, n);
    else issue_march_span<KJ, NF, false, K0, K1>(a_desc, b_desc, tmem_u + g_lo * (uint32_t)NF, n);
  } else {
    issue_march_span<KJ, NF, false, K0, K1>(a_desc, b_desc, tmem_u + g_lo * (uint32_t)NF, n1);
    if (fresh) issue_march_span<KJ, NF, true, K0, K1>(a_desc, b_desc + (uint64_t)(n1 * NF), tmem_u, n - n1);
    else issue_march_span<KJ, NF, false, K0, K1>(a_desc, b_desc + (uint64_t)(n1 * NF), tmem_u, n - n1);
  }
}

// ---- epilogue of the marching schedule ----------------------------------------------------------------------------------
// thread = one voxel of the 16 x 8 face (TMEM lane), unit of work = one output slice, all NF channels; MODE as in
// epilogue_tiles.  Bias + conditioning rows come from a shared-memory table ([B][NF], loaded once per CTA); the residual from
// a cp.async ring in shared memory (kMarchResDepth slices of THIS warp in flight, the cursor runs ahead across units).
// Statistics: per-lane fp32 sums over the warp's slices of a unit, one transpose reduction per unit, per-warp slots folded
// in a fixed order into the CTA's fp64 running sums, fp64 atomics when the CTA moves on to another sample.
template <int NF, int MODE, int EW>
__device__ __forceinline__ void march_epilogue(const ConvKernelParams& p, MarchShared* sh, uint8_t* smem, float* stat_part,
                                               double* stat_acc, float* cadd_s, const uint32_t tmem_base) {
  // EW = epilogue warps per TMEM lane quarter: 3 (warps 4..15), 2 (warps 4..11) when warps 12..15 transform the input, 1 (warps
  // 4..7) for conv_out, where warps 8..15 transform
  constexpr int kThreadsE = 128 * EW;
  constexpr bool RES = (MODE & kEpiRes) != 0, STATS = (MODE & kEpiStats) != 0, FP32 = (MODE & kEpiFp32) != 0;
  constexpr int R = kMarchBlocks, n_chunks = NF / 16, n_planes = NF / 8;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = warp & 3;                        // TMEM lane quarter
  const int ew = warp - (kEpiFirst >> 5);        // 0..11
  const int k3 = ew >> 2;                        // which of the three warps of that quarter: owns slices s = k3 (mod 3)
  const int et = threadIdx.x - kEpiFirst;        // 0..383
  const int r = q * 32 + lane;
  const int lh = r >> 3, lw = r & 7;
  const long long HW = (long long)p.H * p.W, V = (long long)p.D * HW;
  const float* cadd_g = cadd_rows(p);
  const bool cadd_table = p.B * NF <= kMarchCaddMax;
  if (cadd_table) VDM_CADD_TABLE_FILL(cadd_s, cadd_g, p.B, NF, p.c_out, et, kThreadsE);
  // valid 8-channel planes (bf16 output: c_out % 8 == 0)
  const int n_valid_planes = (p.c_out >> 3) < n_planes ? (p.c_out >> 3) : n_planes;
  // residual ring: slot i, plane pl of this thread: r_ring[(i * n_planes + pl) * kMEpiThreads]
  uint4* r_ring = reinterpret_cast<uint4*>(smem + p.res_ring_off) + et;
  int r_slot = 0;
  const uint4* res_base = reinterpret_cast<const uint4*>(p.residual);
  const int r_sh = p.r_up;
  const int r_H = p.H >> r_sh, r_W = p.W >> r_sh;
  const long long r_HW = (long long)r_H * r_W, r_V = (long long)(p.D >> r_sh) * r_HW;
  int r_unit = blockIdx.x - (int)gridDim.x, ru_s = 0, ru_len = 0, r_d0 = 0;
  const uint4* r_ptr = nullptr;
  bool r_hw_ok = false;
  auto res_issue = [&](int slot) __attribute__((always_inline)) {
    bool live = true;
    while (live && ru_s >= ru_len) {               // move the cursor to this CTA's next unit
      r_unit += (int)gridDim.x;
      if (r_unit < p.m_units) {
        const MarchUnit mr = decode_unit(p, r_unit);
        const int hr = mr.h0 + lh, wr = mr.w0 + lw;
        r_hw_ok = (hr < p.H) && (wr < p.W);
        r_d0 = mr.d0;
        ru_len = mr.len;
        r_ptr = res_base + ((long long)mr.b * p.r_planes + p.r_plane0 + (((hr & 1) << 1) | (wr & 1)) * p.r_d2s_planes) * r_V +
                (long long)(hr >> r_sh) * r_W + (wr >> r_sh);
        ru_s = k3;
      } else {
        live = false;
      }
    }
    if (live) {
      const int dz = r_d0 + ru_s;
      ru_s += EW;
      if (r_hw_ok) {
        const uint4* src = r_ptr + (long long)(((dz & 1) << 2) * p.r_d2s_planes) * r_V + (long long)(dz >> r_sh) * r_HW;
        uint4* dst = r_ring + (slot * n_planes) * kMEpiThreads;
#pragma unroll
        for (int pl = 0; pl < n_planes; ++pl)
          if (pl < n_valid_planes) ptx::cp_async16(dst + pl * kMEpiThreads, src + (long long)pl * r_V);
      }
    }
    ptx::cp_async_commit();                        // one group per slice, also when nothing was copied
  };
  if (RES) {
    for (int i = 0; i < kMarchResDepth; ++i) res_issue(i);
  }
  uint32_t ob = 0;
  for (int u = blockIdx.x; u < p.m_units; u += gridDim.x) {
    const MarchUnit m = decode_unit(p, u);
    const int h = m.h0 + lh, w = m.w0 + lw;
    const bool hw_ok = (h < p.H) && (w < p.W);
    const long long vox0 = ((long long)m.d0 * p.H + h) * p.W + w;
    const float* cadd_row = cadd_s + m.b * NF;
    float s1[n_chunks][16], s2[n_chunks][16];
    if (STATS) {
#pragma unroll
      for (int c = 0; c < n_chunks; ++c)
#pragma unroll
        for (int j = 0; j < 16; ++j) s1[c][j] = s2[c][j] = 0.f;
    }
    bf16x8* y_b = reinterpret_cast<bf16x8*>(p.y) + ((long long)m.b * p.y_planes + p.y_plane0) * V + vox0;
    float* y32_b = static_cast<float*>(p.y) + (long long)m.b * p.c_out * V + vox0;
    for (int s = k3; s < m.len; s += EW) {
      const uint32_t o = ob + (uint32_t)s;
      const uint32_t g = o % (uint32_t)R;
      ptx::mbar_wait(&sh->t_full[g], (o / (uint32_t)R) & 1);
      ptx::tc_fence_after();
      const uint32_t tcol = tmem_base + ((uint32_t)(q * 32) << 16) + g * (uint32_t)NF;
      uint32_t raw[n_chunks][16];
#pragma unroll
      for (int c = 0; c < n_chunks; ++c) ptx::tmem_ld16(tcol + (uint32_t)(c * 16), raw[c]);
#pragma unroll
      for (int c = 0; c < n_chunks; ++c) ptx::tmem_ld_wait_dep(raw[c]);
      ptx::tc_fence_before();
      ptx::mbar_arrive(&sh->t_empty[g]);          // the block goes back to the MMA warp before the arithmetic
      if (VDM_DBG(p, 1)) continue;                // (bring-up: the epilogue only drains the accumulators)
      const uint4* slot = r_ring + (r_slot * n_planes) * kMEpiThreads;
      if (RES) ptx::cp_async_wait(kMarchResDepth - 1);
#pragma unroll
      for (int c = 0; c < n_chunks; ++c) {
        float f[16];
        if (cadd_table) {
          load_row16(cadd_row + c * 16, f);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            f[j] = (cadd_g && c * 16 + j < p.c_out) ? __ldg(cadd_g + (long long)m.b * p.c_out + c * 16 + j) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 16; j += 2) add2(f[j], f[j + 1], __uint_as_float(raw[c][j]), __uint_as_float(raw[c][j + 1]));
        if (FP32) {
          if (hw_ok) VDM_STORE_FP32_NCDHW(y32_b + (long long)(c * 16) * V + (long long)s * HW, f, p.c_out - c * 16, V);
          continue;
        }
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const int pl = c * 2 + hf;
          if (pl >= n_valid_planes || !hw_ok) continue;
          VDM_STORE_HALF_BF16(RES, STATS, f, hf, slot[pl * kMEpiThreads], y_b, (long long)pl * V + (long long)s * HW, s1[c], s2[c]);
        }
      }
      if (RES) {
        res_issue(r_slot);                        // refill the slot just consumed
        r_slot = (r_slot + 1 == kMarchResDepth) ? 0 : r_slot + 1;
      }
    }
    ob += (uint32_t)m.len;
    if (STATS) {
#pragma unroll
      for (int c = 0; c < n_chunks; ++c) VDM_STATS_TO_SLOTS(s1[c], s2[c], stat_part, ew, NF, c * 16, kMEpiWarps, lane);
      asm volatile("bar.sync 2, %0;" ::"n"(kThreadsE) : "memory");
      if (et < NF) {
        const int next_u = u + (int)gridDim.x;
        bool flush = next_u >= p.m_units;
        if (!flush) flush = decode_unit(p, next_u).b != m.b;
        VDM_FOLD_STATS(p, stat_part, stat_acc, NF, et, 4 * EW, kMEpiWarps, false, flush, m.b, 0);
      }
      asm volatile("bar.sync 2, %0;" ::"n"(kThreadsE) : "memory");     // the slots are read before the next unit overwrites them
    }
  }
}

// ---- fused GroupNorm + SiLU of the input (XF): warps 12..15 rewrite every landed input slice in place ------------------
// y = h + h tanh(h), h = a_c x + b_c ((a, b) per (sample, channel) from vdm_gn_coef, the 1/2 of silu(2h) folded in), voxels
// outside the grid back to zero (Conv3d's zero padding applies AFTER the non-linearity), fence.proxy.async, arrive on
// a_ready[s] -- the barrier the MMA issuer then waits on instead of a_full[s].  Warp j takes every fourth stage of the main
// tensor WHOLE (so its wait -> LDS -> arithmetic -> STS chain may last four slices: in the tile kernel four warps shared every
// stage and the chain, not the bandwidth, made the transform slower than the MMAs, R2h); a lane owns one 8-channel plane,
// its 16 coefficients stay in registers while the sample does not change.  Skip-tensor stages are not transformed.
// Hand-off with skip-tensor stages interleaved (that of the tile kernel's transform_tiles): EVERY warp waits for EVERY stage
// in order, main and skip alike, and arrives on a_ready[s] (count NXW) when it is done with it -- the owner after its
// transform and fence, the others right away.  No stage can be consumed, and so refilled, before all NXW warps have arrived,
// so no warp can fall two phases behind a barrier it waits on by parity.  Without skip stages all phases of a stage belong to
// its owner (stages j, j + NXW, ...), and the owner alone waits and arrives (count 1): there the all-warp form cost conv_out
// 5 % and the fused 32->32 convs 3 %.  NXW = number of transform warps (the last NXW warps of the CTA): 4, or 8 for conv_out.
template <int KJ, bool SKIP, int NXW>
__device__ __forceinline__ void march_transform(const ConvKernelParams& p, MarchShared* sh, uint8_t* a_smem) {
  constexpr int planes = 2 * KJ, S = kMarchStages;
  constexpr int kSliceBytes = (kTileH + 2) * (kTileW + 2) * 16, kStageBytes = planes * kSliceBytes;
  constexpr int lpp = 32 / planes;                         // lanes per plane
  constexpr int nvox = (kTileH + 2) * (kTileW + 2);
  constexpr int KMAX0 = (nvox + lpp - 1) / lpp;            // voxels per lane: 12 (two planes) or 23 (four)
  constexpr int G = planes == 2 ? 6 : 8;                   // 16-byte loads in flight per lane (R5d: 4 -> 8, conv_out -6 %)
  constexpr int KMAX = (KMAX0 + G - 1) / G * G;
  static_assert(KMAX <= 32, "one bit per voxel of a lane in zmask");
  const int lane = threadIdx.x & 31, j = (threadIdx.x >> 5) - (16 - NXW);      // NXW transform warps: warps 16 - NXW .. 15
  const int pl = lane / lpp, l0 = lane % lpp;
  const int skip_chunks = SKIP ? p.skip_chunks : 0;
  float ca[8], cb[8];
  int cur_b = -1;
  uint32_t it = 0, n_main = 0;                             // stage counter (all stages), main-tensor stages so far
  for (int u = blockIdx.x; u < p.m_units; u += gridDim.x) {
    const MarchUnit m = decode_unit(p, u);
    if (m.b != cur_b) {
      cur_b = m.b;
      load_coef8<true>(p.in_norm + ((long long)m.b * p.c_in + pl * 8) * 2, ca, cb);
    }
    // voxels of this lane that lie outside the grid in h / w (zero padding applies AFTER the non-linearity): bit k = voxel
    // l0 + k * lpp of the (kTileH + 2) x (kTileW + 2) halo slice, the same for every slice of the unit
    uint32_t zmask = 0u;
    if (m.h0 == 0 || m.h0 + kTileH >= p.H || m.w0 == 0 || m.w0 + kTileW >= p.W) {
      for (int k = 0; k < KMAX; ++k) {
        const int v = l0 + k * lpp;
        const int hy = v / (kTileW + 2), wx = v - hy * (kTileW + 2);
        if (v < nvox && ((unsigned)(m.h0 - 1 + hy) >= (unsigned)p.H || (unsigned)(m.w0 - 1 + wx) >= (unsigned)p.W)) zmask |= 1u << k;
      }
    }
    for (int i = 0; i < m.len + 2; ++i, ++n_main) {
      const bool own = (int)(n_main % (uint32_t)NXW) == j;
      if (SKIP || own) {
        const uint32_t s = it % (uint32_t)S;
        ptx::mbar_wait(&sh->a_full[s], (it / (uint32_t)S) & 1);
        const int dz = m.d0 - 1 + i;
        // the owner transforms the slice (one beyond the grid is all zero padding: nothing to do)
        if (own && dz >= 0 && dz < p.D) {
          uint4* base = reinterpret_cast<uint4*>(a_smem + (size_t)s * kStageBytes + (size_t)pl * kSliceBytes);
          // BRANCH-FREE body: G independent 16-byte chains per lane that ptxas can interleave (R5g: with a guard and an edge
          // branch around every voxel the chains ran one after another at ~4.5 cycles per instruction and the four transform
          // warps were busy 90 % of the time -- they, not the MMA issuer, bounded the fused layers).  Slots past the end of the
          // slice read whatever follows it in shared memory (the next plane / stage / the weights) and are not stored.
#pragma unroll 1
          for (int k0 = 0; k0 < KMAX; k0 += G) {
            uint4 xs[G];
#pragma unroll
            for (int g2 = 0; g2 < G; ++g2) xs[g2] = base[l0 + (k0 + g2) * lpp];
#pragma unroll
            for (int g2 = 0; g2 < G; ++g2) {
              const int v = l0 + (k0 + g2) * lpp;
              uint4 y = gn_silu8(xs[g2], ca, cb);
              if ((zmask >> (k0 + g2)) & 1u) y = make_uint4(0u, 0u, 0u, 0u);
              if (v < nvox) base[v] = y;
            }
          }
        }
        ptx::fence_proxy_async();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&sh->a_ready[s]);
      }
      ++it;
      // the skip-tensor stages of this output slice are not transformed: every warp waits for them and arrives all the same
      if (i < m.len) {
        for (int c = 0; c < skip_chunks; ++c, ++it) {
          const uint32_t s = it % (uint32_t)S;
          ptx::mbar_wait(&sh->a_full[s], (it / (uint32_t)S) & 1);
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&sh->a_ready[s]);
        }
      }
    }
  }
}

template <int KJ, int NF, bool SKIP, bool XF>
__global__ void __launch_bounds__(kConvThreads, 1)
conv3d_march_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_x2,
                    const __grid_constant__ ConvKernelParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_window_1024(smem_raw);
  constexpr int planes = 2 * KJ;
  constexpr int kSliceBytes = (kTileH + 2) * (kTileW + 2) * 16;        // one plane of one input slice
  constexpr int kStageBytes = planes * kSliceBytes;
  constexpr int kWBytes = 27 * planes * NF * 16;                       // resident weights, kd-folded order
  constexpr int R = kMarchBlocks, S = kMarchStages;
  uint8_t* a_smem = smem;
  uint8_t* b_smem = smem + (size_t)S * kStageBytes;
  MarchShared* sh = reinterpret_cast<MarchShared*>(b_smem + kWBytes + p.skip_w_bytes);   // (1x1x1 skip weights after the main ones)
  float* stat_part = reinterpret_cast<float*>(sh + 1);                 // [sum | sumsq][epilogue warp][channel]
  double* stat_acc = reinterpret_cast<double*>(stat_part + 2 * kMEpiWarps * NF);   // [sum | sumsq][channel]: this sample so far
  float* cadd_s = reinterpret_cast<float*>(stat_acc + 2 * NF);         // [B][NF] bias + conditioning rows

  // conv_out (16 output columns, one fp32 channel stored): the epilogue is a few instructions per voxel and the layer is
  // bound by the input transform (R5i: 26 % tensor-pipe activity, transform warps busy ~90 %), so eight warps transform
  // and four drain.  Only without the fused skip conv, whose 32-column epilogues (bias + residual + statistics) need their
  // eight warps.
  constexpr bool kWideXf = XF && !SKIP && NF == 16;
  // Arrivals per phase of a_ready (unused without XF): with skip stages interleaved every transform warp arrives, else the
  // owner alone (march_transform).  The count is that of the four-warp form, the only one that runs with skip stages.
  static_assert(!(kWideXf && SKIP), "a_ready expects four arrivals per phase when skip stages are interleaved");
  constexpr int kReadyCount = XF && SKIP ? 4 : 1;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmap_x);
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(&sh->a_full[s], 1);
      ptx::mbar_init(&sh->a_empty[s], 1);
      ptx::mbar_init(&sh->a_ready[s], kReadyCount);
    }
    ptx::mbar_init(&sh->b_full, 1);
    for (int g = 0; g < R; ++g) {
      ptx::mbar_init(&sh->t_full[g], 1);
      ptx::mbar_init(&sh->t_empty[g], 128);      // the four warps (one per lane quarter) that own the slice
    }
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&sh->tmem_base, (uint32_t)(R * NF));
    ptx::tmem_relinquish();
  }
  if (warp >= 4) {
    for (int i = threadIdx.x - kEpiFirst; i < 2 * NF; i += kMEpiThreads) stat_acc[i] = 0.0;
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = sh->tmem_base;

  if (warp < 4) {
    ptx::setmaxnreg_dec<kRegsWg0>();
    if (warp == 0) {
      // ===================== A producer: one input slice per stage =====================
      if (lane == 0) {
        uint32_t it = 0;
        for (int u = blockIdx.x; u < p.m_units; u += gridDim.x) {
          const MarchUnit m = decode_unit(p, u);
          for (int i = 0; i < m.len + 2; ++i) {
            {
              const int s = (int)(it % (uint32_t)S);
              ptx::mbar_wait(&sh->a_empty[s], ((it / (uint32_t)S) & 1) ^ 1);
              if (VDM_DBG(p, 2) && it >= (uint32_t)S) {      // (bring-up: no halo traffic after the pipeline fill)
                ptx::mbar_arrive(&sh->a_full[s]);
              } else {
                ptx::mbar_arrive_expect_tx(&sh->a_full[s], (uint32_t)kStageBytes);
                ptx::tma_load_4d(a_smem + (size_t)s * kStageBytes, &tmap_x, &sh->a_full[s], (m.w0 - 1 + p.x_shift) * 8,
                                 m.h0 - 1 + p.x_shift, m.d0 - 1 + i + p.x_shift, m.b * p.x_planes + p.x_plane0);
              }
              ++it;
            }
            // fused 1x1x1 skip conv: the face of output slice i of the skip tensor (never halo-padded), one stage per chunk
            if (i < m.len) {
              for (int c = 0; c < (SKIP ? p.skip_chunks : 0); ++c, ++it) {
                const int s = (int)(it % (uint32_t)S);
                ptx::mbar_wait(&sh->a_empty[s], ((it / (uint32_t)S) & 1) ^ 1);
                ptx::mbar_arrive_expect_tx(&sh->a_full[s], (uint32_t)(planes * kTileH * kTileW * 16));
                ptx::tma_load_4d(a_smem + (size_t)s * kStageBytes, &tmap_x2, &sh->a_full[s], m.w0 * 8, m.h0, m.d0 + i,
                                 m.b * p.x2_planes + p.x2_plane0 + c * planes);
              }
            }
          }
        }
      }
    } else if (warp == 2) {
      // ===================== B producer: all weights once, kd-folded order [khw][plane][2 - kd][co] =====================
      if (lane == 0 && blockIdx.x < (unsigned)p.m_units) {
        const size_t tap_stride = (size_t)p.c_in8 * p.n_pad * 8, plane_stride = (size_t)p.n_pad * 8;
        ptx::mbar_arrive_expect_tx(&sh->b_full, (uint32_t)kWBytes + (uint32_t)p.skip_w_bytes);
        // 1x1x1 skip-path weights: [plane][co] right after the main weights
        for (int pl = 0; pl < p.skip_chunks * planes; ++pl)
          ptx::bulk_load(b_smem + kWBytes + (size_t)pl * (NF * 16), p.w2 + (size_t)pl * plane_stride, (uint32_t)(NF * 16), &sh->b_full);
        for (int tap = 0; tap < 27; ++tap) {
          const int kd = p.tap_kd[tap], khw = p.tap_khw[tap];
#pragma unroll
          for (int pl = 0; pl < planes; ++pl)
            ptx::bulk_load(b_smem + (size_t)((khw * planes + pl) * 3 + (2 - kd)) * (NF * 16),
                           p.w + (size_t)tap * tap_stride + (size_t)pl * plane_stride, (uint32_t)(NF * 16), &sh->b_full);
        }
      }
    } else if (warp == 1) {
      // ===================== MMA issuer =====================
      const uint32_t a_base16 = ptx::smem_u32(a_smem) >> 4, a_stage16 = (uint32_t)kStageBytes >> 4;
      const uint32_t b_base16 = ptx::smem_u32(b_smem) >> 4;
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const bool leader = ptx::elect_one();
      const uint64_t a_hi = make_planar_desc(0, (uint32_t)kSliceBytes, (uint32_t)(kTileW + 2) * 16u);
      const uint64_t b_hi = make_planar_desc(0, 3u * (uint32_t)NF * 16u, 128u);
      const uint64_t b_desc0 = b_hi | (uint64_t)b_base16;                  // kd-folded weights, row block 0
      // ONE elected lane runs the whole schedule, barrier waits included.  What bounds these layers is this thread: the tensor
      // core's queue holds only a few MMAs, so every stretch of bookkeeping longer than that many x 56 cycles is a bubble
      // (R3o: 125 instructions per slice at ~7 cycles each around 19 MMAs; the pipe was busy 61% of the time).  The steady-state
      // slice therefore issues its MMAs in groups of four with one piece of the bookkeeping between groups: the look-ahead
      // waits for the next stage's barriers, the commits, the index arithmetic.
      if (leader && blockIdx.x < (unsigned)p.m_units) {
        ptx::mbar_wait(&sh->b_full, 0);
        int u = blockIdx.x;
        MarchUnit m = decode_unit(p, u);
        const int skip_chunks = SKIP ? p.skip_chunks : 0;
        uint32_t ita = 0, ob = 0;                 // stage counter, output-slice counter at the start of the unit
        // (landed and, with the fused input transform, rewritten / passed on by the transform warps)
        auto wait_stage = [&](uint32_t ita_) __attribute__((always_inline)) {
          ptx::mbar_wait(XF ? &sh->a_ready[ita_ % (uint32_t)S] : &sh->a_full[ita_ % (uint32_t)S], (ita_ / (uint32_t)S) & 1);
          ptx::tc_fence_after();
        };
        auto wait_skip_stage = [&](uint32_t ita_) __attribute__((always_inline)) { wait_stage(ita_); };
        auto wait_block = [&](uint32_t o) __attribute__((always_inline)) {      // accumulator block of output slice o drained
          ptx::mbar_wait(&sh->t_empty[o % (uint32_t)R], ((o / (uint32_t)R) & 1) ^ 1);
        };
        // input slice ii of a unit: its stage has landed and, if it starts output slice ii (kd = 0), that block is free
        auto wait_slice = [&](int ii, uint32_t ita_, uint32_t ob_, int len_) __attribute__((always_inline)) {
          if (ii < len_) wait_block(ob_ + (uint32_t)ii);
          wait_stage(ita_);
        };
        // skip-path descriptors: A = the slice's own face [plane][16 h][8 w][16 B] (LBO one plane, SBO one h row), B = [plane][co]
        const uint64_t a2_hi = make_planar_desc(0, (uint32_t)(kTileH * kTileW * 16), (uint32_t)kTileW * 16u);
        const uint64_t b2_hi = make_planar_desc(0, (uint32_t)NF * 16u, 128u);
        const uint32_t b2_base16 = b_base16 + ((uint32_t)kWBytes >> 4);
        // y += conv1x1x1(x_skip) for output slice i: KJ MMAs of N = NF per chunk into its accumulator, then the look-ahead for
        // input slice i + 1 (i < len, so that slice exists)
        auto skip_stages = [&](int i, int len) __attribute__((always_inline)) {
          const uint32_t d_s = tmem_u + ((ob + (uint32_t)i) % (uint32_t)R) * (uint32_t)NF;
          for (int c = 0; c < skip_chunks; ++c, ++ita) {
            const uint32_t s2 = ita % (uint32_t)S;
            const uint64_t a2 = a2_hi | (uint64_t)(a_base16 + s2 * a_stage16);
            const uint64_t b2 = b2_hi | (uint64_t)(b2_base16 + (uint32_t)(c * planes * NF));
#pragma unroll
            for (int j = 0; j < KJ; ++j)
              ptx::umma_bf16_off64(d_s, 0u, a2, (uint32_t)(j * 2 * kTileH * kTileW), b2, (uint32_t)(2 * j * NF),
                                   ptx::make_idesc_bf16(128, (uint32_t)NF), 1u);
            if (c + 1 < skip_chunks) wait_skip_stage(ita + 1u);
            else wait_slice(i + 1, ita + 1u, ob, len);
            ptx::umma_commit(&sh->a_empty[s2]);
          }
        };
        wait_slice(0, 0u, 0u, m.len);
        while (true) {
          const int len = m.len;
          // this CTA's next unit (decoded once per unit, needed by the last slice's look-ahead)
          const int nu = u + (int)gridDim.x;
          const bool more_units = nu < p.m_units;
          MarchUnit nm = m;
          if (more_units) nm = decode_unit(p, nu);
          // any slice: edges of a unit (fewer than three output slices, or none of them new) and ring wraps
          auto general_slice = [&](int i) __attribute__((always_inline)) {
            const uint32_t sa = ita % (uint32_t)S;
            const uint64_t a_desc = a_hi | (uint64_t)(a_base16 + sa * a_stage16);
            const bool last = i == len + 1;
            const bool skip_next = SKIP && i < len;                             // the next stage is this slice's skip chunk
            const int s_lo = i - 2 > 0 ? i - 2 : 0, s_hi = i < len - 1 ? i : len - 1;
            const bool fresh = i < len;
            const uint32_t g_lo = (ob + (uint32_t)s_lo) % (uint32_t)R;
            const int n = s_hi - s_lo + 1;
            const int n1 = n < R - (int)g_lo ? n : R - (int)g_lo;
            const uint64_t b_desc = b_desc0 + (uint64_t)((2 - i + s_lo) * NF);
            issue_march_slice<KJ, NF, 0, 5>(a_desc, b_desc, tmem_u, g_lo, n, n1, fresh);
            // the next stage (possibly of this CTA's next unit): its barriers are waited for here
            if (skip_next) wait_skip_stage(ita + 1u);
            else if (!last) wait_slice(i + 1, ita + 1u, ob, len);
            else if (more_units) wait_slice(0, ita + 1u, ob + (uint32_t)len, nm.len);
            issue_march_slice<KJ, NF, 5, 9>(a_desc, b_desc, tmem_u, g_lo, n, n1, fresh);
            ptx::umma_commit(&sh->a_empty[sa]);
            if (i >= 2) ptx::umma_commit(&sh->t_full[(ob + (uint32_t)(i - 2)) % (uint32_t)R]);
            ++ita;
            if (skip_next) skip_stages(i, len);
          };
          int i = 0;
          for (; i < 2 && i < len + 2; ++i) general_slice(i);
          for (; i < len; ++i) {
            const uint32_t g_st = (ob + (uint32_t)(i - 2)) % (uint32_t)R;       // block of output slice i - 2
            if (g_st > (uint32_t)(R - 3)) {
              general_slice(i);
              continue;
            }
            // steady state: output slices i-2, i-1, i (kd = 2, 1, 0), the last one starts here, no ring wrap
            const uint32_t sa = ita % (uint32_t)S;
            const uint64_t a_desc = a_hi | (uint64_t)(a_base16 + sa * a_stage16);
            const uint32_t d_col = tmem_u + g_st * (uint32_t)NF;
            issue_march_span<KJ, NF, true, 0, 2, 3>(a_desc, b_desc0, d_col, 3);
            if (!SKIP && i + 1 < len) wait_block(ob + (uint32_t)(i + 1));
            issue_march_span<KJ, NF, true, 2, 4, 3>(a_desc, b_desc0, d_col, 3);
            if (SKIP) wait_skip_stage(ita + 1u);
            else wait_stage(ita + 1u);
            issue_march_span<KJ, NF, true, 4, 6, 3>(a_desc, b_desc0, d_col, 3);
            issue_march_span<KJ, NF, true, 6, 9, 3>(a_desc, b_desc0, d_col, 3);
            ptx::umma_commit(&sh->a_empty[sa]);
            ptx::umma_commit(&sh->t_full[g_st]);
            ++ita;
            if (SKIP) skip_stages(i, len);
          }
          for (; i < len + 2; ++i) general_slice(i);
          if (!more_units) break;
          ob += (uint32_t)len;
          u = nu;
          m = nm;
        }
      }
      __syncwarp();
    }
  } else {
    // ===================== epilogue (12 warps, three per TMEM lane quarter; with the fused input transform eight, and
    // warps 12..15 transform; conv_out four, and warps 8..15 transform): see march_epilogue / march_transform =====================
    ptx::setmaxnreg_inc<kRegsMEpi>();
    if (kWideXf && p.out_fp32) {
      if (warp >= 8) march_transform<KJ, SKIP, 8>(p, sh, a_smem);
      else march_epilogue<NF, kEpiFp32, 1>(p, sh, smem, stat_part, stat_acc, cadd_s, tmem_base);
    } else if (XF && warp >= 12) {
      march_transform<KJ, SKIP, 4>(p, sh, a_smem);
    } else {
      constexpr int EW = XF ? 2 : 3;
      if (p.out_fp32) march_epilogue<NF, kEpiFp32, EW>(p, sh, smem, stat_part, stat_acc, cadd_s, tmem_base);
      else if (p.residual && p.stats) march_epilogue<NF, kEpiRes | kEpiStats, EW>(p, sh, smem, stat_part, stat_acc, cadd_s, tmem_base);
      else if (p.residual) march_epilogue<NF, kEpiRes, EW>(p, sh, smem, stat_part, stat_acc, cadd_s, tmem_base);
      else if (p.stats) march_epilogue<NF, kEpiStats, EW>(p, sh, smem, stat_part, stat_acc, cadd_s, tmem_base);
      else march_epilogue<NF, 0, EW>(p, sh, smem, stat_part, stat_acc, cadd_s, tmem_base);
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, (uint32_t)(R * NF));
  }
}
