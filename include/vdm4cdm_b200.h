/*
 * vdm4cdm_b200 -- C ABI of the B200 (sm_100a) hot path of cfpark00/vdm4cdm.
 *
 * Every entry point is extern "C", takes plain device pointers + sizes + an explicit
 * cudaStream_t (passed as void*), allocates nothing on the device (cuFFT plans excepted,
 * see vdm_pk_*), returns 0 on success or a negative VDM_E_* code, and leaves a
 * thread-local message retrievable with vdm_last_error_string().  There is no CPU
 * fallback: on a machine without an sm_100 GPU the compute entry points fail.
 *
 * The reference (pure Python) reaches these operations through PyTorch; each entry
 * point cites the reference interface it stands in for (paths relative to the
 * reference checkout; "mltools" lines are the ones recoverable from the traceback in
 * model_test.ipynb:678-692, see SURVEY.md appendix A).
 *
 * Tensor layouts
 *   activations : "channel-planar" bf16 [B][C/8][D][H][W][8]: 8 channels (16 bytes) per voxel and
 *                 plane.  Buffers may hold more planes than one tensor uses (x_planes / *_plane0
 *                 below), which makes channel concatenation a matter of where producers write.
 *   conv weights: bf16 [tap][Cin/8][Cout_pad][8]  (element (tap, ci, co) at
 *                 ((tap*Cin/8 + ci/8)*Cout_pad + co)*8 + ci%8), Cout_pad % 16 == 0
 *   latent z    : fp32 [B][D][H][W] (the reference's (B,1,D,H,W))
 *   TF32 mode   : the *_tf32 / *_f32 entry points take "fp32 channel-planar" activations [B][C/4][D][H][W][4]: 4 fp32
 *                 channels = the same 16 bytes per voxel and plane, so plane counts and plane windows (x_planes,
 *                 VdmTensor.planes, ...) count 4-channel planes there; conv weights are fp32 [tap][Cin/4][Cout_pad][4]
 *                 (vdm_pack_conv_weight_f32).  vdm_pad_circular copies 16-byte units and works on either layout.
 *   chan stats  : double [B][C][2] = (sum, sum of squares) over the D*H*W voxels
 */
#ifndef VDM4CDM_B200_H
#define VDM4CDM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define VDM_API __attribute__((visibility("default")))
#else
#define VDM_API
#endif

#define VDM_OK 0
#define VDM_E_BADARG (-1)
#define VDM_E_UNSUPPORTED (-2)
#define VDM_E_CUDA (-3)
#define VDM_E_CUFFT (-4)
#define VDM_E_DRIVER (-5)

#define VDM_MAX_TAPS 27

/* ---- library ------------------------------------------------------------------- */
VDM_API int vdm_version(void);                       /* 10000*major + 100*minor + patch */
VDM_API const char* vdm_last_error_string(void);     /* thread-local, never NULL */
/* 0 if device `dev` is an sm_100 part this library can run on, else VDM_E_UNSUPPORTED. */
VDM_API int vdm_device_supported(int dev);

/* ---- conv3d as implicit GEMM on tcgen05 ------------------------------------------
 * Stands in for every torch.nn.Conv3d executed by mltools' CUNet (forward: cuDNN conv3d
 * fprop; with transposed/flipped weights the same entry point is the dgrad), reached from
 * CUNet.forward (networks.py:259-265) -> ResNetBlock.forward (blocks.py:129-132).
 */
typedef struct VdmConvDesc {
  int32_t batch, depth, height, width;   /* B, D, H, W of input == output grid (stride 1, "same") */
  int32_t c_in;                          /* input channels read, multiple of 16 */
  int32_t c_out;                         /* real output channels written (multiple of 8 unless out_fp32) */
  int32_t c_out_pad;                     /* rows per (tap, plane) in the weight tensor, multiple of 16, <= 256 */
  int32_t n_taps;                        /* 1..27 */
  int8_t tap_offset[VDM_MAX_TAPS][3];    /* (dd, dh, dw) read offset of each tap, each in [-1, 1] */
  int32_t circular;                      /* 0: zero padding (TMA out-of-bounds fill).  1: periodic (Conv3d padding_mode="circular",
                                          *    the cropsize == 256 models, src/utils.py:460): x is a buffer with a one-voxel periodic
                                          *    halo, [B][planes][D+2][H+2][W+2][8], as written by vdm_pad_circular */
  int32_t out_fp32;                      /* 0: y is bf16 channel-planar; 1: y is fp32 [B][c_out][D][H][W] */
  int32_t x_planes, x_plane0;            /* planes per sample of the x buffer (0: c_in/8), first plane read */
  int32_t y_planes, y_plane0;            /* same for y (bf16 output only) */
  int32_t r_planes, r_plane0;            /* same for the residual */
} VdmConvDesc;

typedef struct VdmConvEpilogue {
  const float* chan_add;        /* fp32 [n_steps][B][c_out] bias + conditioning projection, or NULL */
  const int32_t* step_ptr;      /* device int: row block of chan_add to use (CUDA-graph replay), or NULL */
  int64_t chan_add_step_stride; /* elements between consecutive steps of chan_add */
  const void* residual;         /* bf16 channel-planar, same grid, c_out channels, added to the output, or NULL */
  double* stats;                /* double [B][stats_channels][2], atomically accumulated (sum, sumsq), or NULL */
  int32_t stats_channels;       /* channels per sample of the stats buffer (0: c_out) */
  int32_t stats_c0;             /* first stats channel this conv's output maps to */
  int32_t residual_upsample;    /* != 0: the residual lives on the HALF-resolution grid (D/2, H/2, W/2) and is read through a
                                 *       nearest x2 up-sampling (a 1x1x1 conv commutes with it: the up blocks' skip conv over
                                 *       cat([interpolate(h), skip]) = conv(skip) + interpolate(conv(h)));
                                 * 2: the half-resolution residual holds EIGHT blocks of c_out channels, block
                                 *       (d&1)*4 + (h&1)*2 + (w&1) for the fine voxel (d, h, w), and is read through that
                                 *       depth-to-space shuffle: the polyphase form of conv3x3x3(interpolate(a)) -- eight
                                 *       2x2x2-tap convolutions of the COARSE tensor, one per output parity (27 -> 8 taps,
                                 *       the up-sampled tensor is never written) -- lands in such a buffer */
  int32_t reserved;
  /* Fused 1x1x1 skip-path conv of a ResNet block (blocks.py ResNetBlock: h + skip_conv(x)): y += conv1x1x1(skip_x, skip_w)
   * inside the same launch, as one more channel chunk of which only the centre tap is multiplied.  Only for the
   * kd-folded layers (3x3x3, c_out <= 32, bf16 output) whose weights stay resident in shared memory;
   * VDM_E_UNSUPPORTED otherwise (the caller then runs the skip conv as its own launch).  The skip conv's bias goes
   * through chan_add or the residual. */
  const void* skip_x;           /* bf16 channel-planar tensor on the same grid (never halo-padded), or NULL */
  const void* skip_w;           /* vdm_pack_conv_weight of the (c_out, skip_c_in, 1, 1, 1) filter */
  int32_t skip_c_in;            /* 16, 32, 48 or 64; a multiple of the layer's channel chunk */
  int32_t skip_planes;          /* planes per sample of the skip_x buffer (0: skip_c_in/8) */
  int32_t skip_plane0;          /* first plane read */
  int32_t reserved2;
  /* Fused INPUT transform (inference): x holds the RAW tensor and the kernel applies GroupNorm + SiLU to every halo tile
   * in shared memory before the tensor cores read it -- stands in for the ATen group_norm + silu launches in front of
   * the conv (blocks.py:129-132: net1 / net2 = Sequential(GroupNorm, SiLU, [Dropout], Conv3d), model_test.ipynb:688-692).
   * in_norm: fp32 [batch][c_in][2] = (a, b) from vdm_gn_coef, silu(gn(x)) = h + h tanh(h) with h = a x + b; NULL: x is
   * used as it is.  Zero padding stays zero AFTER the non-linearity.  Not with circular padding (VDM_E_UNSUPPORTED);
   * the fused skip-path chunk (skip_x) is never transformed. */
  const float* in_norm;
} VdmConvEpilogue;

/* y = conv(x, w) [+ chan_add[b][co]] [+ residual]; also the dgrad when w holds the flipped,
 * transposed filter. */
VDM_API int vdm_conv3d(const VdmConvDesc* desc, const void* x, const void* w, void* y,
               const VdmConvEpilogue* epi, void* stream);

/* The same conv at TF32 precision (tcgen05.mma kind::tf32, fp32 accumulate): x, the residual and a planar y are fp32
 * channel-planar (4 channels per plane; x_planes / y_planes / r_planes and the *_plane0 windows count those planes),
 * w is vdm_pack_conv_weight_f32's layout; c_in is a multiple of 8.  The epilogue adds chan_add and the residual to the
 * fp32 accumulator and stores it unrounded; statistics are those of the stored values.  out_fp32 = 1 writes fp32
 * [B][c_out][D][H][W] as vdm_conv3d does.  in_norm, skip_x and residual_upsample are bf16-only: VDM_E_UNSUPPORTED.
 * Inference precision option: a TF32 operand keeps 10 mantissa bits against bf16's 7, and activations are never
 * rounded for storage. */
VDM_API int vdm_conv3d_tf32(const VdmConvDesc* desc, const void* x, const void* w, void* y,
                    const VdmConvEpilogue* epi, void* stream);

#ifdef VDM_BRINGUP
/* NOT part of the release library.  `make -C vdm4cdm_b200/csrc bringup` builds libvdm4cdm_b200_bringup.so with
 * -DVDM_BRINGUP, the only build in which this symbol and the ablation branches of the conv kernel exist
 * (tools/bench_epilogue.py, tools/bench_conv.py load it with VDM4CDM_BRINGUP=1).  Knobs (value 0 = automatic): 1 force
 * MT, 2 force KC, 3 force n_split, 4 no resident weights, 5 ablation flags (timing experiments; results are wrong by
 * construction), 6 no kd-folded schedule (1: resident variants off, 2: all off). */
#define VDM_BRINGUP_API __attribute__((visibility("default")))
VDM_BRINGUP_API int vdm_debug_set(int key, int value);
#endif

/* ---- conv3d weight gradient (tcgen05, both operands MN-major straight from the planar tensors) ----
 * Stands in for the cuDNN conv3d backward-filter autograd launches for every torch.nn.Conv3d of the
 * CUNet during LightVDM / LightSFM training_step (ctor + Trainer.fit:
 * trainVDM3D128_c_c_from_field_name_thick_lowbatch.py:128-160; trainSFM3D160_...:124-150).
 *   dw[tap][ci][co] += sum_{b,d,h,w} a[b][ci][d+kd-p][h+kh-p][w+kw-p] * g[b][co][d][h][w]
 * a: the conv's input activations, g: the gradient of its output, both channel-planar bf16 on the same
 * grid; dw: fp32 [kernel^3][c_in][c_out], ACCUMULATED with atomics (the caller zeroes it or keeps
 * accumulating micro-batches into a gradient bucket). */
typedef struct VdmWgradDesc {
  int32_t batch, depth, height, width;
  int32_t c_in;                 /* channels of `a` read, multiple of 16 */
  int32_t c_out;                /* real channels of g, 1..256; the g window must hold c_out rounded up to 16 */
  int32_t kernel;               /* 3 (3x3x3, zero padding 1) or 1 */
  int32_t a_planes, a_plane0;   /* planes per sample of the a buffer (0: c_in/8), first plane read */
  int32_t g_planes, g_plane0;   /* same for g */
  /* dw addressing (elements): dw[tap*stride_tap + ci*stride_ci + co*stride_co], rows ci >= c_in_real skipped.
   * All three strides 0 selects the packed default [tap][c_in][c_out] (c_in_real = c_in).  torch's Conv3d
   * layout (c_out, c_in_real, k, k, k) is stride_tap = 1, stride_ci = k^3, stride_co = c_in_real*k^3, which lets
   * the kernel accumulate straight into the parameter's .grad inside a flat gradient bucket. */
  int64_t dw_stride_tap, dw_stride_ci, dw_stride_co;
  int32_t c_in_real;
  int32_t a_padded;             /* 1: `a` carries a one-voxel periodic halo ([D+2][H+2][W+2], circular convs) */
  int32_t g_padded;             /* 1: so does g (required with a_padded for 3x3x3 filters: the kw taps of the narrow-layer
                                 *    kernel read w-shifted g tiles, which must wrap periodically too) */
} VdmWgradDesc;

VDM_API int vdm_conv3d_wgrad(const VdmWgradDesc* desc, const void* a, const void* g, float* dw, void* stream);

/* fp32 torch Conv3d weight (c_out, c_in, k, k, k) -> bf16 kernel layout [k^3][c_in_pad/8][c_out_pad][8], zero padded
 * (what vdm_conv3d reads).  transpose_flip != 0 packs the dgrad filter instead: the roles of c_in / c_out are
 * exchanged and the taps mirrored; [ci0, ci0 + n_ci) then selects the slice of the conv's INPUT channels that
 * becomes the dgrad's output channels (dgrads of convs with more than 256 input channels run as several launches).
 * c_in_pad / c_out_pad are the padded sizes of the PACKED tensor's K and N dimensions (multiples of 16). */
VDM_API int vdm_pack_conv_weight(const float* w, void* packed, int c_out, int c_in, int kernel, int transpose_flip,
                         int ci0, int n_ci, int c_in_pad, int c_out_pad, void* stream);
/* Forward filter for vdm_conv3d_tf32: fp32 [k^3][c_in_pad/4][c_out_pad][4], every weight rounded to the nearest TF32
 * value (cvt.rna.tf32.f32), zero padded; c_in_pad a multiple of 8, c_out_pad of 16. */
VDM_API int vdm_pack_conv_weight_f32(const float* w, void* packed, int c_out, int c_in, int kernel, int c_in_pad,
                             int c_out_pad, void* stream);

/* The same for a whole network in ONE launch: `jobs_device` is an array of n_jobs descriptors IN DEVICE MEMORY (the
 * arguments of vdm_pack_conv_weight with k3 = kernel^3; pointers must stay valid, e.g. for a captured CUDA graph).
 * Replaces the ~56 per-filter launches of a training step (forward and dgrad variants of every Conv3d). */
typedef struct VdmPackJob {
  const float* w;
  void* packed;
  int32_t c_out, c_in, k3, transpose_flip, ci0, n_ci, c_in_pad, c_out_pad;
} VdmPackJob;
VDM_API int vdm_pack_conv_weight_batched(const VdmPackJob* jobs_device, int n_jobs, void* stream);

/* ---- fused elementwise passes (ATen group_norm / silu / dropout / avg_pool3d / interpolate /
 *      cat in the reference's ResNetBlock / ResNetDown; blocks.py:129-170) ------------------- */

/* View of `channels` consecutive channels inside a channel-planar buffer: plane (b, p) of the view
 * starts at data + ((b*planes + plane0 + p) * voxels) * 16 bytes. */
typedef struct VdmTensor {
  void* data;
  int32_t planes;   /* planes per sample of the whole buffer */
  int32_t plane0;   /* first plane of this view */
} VdmTensor;

/* stats[b][stats_c0 + c] += (sum, sumsq) of x over voxels; stats must be zeroed by the caller. */
VDM_API int vdm_channel_stats(const VdmTensor* x, int batch, int64_t voxels, int channels, double* stats,
                      int stats_channels, int stats_c0, void* stream);

/* y = dropout(silu(groupnorm(x))) ; statistics come from `stats` (double [B][channels][2]).
 * dropout_p == 0 disables dropout; otherwise keep-mask = Philox(seed, layer_tag, element). */
VDM_API int vdm_gn_silu(const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels, int groups,
                const double* stats, const float* gamma, const float* beta, float eps,
                float dropout_p, uint64_t seed, uint32_t layer_tag, void* stream);

/* silu(groupnorm(.)) restricted to channels [c_off, c_off + channels) of a channels_total-channel norm whose
 * statistics are stats (double [B][channels_total][2], of the tensor at the resolution of y); gamma / beta are the
 * norm's full vectors.  (depth, height, width) is the grid of y.  upsample != 0: x is at HALF that resolution and
 * y = silu(gn(nearest_upsample2(x))) -- the up blocks' torch.cat([interpolate(h), skip]) -> GroupNorm -> SiLU
 * (blocks.py ResNetUp / ResNetBlock.net1) without ever writing the up-sampled tensor (its per-channel sums are 8x
 * the coarse tensor's).  upsample == 2: x AND y are at half the resolution of (depth, height, width), the grid the
 * statistics refer to: y = silu(gn(x)) of the coarse tensor itself, the input of the polyphase up-conv (eight 2x2x2-tap
 * convolutions on the coarse grid, VdmConvEpilogue.residual_upsample == 2).  No dropout: net1 has none. */
VDM_API int vdm_gn_silu_view(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                     int channels, int c_off, int channels_total, int groups, const double* stats,
                     const float* gamma, const float* beta, float eps, int upsample, void* stream);
/* (a, b) pairs for VdmConvEpilogue.in_norm from the fp64 (sum, sumsq) statistics of the tensor: fp32 [batch][channels][2]. */
VDM_API int vdm_gn_coef(const double* stats, int batch, int channels, int groups, int64_t voxels, const float* gamma,
                const float* beta, float eps, float* coef, void* stream);
/* Same with the dropout seed advanced on the device: seed_eff = seed + *seed_step (CUDA-graph replay). */
VDM_API int vdm_gn_silu_step(const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels, int groups,
                     const double* stats, const float* gamma, const float* beta, float eps, float dropout_p,
                     uint64_t seed, const int32_t* seed_step, uint32_t layer_tag, void* stream);

/* vdm_gn_silu on fp32 channel-planar views (4 channels per plane; channels a multiple of 4), without dropout.  SiLU is
 * x / (1 + exp(-x)) in fp32 (not the ~2^-11 hardware tanh of the bf16 passes). */
VDM_API int vdm_gn_silu_f32(const VdmTensor* x, const VdmTensor* y, int batch, int64_t voxels, int channels, int groups,
                    const double* stats, const float* gamma, const float* beta, float eps, void* stream);

/* 2x2x2 average pooling of a (depth,height,width) grid; accumulates channel stats of y when stats != NULL. */
VDM_API int vdm_avgpool2(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                 int channels, double* stats, int stats_channels, int stats_c0, void* stream);

/* y = nearest_upsample_x2(coarse); (depth,height,width) is the fine grid.  Writing into a plane
 * window of a wider buffer is how channel concatenation with the skip tensor happens.
 * Accumulates channel stats of y when stats != NULL. */
VDM_API int vdm_upsample2(const VdmTensor* coarse, const VdmTensor* y, int batch, int depth, int height, int width,
                  int channels, double* stats, int stats_channels, int stats_c0, void* stream);
/* vdm_avgpool2 / vdm_upsample2 on fp32 channel-planar views (statistics of the fp32 values). */
VDM_API int vdm_avgpool2_f32(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                     int channels, double* stats, int stats_channels, int stats_c0, void* stream);
VDM_API int vdm_upsample2_f32(const VdmTensor* coarse, const VdmTensor* y, int batch, int depth, int height, int width,
                      int channels, double* stats, int stats_channels, int stats_c0, void* stream);

/* ---- backward of the fused elementwise passes (autograd's native_group_norm_backward /
 *      silu_backward / dropout mask / avg_pool3d_backward / upsample_nearest3d_backward launches
 *      during training_step) ----------------------------------------------------------------------
 * For y = dropout(silu(u)), u = gamma*xhat + beta, xhat = (x - mean_g)*rstd_g:
 *   du = dy * keep/(1-p) * silu'(u)
 *   reduce: sums[b][c] += (sum_v du, sum_v du*xhat)            (-> dbeta, dgamma after a sum over b)
 *   apply : dx = rstd_g*(gamma_c*du - mean_g(gamma*du) - xhat*mean_g(gamma*du*xhat)) [+ add]
 * `stats` are the forward statistics of x (double [B][channels][2]); the dropout mask is regenerated
 * from (seed, layer_tag).  apply also accumulates (sum, sumsq) of dx into out_stats when not NULL
 * (the per-sample channel sums are the gradients of the conv bias / conditioning rows).
 * `sums` is a window of a double [B][sums_channels][2] table starting at channel sums_c0 (sums_channels = 0:
 * a tight [B][channels][2]).  seed_step (device int32, may be NULL) is added to the dropout seed on the device,
 * so a captured CUDA graph draws a new mask every replay. */
VDM_API int vdm_gn_silu_bwd_reduce(const VdmTensor* x, const VdmTensor* dy, int batch, int64_t voxels, int channels,
                           int groups, const double* stats, const float* gamma, const float* beta, float eps,
                           float dropout_p, uint64_t seed, const int32_t* seed_step, uint32_t layer_tag, double* sums,
                           int sums_channels, int sums_c0, void* stream);
VDM_API int vdm_gn_silu_bwd_apply(const VdmTensor* x, const VdmTensor* dy, const VdmTensor* add, const VdmTensor* dx,
                          int batch, int64_t voxels, int channels, int groups, const double* stats,
                          const float* gamma, const float* beta, float eps, float dropout_p, uint64_t seed,
                          const int32_t* seed_step, uint32_t layer_tag, const double* sums, int sums_channels,
                          int sums_c0, double* out_stats, int out_stats_channels, int out_stats_c0, void* stream);

/* Gradient of vdm_avgpool2: dx = (accumulate ? dx : 0) + nearest_upsample_x2(dy) / 8 on the fine grid
 * (depth,height,width); stats (optional) accumulate (sum, sumsq) of the resulting dx. */
VDM_API int vdm_avgpool2_bwd(const VdmTensor* dy, const VdmTensor* dx, int batch, int depth, int height, int width,
                     int channels, int accumulate, double* stats, int stats_channels, int stats_c0, void* stream);

/* Gradient of vdm_upsample2: dcoarse = sum of the 2x2x2 fine gradients; (depth,height,width) is the fine grid. */
VDM_API int vdm_upsample2_bwd(const VdmTensor* dy, const VdmTensor* dcoarse, int batch, int depth, int height, int width,
                      int channels, double* stats, int stats_channels, int stats_c0, void* stream);

/* ---- training-batch preparation: periodic crop + log-normalise + flip + permute in one gather -----------------
 * AstroDataset.__getitem__ (src/dataset/CAMELS_3D_dataset.py:53-74) with Crop / LogTransform / Normalize / Flip /
 * Permutate (src/dataset/augmentation.py:8-127).  in: fp32 [S0][S1][S2] raw box; out: fp32 [n0][n1][n2] with
 * n[d] = crop_size[perm[d]]:
 *   out[o] = do_log ? (log10(in[src] + alpha) - mean) / std : in[src],
 *   cropped index c with c[perm[d]] = o[d];  c'[a] = flip[a] ? crop_size[a]-1-c[a] : c[a];  src[a] = (anchor[a] + c'[a]) mod S[a].
 * All five index arrays are HOST int32[3]. */
VDM_API int vdm_augment_crop(const float* in, float* out, const int32_t* full_size, const int32_t* crop_size,
                     const int32_t* anchor, const int32_t* flip, const int32_t* perm, float alpha, float mean, float std,
                     int do_log, void* stream);

/* ---- optimizer step on a flat fp32 parameter bucket (torch.optim.AdamW + Trainer(gradient_clip_val=0.5),
 *      trainVDM3D128_c_c_from_field_name_thick_lowbatch.py:134-160) --------------------------------- */
/* *out += sum_i x[i]^2 (double, atomically). */
VDM_API int vdm_sumsq(const float* x, int64_t n, double* out, void* stream);
/* AdamW with decoupled weight decay; the gradient is first multiplied by grad_scale (1/world for a
 * summed all-reduce) and by min(1, max_norm / (grad_scale*sqrt(*grad_sumsq) + 1e-6)) when grad_sumsq != NULL
 * and max_norm > 0 (torch.nn.utils.clip_grad_norm_).  `step` is the 1-based step number. */
VDM_API int vdm_adamw_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                   float beta1, float beta2, float eps, float weight_decay, int step, const double* grad_sumsq,
                   float max_norm, float grad_scale, void* stream);
/* Same with the step number read from the device: step_eff = step + *step_ptr (CUDA-graph replay). */
VDM_API int vdm_adamw_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                       float beta1, float beta2, float eps, float weight_decay, int step, const int32_t* step_ptr,
                       const double* grad_sumsq, float max_norm, float grad_scale, void* stream);

/* ---- continuous-time VDM training loss around the denoiser call (mltools vdm_model.py:429-442 in model_test.ipynb:680;
 *      restated in oracle/vdm_ref.py:158-184).  gamma(t) = *gamma_b + |*gamma_w| t when learned != 0 (LearnedLinearSchedule),
 *      *gamma_b + *gamma_w t otherwise; the schedule parameters are read from DEVICE memory (CUDA-graph replay of a training
 *      step).  All tensors fp32 [batch][n], n % 4 == 0, 16-byte aligned. ---- */

/* z_t = alpha_t x + sigma_t noise with alpha^2 = sigmoid(-gamma(times[b])), sigma^2 = sigmoid(gamma(times[b])). */
VDM_API int vdm_loss_zt(const float* x, const float* noise, const float* times, const float* gamma_b, const float* gamma_w,
                int learned, float* zt, int batch, int64_t n, void* stream);
/* Backward of vdm_loss_zt with respect to the schedule: grads2 = (d b, d w) from g_zt = dL/dz_t.
 * work: 2 * batch doubles of scratch. */
VDM_API int vdm_loss_zt_bwd(const float* g_zt, const float* x, const float* noise, const float* times, const float* gamma_b,
                    const float* gamma_w, int learned, double* work, float* grads2, int batch, int64_t n, void* stream);
/* out8 = (loss, diffusion, latent, reconstruction) in bits per dimension (batch means), then k gamma' (the scalar of
 * d eps_hat, k = 1 / (batch n log 2)), d b and d w of the three terms at fixed eps_hat, and one unused float.
 * work: 3 * batch doubles of scratch. */
VDM_API int vdm_loss_terms(const float* pred, const float* noise, const float* x, const float* noise0, const float* gamma_b,
                   const float* gamma_w, int learned, double data_noise, double* work, float* out8, int batch, int64_t n,
                   void* stream);
/* d_pred = *g_loss * *coef * (pred - noise)  (coef = out8[4] of vdm_loss_terms; g_loss = dL/dloss), total elements. */
VDM_API int vdm_loss_dpred(const float* pred, const float* noise, const float* coef, const float* g_loss, float* d_pred,
                   int64_t total, void* stream);

/* Periodic one-voxel halo: y[b][p][dp][hp][wp] = x[b][p][(dp-1) mod D][(hp-1) mod H][(wp-1) mod W] for
 * dp in [0, D+2) etc.  x: [B][planes][D][H][W][8] view, y: [B][planes][D+2][H+2][W+2][8] view.  The kernel copies
 * 16-byte units: an fp32 channel-planar tensor is padded by passing 2 * its channel count (= 8 * its planes). */
VDM_API int vdm_pad_circular(const VdmTensor* x, const VdmTensor* y, int batch, int depth, int height, int width,
                     int channels, void* stream);

/* Pack the network input: plane 0 of out = (z, cond_1..cond_n, 0...) per voxel, planes 1.. = 0.
 * z: fp32 [B][V]; cond: fp32 [B][n_cond][V] (NCDHW) or NULL; out: c_pad/8 planes; n_cond <= 7. */
VDM_API int vdm_pack_input(const float* z, const float* cond, const VdmTensor* out, int batch, int64_t voxels,
                   int n_cond, int c_pad, void* stream);
/* The same into an fp32 channel-planar tensor: planes 0 and 1 hold (z, cond_1..cond_n, 0...), the rest are 0;
 * c_pad a multiple of 8, n_cond <= 7. */
VDM_API int vdm_pack_input_f32(const float* z, const float* cond, const VdmTensor* out, int batch, int64_t voxels,
                       int n_cond, int c_pad, void* stream);

/* ---- fused VDM ancestral-sampler update ------------------------------------------------
 * VDM.sample_zs_given_zt (vdm_model.py:370-378): mean = alpha_s/alpha_t*(zt - c*sigma_t*eps_hat),
 * z_s = mean + sigma_s*sqrt(c)*N(0,1).  coef[step] = (w_z, w_eps, noise_scale, out_scale):
 *   z_out = out_scale * (w_z * z + w_eps * eps_hat + noise_scale * noise)
 * noise = Philox4x32-10 + Box-Muller keyed by (seed, realisation_id[b], draw, element), or
 * `noise_in` (fp32 [B][V]) when it is not NULL (injected noise, parity tests).
 * When packed_out != NULL (plane 0 of sample 0 of a packed network input with `packed_planes`
 * planes per sample, see vdm_pack_input) also rewrites that plane for the next step.
 * step_ptr == NULL means step 0 of coef / draw = draw_base. */
VDM_API int vdm_sampler_step(const float* z, const float* eps_hat, float* z_out, int batch, int64_t voxels,
                     const float* coef, const int32_t* step_ptr, uint64_t seed,
                     const int32_t* realisation_id, int32_t draw_base, const float* noise_in,
                     const float* cond, int n_cond, void* packed_out, int packed_planes, void* stream);

/* out[b][v] = N(0,1) noise of draw `draw` (the definition used by vdm_sampler_step). */
VDM_API int vdm_philox_normal(float* out, int batch, int64_t voxels, uint64_t seed,
                      const int32_t* realisation_id, int32_t draw, void* stream);

/* step counter helper for CUDA-graph replay: *counter += 1 on the stream. */
VDM_API int vdm_increment(int32_t* counter, void* stream);

/* ---- P(k) / r(k): cuFFT R2C + k-shell binning ---------------------------------------------
 * power() at src/utils.py:16-83 (and pk :85-102, get_ccs :110-128).  `fields` is fp32
 * [n_fields][batch][chan][n0][n1][n2] (n0 == 1 for 2-D inputs); for every field the spectrum is
 * the batch mean of the channel sum of Re(X conj(X2)), binned by ceil(|k|) with Hermitian
 * weights.  Outputs are per field and per bin 1..kmax (kmax = min(n)//2):
 *   k_mean, p_mean : double [n_fields][kmax];  n_modes : int64 [n_fields][kmax].
 * fields2 == NULL computes the auto spectrum.  `work` is a caller-owned complex64 scratch of
 * vdm_pk_work_bytes(...) bytes.  cuFFT plans are cached inside the library per (dims, count). */
VDM_API size_t vdm_pk_work_bytes(int n_fields, int batch, int chan, int n0, int n1, int n2, int cross);
VDM_API int vdm_pk(const float* fields, const float* fields2, int n_fields, int batch, int chan, int n0,
           int n1, int n2, void* work, size_t work_bytes, double* k_mean, double* p_mean,
           int64_t* n_modes, void* stream);
/* One pass over two transforms: P11, P22 and P12 together (get_ccs without the four FFTs). */
VDM_API int vdm_pk_cross3(const float* fields1, const float* fields2, int n_fields, int batch, int chan,
                  int n0, int n1, int n2, void* work, size_t work_bytes, double* k_mean,
                  double* p11, double* p22, double* p12, int64_t* n_modes, void* stream);

/* ---- log-PDF histograms (calc_SS.py:51-65 get_logpdf_3d / get_logpdf_2d) -----------------------------------------
 * counts[f][b] += #{voxels v of field f : log10(fields[f][v] + add) in bin b} for nbins equal bins on [lo, hi]
 * (numpy.histogram semantics: left-closed bins, the last one closed on the right, values outside ignored).
 * fields: fp32 [n_fields][voxels]; counts: int64 [n_fields][nbins], accumulated (the caller zeroes it). */
VDM_API int vdm_log_histogram(const float* fields, int n_fields, int64_t voxels, float add, double lo, double hi, int nbins,
                      int64_t* counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VDM4CDM_B200_H */
