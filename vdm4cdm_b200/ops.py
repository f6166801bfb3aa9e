"""Torch-tensor front end of the C ABI (``include/vdm4cdm_b200.h``): every function here checks
shapes/dtypes, hands raw device pointers and the current CUDA stream to ``libvdm4cdm_b200.so`` and
raises ``RuntimeError`` on failure.  There is no PyTorch fallback for any of them.

Channel-planar activations are torch bf16 tensors of shape ``[B, P, D, H, W, 8]`` (P planes of 8
channels); a *view* ``(buf, plane0, channels)`` addresses ``channels`` consecutive channels of a
wider buffer, which is how channel concatenation is expressed without copies.

The TF32 inference mode uses fp32 channel-planar tensors ``[B, P, D, H, W, 4]`` (P planes of 4 channels, the same
16 bytes per voxel and plane).  ``conv3d``, ``gn_silu``, ``avgpool2``, ``upsample2``, ``pad_circular``, ``pack_input``
and ``pack_conv_weight_into`` dispatch on the planar tensors' dtype; mixing bf16 and fp32 in one call raises
``ValueError``.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Sequence, Tuple

import torch

from . import _C

TAPS_3X3X3 = tuple((kd - 1, kh - 1, kw - 1) for kd in range(3) for kh in range(3) for kw in range(3))
TAPS_1X1X1 = ((0, 0, 0),)


_LAUNCHES = 0


def launch_count() -> int:
    """Kernels of libvdm4cdm_b200.so launched through this module so far (cuFFT's own kernels not counted)."""
    return _LAUNCHES


def _launched(n: int = 1) -> None:
    global _LAUNCHES
    _LAUNCHES += n


_CONV_PROFILE = None


def set_conv_profiler(records) -> None:
    """bench.py hook: when ``records`` is a list, every conv3d call appends (start_event, end_event, flops)
    recorded on the launching stream; ``None`` switches it off."""
    global _CONV_PROFILE
    _CONV_PROFILE = records


_PROFILE_TAG = ""


def set_profile_tag(tag: str) -> None:
    """Prefix for the labels the conv profiler records (``"dgrad "`` while the backward pass issues dgrads)."""
    global _PROFILE_TAG
    _PROFILE_TAG = tag


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need(cond: bool, msg: str) -> None:
    if not cond:
        raise ValueError(msg)


def _planar_ok(t: torch.Tensor, name: str) -> None:
    _need(t.is_cuda and t.dtype == torch.bfloat16 and t.dim() == 6 and t.shape[-1] == 8 and t.is_contiguous(),
          f"{name}: expected a contiguous CUDA bf16 [B,P,D,H,W,8] tensor, got {tuple(t.shape)} {t.dtype} {t.device}")


_LANES = {torch.bfloat16: 8, torch.float32: 4}       # channels per 16-byte plane of a planar tensor


def _planar_lanes(t: torch.Tensor, name: str) -> int:
    """Channels per plane (8: bf16, 4: fp32) of a contiguous CUDA channel-planar tensor."""
    lanes = _LANES.get(t.dtype)
    _need(t.is_cuda and lanes is not None and t.dim() == 6 and t.shape[-1] == lanes and t.is_contiguous(),
          f"{name}: expected a contiguous CUDA bf16 [B,P,D,H,W,8] or fp32 [B,P,D,H,W,4] tensor, got "
          f"{tuple(t.shape)} {t.dtype} {t.device}")
    return lanes


def _same_lanes(lanes: int, t: torch.Tensor, name: str) -> None:
    _need(_planar_lanes(t, name) == lanes, f"{name}: bf16 and fp32 planar tensors mixed in one call")


def _view(t: torch.Tensor, plane0: int) -> _C.Tensor:
    return _C.Tensor(t.data_ptr(), t.shape[1], plane0)


# ---- layout helpers (host-side glue; run on whatever device the tensor lives on) -------------------
def to_planar(x: torch.Tensor, pad_to: int = 8, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """(B, C, D, H, W) any float dtype -> bf16 [B, ceil(C/pad_to)*pad_to/8, D, H, W, 8] (zero padded), or with
    ``dtype=torch.float32`` fp32 [B, ceil(C/pad_to)*pad_to/4, D, H, W, 4]."""
    lanes = _LANES[dtype]
    b, c, d, h, w = x.shape
    cp = -(-c // pad_to) * pad_to
    if cp != c:
        x = torch.cat([x, x.new_zeros(b, cp - c, d, h, w)], dim=1)
    return x.reshape(b, cp // lanes, lanes, d, h, w).permute(0, 1, 3, 4, 5, 2).contiguous().to(dtype)


def from_planar(x: torch.Tensor, channels: Optional[int] = None) -> torch.Tensor:
    """bf16 [B, P, D, H, W, 8] or fp32 [B, P, D, H, W, 4] -> fp32 (B, C, D, H, W)."""
    b, p, d, h, w, lanes = x.shape
    y = x.permute(0, 1, 5, 2, 3, 4).reshape(b, p * lanes, d, h, w).float()
    return y if channels is None else y[:, :channels]


def pack_conv_weight(w: torch.Tensor, c_in_pad: Optional[int] = None, c_out_pad: Optional[int] = None,
                     transpose_flip: bool = False) -> torch.Tensor:
    """torch Conv3d weight (Cout, Cin, kd, kh, kw) -> bf16 [taps][Cin_pad/8][Cout_pad][8].

    ``transpose_flip=True`` packs the dgrad filter: roles of Cin/Cout exchanged and taps mirrored.
    Tap order matches ``TAPS_3X3X3`` / ``TAPS_1X1X1``.
    """
    if transpose_flip:
        w = w.transpose(0, 1).flip(2, 3, 4)
    co, ci, kd, kh, kw = w.shape
    cip = -(-ci // 16) * 16 if c_in_pad is None else c_in_pad
    cop = -(-co // 16) * 16 if c_out_pad is None else c_out_pad
    t = w.permute(2, 3, 4, 1, 0).reshape(kd * kh * kw, ci, co).float()
    full = t.new_zeros(kd * kh * kw, cip, cop)
    full[:, :ci, :co] = t
    return full.reshape(kd * kh * kw, cip // 8, 8, cop).permute(0, 1, 3, 2).contiguous().to(torch.bfloat16)


def packed_weight_shape(conv_weight_shape, transpose_flip: bool = False, n_ci: Optional[int] = None,
                        dtype: torch.dtype = torch.bfloat16):
    """Shape of the packed bf16 filter for a torch Conv3d weight (Cout, Cin, k, k, k); with ``dtype=torch.float32`` the
    TF32 forward filter [k^3, ceil(Cin/8)*2, Cout_pad, 4]."""
    co, ci, k = conv_weight_shape[0], conv_weight_shape[1], conv_weight_shape[2]
    if dtype == torch.float32:
        _need(not transpose_flip, "packed_weight_shape: the fp32 (TF32) filter is forward-only")
        return (k ** 3, -(-ci // 8) * 8 // 4, -(-co // 16) * 16, 4)
    if transpose_flip:
        kdim, ndim = co, (ci if n_ci is None else n_ci)
    else:
        kdim, ndim = ci, co
    return (k ** 3, -(-kdim // 16) * 16 // 8, -(-ndim // 16) * 16, 8)


def pack_conv_weight_into(w: torch.Tensor, out: torch.Tensor, transpose_flip: bool = False, ci0: int = 0,
                          n_ci: Optional[int] = None) -> torch.Tensor:
    """``vdm_pack_conv_weight``: fp32 CUDA Conv3d weight -> ``out`` (bf16 [k^3, K_pad/8, N_pad, 8]) in one launch.
    With ``transpose_flip`` the dgrad filter of input channels [ci0, ci0 + n_ci) is packed.  An fp32 ``out``
    ([k^3, K_pad/4, N_pad, 4], ``packed_weight_shape(..., dtype=torch.float32)``) receives the TF32-rounded forward
    filter of ``vdm_conv3d_tf32`` (``vdm_pack_conv_weight_f32``)."""
    _need(w.is_cuda and w.dtype == torch.float32 and w.is_contiguous() and w.dim() == 5, "pack_conv_weight_into: w must be contiguous CUDA fp32 (Cout, Cin, k, k, k)")
    co, ci, k = w.shape[0], w.shape[1], w.shape[2]
    if out.dtype == torch.float32:
        _need(not transpose_flip and ci0 == 0 and n_ci in (None, ci), "pack_conv_weight_into: the fp32 (TF32) filter is forward-only")
        _need(out.is_cuda and out.is_contiguous() and tuple(out.shape) == packed_weight_shape(w.shape, dtype=torch.float32),
              "pack_conv_weight_into: bad out tensor")
        rc = _C.lib().vdm_pack_conv_weight_f32(w.data_ptr(), out.data_ptr(), co, ci, k, out.shape[1] * 4, out.shape[2], _stream())
        _C.check(rc, "vdm_pack_conv_weight_f32")
        _launched(1)
        return out
    n_ci = ci if n_ci is None else n_ci
    _need(out.is_cuda and out.dtype == torch.bfloat16 and out.is_contiguous() and
          tuple(out.shape) == packed_weight_shape(w.shape, transpose_flip, n_ci), "pack_conv_weight_into: bad out tensor")
    rc = _C.lib().vdm_pack_conv_weight(w.data_ptr(), out.data_ptr(), co, ci, k, 1 if transpose_flip else 0, ci0, n_ci,
                                       out.shape[1] * 8, out.shape[2], _stream())
    _C.check(rc, "vdm_pack_conv_weight")
    _launched(1)
    return out


def pack_job_table(jobs, device) -> torch.Tensor:
    """Device copy of a ``VdmPackJob`` array for ``pack_conv_weights_batched``.  ``jobs``: (w fp32 CUDA (Cout, Cin, k, k, k)
    contiguous, out bf16 packed buffer, transpose_flip, ci0, n_ci) tuples; the tensors must outlive the table."""
    arr = (_C.PackJob * len(jobs))()
    for j, (w, out, transpose_flip, ci0, n_ci) in zip(arr, jobs):
        _need(w.is_cuda and w.dtype == torch.float32 and w.is_contiguous() and w.dim() == 5, "pack_job_table: bad weight")
        _need(out.is_cuda and out.dtype == torch.bfloat16 and out.is_contiguous() and
              tuple(out.shape) == packed_weight_shape(w.shape, transpose_flip, n_ci), "pack_job_table: bad out tensor")
        j.w, j.packed = w.data_ptr(), out.data_ptr()
        j.c_out, j.c_in, j.k3 = w.shape[0], w.shape[1], w.shape[2] ** 3
        j.transpose_flip, j.ci0, j.n_ci = (1 if transpose_flip else 0), ci0, n_ci
        j.c_in_pad, j.c_out_pad = out.shape[1] * 8, out.shape[2]
    raw = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
    return raw.to(device)


def pack_conv_weights_batched(table: torch.Tensor, n_jobs: int) -> None:
    """``vdm_pack_conv_weight_batched``: every job of ``pack_job_table`` in one launch."""
    rc = _C.lib().vdm_pack_conv_weight_batched(table.data_ptr(), n_jobs, _stream())
    _C.check(rc, "vdm_pack_conv_weight_batched")
    _launched(1)


# ---- VDM training loss (csrc/vdm_loss.cu) ---------------------------------------------------------------
def _loss_args_ok(*tensors):
    n = tensors[0][0].numel()
    for t in tensors:
        _need(t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == tensors[0].shape,
              "VDM loss kernels take contiguous fp32 CUDA tensors of one shape")
    _need(n % 4 == 0, "VDM loss kernels need a multiple of 4 elements per sample")
    return tensors[0].shape[0], n


def loss_zt(x, noise, times, gamma_b, gamma_w, learned: bool) -> torch.Tensor:
    """``vdm_loss_zt``: z_t = alpha_t x + sigma_t noise, schedule parameters read on the device."""
    b, n = _loss_args_ok(x, noise)
    zt = torch.empty_like(x)
    rc = _C.lib().vdm_loss_zt(x.data_ptr(), noise.data_ptr(), times.data_ptr(), gamma_b.data_ptr(), gamma_w.data_ptr(),
                              1 if learned else 0, zt.data_ptr(), b, n, _stream())
    _C.check(rc, "vdm_loss_zt")
    _launched(1)
    return zt


def loss_zt_bwd(g_zt, x, noise, times, gamma_b, gamma_w, learned: bool) -> torch.Tensor:
    """``vdm_loss_zt_bwd``: fp32 [2] = (d b, d w) of the schedule through z_t."""
    b, n = _loss_args_ok(g_zt, x, noise)
    work = torch.empty(2 * b, dtype=torch.float64, device=x.device)
    out = torch.empty(2, dtype=torch.float32, device=x.device)
    rc = _C.lib().vdm_loss_zt_bwd(g_zt.data_ptr(), x.data_ptr(), noise.data_ptr(), times.data_ptr(), gamma_b.data_ptr(),
                                  gamma_w.data_ptr(), 1 if learned else 0, work.data_ptr(), out.data_ptr(), b, n, _stream())
    _C.check(rc, "vdm_loss_zt_bwd")
    _launched(2)
    return out


def loss_terms(pred, noise, x, noise0, gamma_b, gamma_w, learned: bool, data_noise: float) -> torch.Tensor:
    """``vdm_loss_terms``: fp32 [8] = (loss, diffusion, latent, reconstruction, k gamma', d b, d w, -)."""
    b, n = _loss_args_ok(pred, noise, x, noise0)
    work = torch.empty(3 * b, dtype=torch.float64, device=x.device)
    out = torch.empty(8, dtype=torch.float32, device=x.device)
    rc = _C.lib().vdm_loss_terms(pred.data_ptr(), noise.data_ptr(), x.data_ptr(), noise0.data_ptr(), gamma_b.data_ptr(),
                                 gamma_w.data_ptr(), 1 if learned else 0, float(data_noise), work.data_ptr(), out.data_ptr(),
                                 b, n, _stream())
    _C.check(rc, "vdm_loss_terms")
    _launched(2)
    return out


def loss_dpred(pred, noise, coef, g_loss) -> torch.Tensor:
    """``vdm_loss_dpred``: d eps_hat = g_loss * coef * (eps_hat - eps) (coef, g_loss: one-element fp32 CUDA tensors)."""
    _loss_args_ok(pred, noise)
    d = torch.empty_like(pred)
    rc = _C.lib().vdm_loss_dpred(pred.data_ptr(), noise.data_ptr(), coef.data_ptr(), g_loss.data_ptr(), d.data_ptr(),
                                 pred.numel(), _stream())
    _C.check(rc, "vdm_loss_dpred")
    _launched(1)
    return d


UnsupportedFusion = _C.UnsupportedFusion


# ---- conv ------------------------------------------------------------------------------------------
def conv3d(x: torch.Tensor, w_packed: torch.Tensor, c_out: int, *, taps: Sequence[Tuple[int, int, int]] = TAPS_3X3X3,
           x_plane0: int = 0, c_in: Optional[int] = None, out: Optional[torch.Tensor] = None, out_plane0: int = 0,
           out_fp32: bool = False, chan_add: Optional[torch.Tensor] = None, step_ptr: Optional[torch.Tensor] = None,
           residual: Optional[torch.Tensor] = None, residual_plane0: int = 0, stats: Optional[torch.Tensor] = None,
           stats_c0: int = 0, circular: bool = False, residual_upsample=False,
           skip_x: Optional[torch.Tensor] = None, skip_w: Optional[torch.Tensor] = None, skip_plane0: int = 0,
           in_norm: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``vdm_conv3d``: y = conv(x, w) [+ chan_add[b, co]] [+ residual], optional GroupNorm statistics.
    ``residual_upsample``: the residual lives on the half-resolution grid and is added through a nearest x2 up-sampling.
    ``skip_x`` / ``skip_w``: y += conv1x1x1(skip_x[window at skip_plane0], skip_w) fused into the launch (narrow
    kd-folded layers only; raises ``UnsupportedFusion`` when the layer cannot take it).

    ``in_norm`` (``gn_coef`` output, fp32 [B, c_in, 2]): ``x`` is the RAW tensor and the kernel applies GroupNorm + SiLU to
    every input tile on the fly (raises ``UnsupportedFusion`` where the layer cannot take it).

    x: planar buffer; the conv reads ``c_in`` channels starting at plane ``x_plane0``.
    w_packed: ``pack_conv_weight`` output, shape [taps, c_in/8, c_out_pad, 8].
    out: planar buffer written at plane ``out_plane0`` (allocated when None); with ``out_fp32`` the
    result is fp32 (B, c_out, D, H, W) instead.
    chan_add: fp32 [B, c_out] or [steps, B, c_out] (then ``step_ptr`` selects the row block on device).
    stats: double [B, Cs, 2], accumulated at channel ``stats_c0``.

    fp32 planar ``x`` (TF32 mode, ``vdm_conv3d_tf32``): ``w_packed``, a planar ``out`` and ``residual`` are fp32 planar
    too (plane windows count 4-channel planes); ``skip_x``, ``in_norm`` and ``residual_upsample`` raise
    ``UnsupportedFusion``.
    """
    lanes = _planar_lanes(x, "conv3d x")
    tf32 = lanes == 4
    b, xp, d, h, w_, _ = x.shape
    if circular:                       # x carries a one-voxel periodic halo (``pad_circular``)
        d, h, w_ = d - 2, h - 2, w_ - 2
    n_taps, cin_pl, c_out_pad, w_lanes = w_packed.shape
    _need(w_packed.is_cuda and _LANES.get(w_packed.dtype) == lanes and w_packed.is_contiguous() and w_lanes == lanes,
          "conv3d: w_packed must be a contiguous CUDA bf16 [taps, Cin/8, Cout_pad, 8] tensor (fp32 [taps, Cin/4, Cout_pad, 4] "
          "with an fp32 x)")
    c_in = cin_pl * lanes if c_in is None else c_in
    _need(c_in == cin_pl * lanes, f"conv3d: weight packs {cin_pl * lanes} input channels, c_in={c_in}")
    _need(n_taps == len(taps), f"conv3d: weight has {n_taps} taps, {len(taps)} offsets given")
    desc = _C.ConvDesc()
    desc.batch, desc.depth, desc.height, desc.width = b, d, h, w_
    desc.c_in, desc.c_out, desc.c_out_pad, desc.n_taps = c_in, c_out, c_out_pad, n_taps
    for i, t in enumerate(taps):
        for k in range(3):
            desc.tap_offset[i][k] = t[k]
    desc.circular = 1 if circular else 0
    desc.out_fp32 = 1 if out_fp32 else 0
    desc.x_planes, desc.x_plane0 = xp, x_plane0
    if out is None:
        if out_fp32:
            out = torch.empty((b, c_out, d, h, w_), dtype=torch.float32, device=x.device)
        else:
            out = torch.empty((b, c_out // lanes, d, h, w_, lanes), dtype=x.dtype, device=x.device)
    if out_fp32:
        _need(out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (b, c_out, d, h, w_),
              "conv3d: fp32 output must be contiguous (B, c_out, D, H, W)")
    else:
        _same_lanes(lanes, out, "conv3d out")
        _need(tuple(out.shape[2:5]) == (d, h, w_) and out.shape[0] == b, "conv3d: out grid mismatch")
        desc.y_planes, desc.y_plane0 = out.shape[1], out_plane0
    epi = _C.ConvEpilogue()
    if chan_add is not None:
        _need(chan_add.is_cuda and chan_add.dtype == torch.float32 and chan_add.is_contiguous() and
              chan_add.shape[-1] == c_out and chan_add.shape[-2] == b, "conv3d: chan_add must be fp32 [..., B, c_out]")
        epi.chan_add = chan_add.data_ptr()
        epi.chan_add_step_stride = b * c_out
        if step_ptr is not None:
            _need(step_ptr.is_cuda and step_ptr.dtype == torch.int32, "conv3d: step_ptr must be a CUDA int32 tensor")
            epi.step_ptr = step_ptr.data_ptr()
    if residual is not None:
        _same_lanes(lanes, residual, "conv3d residual")
        r_grid = (d // 2, h // 2, w_ // 2) if residual_upsample else (d, h, w_)
        _need(tuple(residual.shape[2:5]) == r_grid and residual.shape[0] == b, "conv3d: residual grid mismatch")
        epi.residual = residual.data_ptr()
        # residual_upsample="d2s": eight parity blocks of c_out channels on the half-resolution grid (see polyphase_upconv)
        epi.residual_upsample = 2 if residual_upsample == "d2s" else (1 if residual_upsample else 0)
        if residual_upsample == "d2s":
            _need(c_out % 8 == 0 and residual.shape[1] >= residual_plane0 + c_out, "conv3d: a depth-to-space residual holds 8 x c_out channels")
        desc.r_planes, desc.r_plane0 = residual.shape[1], residual_plane0
    if skip_x is not None:
        _same_lanes(lanes, skip_x, "conv3d skip_x")
        _need(tuple(skip_x.shape[2:5]) == (d, h, w_) and skip_x.shape[0] == b, "conv3d: skip_x grid mismatch")
        _need(skip_w is not None and skip_w.is_cuda and skip_w.dtype == torch.bfloat16 and skip_w.is_contiguous() and
              skip_w.dim() == 4 and skip_w.shape[0] == 1 and skip_w.shape[2] == c_out_pad,
              "conv3d: skip_w must be the packed (c_out, skip_c_in, 1, 1, 1) filter")
        epi.skip_x, epi.skip_w = skip_x.data_ptr(), skip_w.data_ptr()
        epi.skip_c_in, epi.skip_planes, epi.skip_plane0 = skip_w.shape[1] * 8, skip_x.shape[1], skip_plane0
    if in_norm is not None:
        _need(in_norm.is_cuda and in_norm.dtype == torch.float32 and in_norm.is_contiguous() and
              tuple(in_norm.shape) == (b, c_in, 2), "conv3d: in_norm must be contiguous CUDA fp32 [B, c_in, 2]")
        epi.in_norm = in_norm.data_ptr()
    if stats is not None:
        _need(stats.is_cuda and stats.dtype == torch.float64 and stats.is_contiguous() and stats.dim() == 3 and
              stats.shape[0] == b and stats.shape[2] == 2, "conv3d: stats must be double [B, C, 2]")
        epi.stats = stats.data_ptr()
        epi.stats_channels = stats.shape[1]
        epi.stats_c0 = stats_c0
    prof = _CONV_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    fn = _C.lib().vdm_conv3d_tf32 if tf32 else _C.lib().vdm_conv3d
    rc = fn(ctypes.byref(desc), x.data_ptr(), w_packed.data_ptr(), out.data_ptr(), ctypes.byref(epi), _stream())
    if rc == _C.E_UNSUPPORTED and (skip_x is not None or in_norm is not None or (tf32 and residual_upsample)):
        raise _C.UnsupportedFusion(_C.lib().vdm_last_error_string().decode("utf-8", "replace"))
    _C.check(rc, "vdm_conv3d_tf32" if tf32 else "vdm_conv3d")
    _launched(1)
    if prof is not None:
        e1.record()
        # algorithmic FLOPs: real (un-padded) output channels, the channels the caller says it reads
        prof.append((e0, e1, 2.0 * n_taps * c_in * c_out * b * d * h * w_,
                     f"{_PROFILE_TAG}{'tf32 ' if tf32 else ''}{c_in}->{c_out} taps={n_taps} grid={d}x{h}x{w_} B={b}"))
    return out


# ---- polyphase form of conv3x3x3(interpolate(a, scale_factor=2, mode="nearest")) ------------------------------
# Fine voxel 2i + p (per axis, parity p in {0, 1}) reads the up-sampled input at 2i + p + t, t in {-1, 0, 1}, i.e. the COARSE
# voxel i + floor((p + t) / 2):   p = 0: t = -1 -> i - 1, t = 0, +1 -> i;      p = 1: t = -1, 0 -> i, t = +1 -> i + 1.
# Per output parity the 27 taps therefore collapse to 2 x 2 x 2 taps on the coarse grid whose weights are sums of the
# original ones: 8 / 27 of the multiply-adds, and the up-sampled tensor (8x the coarse one) is never materialised.
# Zero padding carries over exactly: fine index -1 / 2n is coarse index -1 / n.
_POLY_SETS = {0: ((-1, (0,)), (0, (1, 2))), 1: ((0, (0, 1)), (1, (2,)))}      # parity -> ((coarse offset, filter taps), ...)


def polyphase_taps(parity: Tuple[int, int, int]):
    """Coarse-grid tap offsets (8 triples in {-1, 0, 1}) of output parity (pd, ph, pw), in the order of
    ``polyphase_weight``'s taps."""
    return tuple((od, oh, ow) for od, _ in _POLY_SETS[parity[0]] for oh, _ in _POLY_SETS[parity[1]]
                 for ow, _ in _POLY_SETS[parity[2]])


def polyphase_weight(w: torch.Tensor, parity: Tuple[int, int, int]) -> torch.Tensor:
    """(c_out, c_in, 3, 3, 3) -> (c_out, c_in, 2, 2, 2): the effective filter of output parity (pd, ph, pw), fp32."""
    out = []
    for _, kd in _POLY_SETS[parity[0]]:
        for _, kh in _POLY_SETS[parity[1]]:
            for _, kw in _POLY_SETS[parity[2]]:
                out.append(w[:, :, list(kd)][:, :, :, list(kh)][:, :, :, :, list(kw)].sum(dim=(2, 3, 4)))
    return torch.stack(out, dim=2).reshape(w.shape[0], w.shape[1], 2, 2, 2).contiguous()


def polyphase_group(w: torch.Tensor, group: int, n_par: int):
    """Several output parities in ONE conv launch: the ``n_par`` (2, 4 or 8) parities that share the leading parity bits
    ``group`` (n_par = 4: group = pd; n_par = 2: group = pd * 2 + ph) are stacked along the output channels, block
    ``j`` = parity ``group * n_par + j``, over the union of their coarse taps; a (tap, block) pair the parity does not use
    holds zeros.  The parities of a group share the halo tile, so the coarse tensor is read once per group instead of
    once per parity, and N = n_par * c_out keeps the tensor cores busy where a single parity (N = c_out) is bound by
    the latency of its tile loads (profiles/R2k_poly_tiles.txt).
    Returns (weight fp32 (n_par * c_out, c_in, Td, Th, Tw), taps as a tuple of coarse offsets in the weight's tap order)."""
    co, ci = w.shape[0], w.shape[1]
    if n_par == 1:
        parity = (group >> 2, (group >> 1) & 1, group & 1)
        return polyphase_weight(w.float(), parity), polyphase_taps(parity)
    n_fixed = {8: 0, 4: 1, 2: 2}[n_par]
    fixed = [(group >> (n_fixed - 1 - i)) & 1 for i in range(n_fixed)]
    offs = [[p - 1, p] for p in fixed] + [[-1, 0, 1]] * (3 - n_fixed)
    taps = tuple((od, oh, ow) for od in offs[0] for oh in offs[1] for ow in offs[2])
    out = w.new_zeros((n_par * co, ci, len(offs[0]), len(offs[1]), len(offs[2])), dtype=torch.float32)
    for j in range(n_par):
        pi = group * n_par + j
        parity = (pi >> 2, (pi >> 1) & 1, pi & 1)
        sets = [dict(_POLY_SETS[p]) for p in parity]
        for a, od in enumerate(offs[0]):
            for b_, oh in enumerate(offs[1]):
                for c, ow in enumerate(offs[2]):
                    if od in sets[0] and oh in sets[1] and ow in sets[2]:
                        kd, kh, kw = list(sets[0][od]), list(sets[1][oh]), list(sets[2][ow])
                        out[j * co:(j + 1) * co, :, a, b_, c] = \
                            w[:, :, kd][:, :, :, kh][:, :, :, :, kw].float().sum(dim=(2, 3, 4))
    return out, taps


# ---- elementwise ---------------------------------------------------------------------------------
def channel_stats(x: torch.Tensor, channels: int, x_plane0: int = 0, stats: Optional[torch.Tensor] = None,
                  stats_c0: int = 0) -> torch.Tensor:
    _planar_ok(x, "channel_stats x")
    b = x.shape[0]
    voxels = x.shape[2] * x.shape[3] * x.shape[4]
    if stats is None:
        stats = torch.zeros((b, channels, 2), dtype=torch.float64, device=x.device)
    v = _view(x, x_plane0)
    rc = _C.lib().vdm_channel_stats(ctypes.byref(v), b, voxels, channels, stats.data_ptr(), stats.shape[1], stats_c0,
                                    _stream())
    _C.check(rc, "vdm_channel_stats")
    _launched(1)
    return stats


def gn_silu(x: torch.Tensor, channels: int, groups: int, stats: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor,
            eps: float = 1e-5, *, x_plane0: int = 0, out: Optional[torch.Tensor] = None, out_plane0: int = 0,
            dropout_p: float = 0.0, seed: int = 0, layer_tag: int = 0, seed_step: Optional[torch.Tensor] = None) -> torch.Tensor:
    """y = dropout(silu(groupnorm(x))).  ``seed_step`` (device int32) is added to ``seed`` on the device.
    fp32 planar tensors (TF32 mode): ``vdm_gn_silu_f32``, no dropout."""
    lanes = _planar_lanes(x, "gn_silu x")
    b = x.shape[0]
    voxels = x.shape[2] * x.shape[3] * x.shape[4]
    _need(stats.dtype == torch.float64 and tuple(stats.shape) == (b, channels, 2) and stats.is_contiguous(),
          "gn_silu: stats must be double [B, channels, 2]")
    _need(gamma.dtype == torch.float32 and beta.dtype == torch.float32 and gamma.numel() == channels and
          beta.numel() == channels and gamma.is_cuda and beta.is_cuda, "gn_silu: gamma/beta must be CUDA fp32 [channels]")
    if out is None:
        out = torch.empty((b, channels // lanes) + tuple(x.shape[2:5]) + (lanes,), dtype=x.dtype, device=x.device)
    _same_lanes(lanes, out, "gn_silu out")
    vx, vy = _view(x, x_plane0), _view(out, out_plane0)
    if lanes == 4:
        _need(dropout_p == 0.0, "gn_silu: the fp32 (TF32 inference) form has no dropout")
        rc = _C.lib().vdm_gn_silu_f32(ctypes.byref(vx), ctypes.byref(vy), b, voxels, channels, groups, stats.data_ptr(),
                                      gamma.data_ptr(), beta.data_ptr(), eps, _stream())
        _C.check(rc, "vdm_gn_silu_f32")
        _launched(1)
        return out
    rc = _C.lib().vdm_gn_silu_step(ctypes.byref(vx), ctypes.byref(vy), b, voxels, channels, groups, stats.data_ptr(),
                                   gamma.data_ptr(), beta.data_ptr(), eps, dropout_p, seed, _ptr(seed_step), layer_tag,
                                   _stream())
    _C.check(rc, "vdm_gn_silu")
    _launched(1)
    return out


def gn_coef(stats: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int, voxels: int, eps: float = 1e-5,
            out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``vdm_gn_coef``: fp32 [B, C, 2] pairs (a, b) with silu(groupnorm(x)) = h + h tanh(h), h = a x + b, from the fp64
    (sum, sumsq) table of the tensor -- the ``in_norm`` argument of ``conv3d`` (GroupNorm + SiLU applied by the conv
    kernel to its input tile instead of by a separate pass)."""
    _need(stats.is_cuda and stats.dtype == torch.float64 and stats.is_contiguous() and stats.dim() == 3 and stats.shape[2] == 2,
          "gn_coef: stats must be a contiguous CUDA double [B, C, 2]")
    b, c, _ = stats.shape
    _need(gamma.dtype == torch.float32 and beta.dtype == torch.float32 and gamma.numel() == c and beta.numel() == c and
          gamma.is_cuda and beta.is_cuda, "gn_coef: gamma/beta must be CUDA fp32 [C]")
    if out is None:
        out = torch.empty((b, c, 2), dtype=torch.float32, device=stats.device)
    _need(out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (b, c, 2),
          "gn_coef: out must be contiguous CUDA fp32 [B, C, 2]")
    rc = _C.lib().vdm_gn_coef(stats.data_ptr(), b, c, groups, voxels, gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(),
                              _stream())
    _C.check(rc, "vdm_gn_coef")
    _launched(1)
    return out


def gn_silu_view(x: torch.Tensor, channels: int, c_off: int, channels_total: int, groups: int, stats: torch.Tensor,
                 gamma: torch.Tensor, beta: torch.Tensor, eps: float, out: torch.Tensor, *, x_plane0: int = 0,
                 out_plane0: int = 0, upsample=False) -> torch.Tensor:
    """silu(groupnorm(.)) of channels [c_off, c_off + channels) of a ``channels_total``-channel norm, written to a plane
    window of ``out``; with ``upsample`` x is at half the resolution of ``out`` (``vdm_gn_silu_view``)."""
    _planar_ok(x, "gn_silu_view x")
    _planar_ok(out, "gn_silu_view out")
    b, _, d, h, w, _ = out.shape
    if upsample == "coarse":         # x and out on the half grid of the (2d, 2h, 2w) concat the statistics refer to
        _need(tuple(x.shape[2:5]) == (d, h, w) and x.shape[0] == b, "gn_silu_view: x grid does not match out")
        d, h, w = 2 * d, 2 * h, 2 * w
    else:
        _need(tuple(x.shape[2:5]) == ((d // 2, h // 2, w // 2) if upsample else (d, h, w)) and x.shape[0] == b,
              "gn_silu_view: x grid does not match out")
    _need(stats.dtype == torch.float64 and tuple(stats.shape) == (b, channels_total, 2) and stats.is_contiguous(),
          "gn_silu_view: stats must be double [B, channels_total, 2]")
    _need(gamma.dtype == torch.float32 and beta.dtype == torch.float32 and gamma.numel() == channels_total and
          beta.numel() == channels_total and gamma.is_cuda and beta.is_cuda,
          "gn_silu_view: gamma/beta must be CUDA fp32 [channels_total]")
    vx, vy = _view(x, x_plane0), _view(out, out_plane0)
    rc = _C.lib().vdm_gn_silu_view(ctypes.byref(vx), ctypes.byref(vy), b, d, h, w, channels, c_off, channels_total, groups,
                                   stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), eps,
                                   2 if upsample == "coarse" else (1 if upsample else 0), _stream())
    _C.check(rc, "vdm_gn_silu_view")
    _launched(1)
    return out


def avgpool2(x: torch.Tensor, channels: int, *, x_plane0: int = 0, out: Optional[torch.Tensor] = None,
             out_plane0: int = 0, stats: Optional[torch.Tensor] = None, stats_c0: int = 0) -> torch.Tensor:
    lanes = _planar_lanes(x, "avgpool2 x")
    b, _, d, h, w, _ = x.shape
    if out is None:
        out = torch.empty((b, channels // lanes, d // 2, h // 2, w // 2, lanes), dtype=x.dtype, device=x.device)
    _same_lanes(lanes, out, "avgpool2 out")
    vx, vy = _view(x, x_plane0), _view(out, out_plane0)
    fn = _C.lib().vdm_avgpool2_f32 if lanes == 4 else _C.lib().vdm_avgpool2
    rc = fn(ctypes.byref(vx), ctypes.byref(vy), b, d, h, w, channels, _ptr(stats), 0 if stats is None else stats.shape[1],
            stats_c0, _stream())
    _C.check(rc, "vdm_avgpool2_f32" if lanes == 4 else "vdm_avgpool2")
    _launched(1)
    return out


def upsample2(coarse: torch.Tensor, channels: int, out: torch.Tensor, *, coarse_plane0: int = 0, out_plane0: int = 0,
              stats: Optional[torch.Tensor] = None, stats_c0: int = 0) -> torch.Tensor:
    lanes = _planar_lanes(coarse, "upsample2 coarse")
    _same_lanes(lanes, out, "upsample2 out")
    b, _, d, h, w, _ = out.shape
    _need(tuple(coarse.shape[2:5]) == (d // 2, h // 2, w // 2), "upsample2: coarse grid must be half the fine grid")
    vx, vy = _view(coarse, coarse_plane0), _view(out, out_plane0)
    fn = _C.lib().vdm_upsample2_f32 if lanes == 4 else _C.lib().vdm_upsample2
    rc = fn(ctypes.byref(vx), ctypes.byref(vy), b, d, h, w, channels, _ptr(stats), 0 if stats is None else stats.shape[1],
            stats_c0, _stream())
    _C.check(rc, "vdm_upsample2_f32" if lanes == 4 else "vdm_upsample2")
    _launched(1)
    return out


def pad_circular(x: torch.Tensor, channels: int, *, x_plane0: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``vdm_pad_circular``: planar [B, P, D, H, W, L] -> [B, channels/L, D+2, H+2, W+2, L] with a periodic one-voxel halo
    (L = 8 bf16 or 4 fp32 channels per plane; the kernel copies 16-byte units)."""
    lanes = _planar_lanes(x, "pad_circular x")
    b, _, d, h, w, _ = x.shape
    if out is None:
        out = torch.empty((b, channels // lanes, d + 2, h + 2, w + 2, lanes), dtype=x.dtype, device=x.device)
    _same_lanes(lanes, out, "pad_circular out")
    _need(tuple(out.shape[2:5]) == (d + 2, h + 2, w + 2) and out.shape[0] == b, "pad_circular: out must have the padded grid")
    _need(channels % lanes == 0, f"pad_circular: channels={channels} is not a whole number of planes")
    vx, vy = _view(x, x_plane0), _view(out, 0)
    # the C entry point counts 8 channels per 16-byte plane
    rc = _C.lib().vdm_pad_circular(ctypes.byref(vx), ctypes.byref(vy), b, d, h, w, channels * 8 // lanes, _stream())
    _C.check(rc, "vdm_pad_circular")
    _launched(1)
    return out


def pack_input(z: torch.Tensor, cond: Optional[torch.Tensor], c_pad: int = 16,
               out: Optional[torch.Tensor] = None, dtype: torch.dtype = torch.bfloat16) -> torch.Tensor:
    """z: fp32 (B, 1, D, H, W) or (B, D, H, W); cond: fp32 (B, n_cond, D, H, W) -> planar [B, c_pad/8, D, H, W, 8], or
    fp32 planar [B, c_pad/4, D, H, W, 4] when ``out`` (or, without ``out``, ``dtype``) is fp32."""
    _need(z.is_cuda and z.dtype == torch.float32 and z.is_contiguous(), "pack_input: z must be contiguous CUDA fp32")
    if z.dim() == 5:
        _need(z.shape[1] == 1, "pack_input: z must have one channel")
        b, _, d, h, w = z.shape
    else:
        b, d, h, w = z.shape
    n_cond = 0
    if cond is not None:
        _need(cond.is_cuda and cond.dtype == torch.float32 and cond.is_contiguous() and cond.dim() == 5 and
              tuple(cond.shape[2:]) == (d, h, w) and cond.shape[0] == b, "pack_input: cond must be fp32 (B, n, D, H, W)")
        n_cond = cond.shape[1]
    if out is None:
        lanes = _LANES[dtype]
        out = torch.empty((b, c_pad // lanes, d, h, w, lanes), dtype=dtype, device=z.device)
    lanes = _planar_lanes(out, "pack_input out")
    vo = _view(out, 0)
    fn = _C.lib().vdm_pack_input_f32 if lanes == 4 else _C.lib().vdm_pack_input
    rc = fn(z.data_ptr(), _ptr(cond), ctypes.byref(vo), b, d * h * w, n_cond, c_pad, _stream())
    _C.check(rc, "vdm_pack_input_f32" if lanes == 4 else "vdm_pack_input")
    _launched(1)
    return out


# ---- backward (training) ---------------------------------------------------------------------------
def conv3d_wgrad(a: torch.Tensor, g: torch.Tensor, c_in: int, c_out: int, kernel: int = 3, *, a_plane0: int = 0,
                 g_plane0: int = 0, out: Optional[torch.Tensor] = None, grad_out: Optional[torch.Tensor] = None,
                 a_padded: bool = False, g_padded: bool = False) -> torch.Tensor:
    """``vdm_conv3d_wgrad``: dw[tap, ci, co] += sum_v a[ci, v + tap] g[co, v]  (fp32 [k^3, c_in, c_out]).

    a, g: planar buffers on the same grid; the g window must hold c_out rounded up to 16 channels.
    ``out`` is accumulated into (allocated and zeroed when None)."""
    _planar_ok(a, "conv3d_wgrad a")
    _planar_ok(g, "conv3d_wgrad g")
    b, ap, d, h, w_, _ = a.shape
    if a_padded:                       # a carries a one-voxel periodic halo (circular convs)
        d, h, w_ = d - 2, h - 2, w_ - 2
    gd = tuple(int(v) - (2 if g_padded else 0) for v in g.shape[2:5])
    _need(gd == (d, h, w_) and g.shape[0] == b, "conv3d_wgrad: a / g grid mismatch")
    desc = _C.WgradDesc()
    if grad_out is not None:
        # accumulate straight into a torch-layout gradient (c_out, c_in_real, k, k, k), e.g. a view of the flat bucket
        _need(grad_out.is_cuda and grad_out.dtype == torch.float32 and grad_out.is_contiguous() and grad_out.dim() == 5 and
              grad_out.shape[0] == c_out and grad_out.shape[1] <= c_in and tuple(grad_out.shape[2:]) == (kernel,) * 3,
              "conv3d_wgrad: grad_out must be contiguous fp32 (c_out, c_in_real <= c_in, k, k, k)")
        desc.dw_stride_tap, desc.dw_stride_ci, desc.dw_stride_co = 1, kernel ** 3, grad_out.shape[1] * kernel ** 3
        desc.c_in_real = grad_out.shape[1]
        out = grad_out
    else:
        if out is None:
            out = torch.zeros((kernel ** 3, c_in, c_out), dtype=torch.float32, device=a.device)
        _need(out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and
              tuple(out.shape) == (kernel ** 3, c_in, c_out), "conv3d_wgrad: out must be fp32 [k^3, c_in, c_out]")
    desc.batch, desc.depth, desc.height, desc.width = b, d, h, w_
    desc.c_in, desc.c_out, desc.kernel = c_in, c_out, kernel
    desc.a_planes, desc.a_plane0 = ap, a_plane0
    desc.g_planes, desc.g_plane0 = g.shape[1], g_plane0
    desc.a_padded = 1 if a_padded else 0
    desc.g_padded = 1 if g_padded else 0
    prof = _CONV_PROFILE
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    rc = _C.lib().vdm_conv3d_wgrad(ctypes.byref(desc), a.data_ptr(), g.data_ptr(), out.data_ptr(), _stream())
    _C.check(rc, "vdm_conv3d_wgrad")
    _launched(1)
    if prof is not None:
        e1.record()
        prof.append((e0, e1, 2.0 * kernel ** 3 * c_in * c_out * b * d * h * w_,
                     f"wgrad {c_in}->{c_out} taps={kernel ** 3} grid={d}x{h}x{w_} B={b}"))
    return out


def wgrad_to_torch(dw: torch.Tensor, kernel: int) -> torch.Tensor:
    """fp32 [k^3, c_in, c_out] -> torch Conv3d weight layout (c_out, c_in, k, k, k)."""
    k3, ci, co = dw.shape
    return dw.reshape(kernel, kernel, kernel, ci, co).permute(4, 3, 0, 1, 2).contiguous()


def _gn_common(x, channels, stats, gamma, beta, who):
    _planar_ok(x, f"{who} x")
    b = x.shape[0]
    _need(stats.dtype == torch.float64 and tuple(stats.shape) == (b, channels, 2) and stats.is_contiguous(),
          f"{who}: stats must be double [B, channels, 2]")
    _need(gamma.dtype == torch.float32 and beta.dtype == torch.float32 and gamma.numel() == channels and
          beta.numel() == channels and gamma.is_cuda and beta.is_cuda, f"{who}: gamma/beta must be CUDA fp32 [channels]")
    return b, x.shape[2] * x.shape[3] * x.shape[4]


def gn_silu_bwd(x: torch.Tensor, dy: torch.Tensor, channels: int, groups: int, stats: torch.Tensor, gamma: torch.Tensor,
                beta: torch.Tensor, eps: float = 1e-5, *, x_plane0: int = 0, dy_plane0: int = 0,
                add: Optional[torch.Tensor] = None, add_plane0: int = 0, out: Optional[torch.Tensor] = None,
                out_plane0: int = 0, dropout_p: float = 0.0, seed: int = 0, layer_tag: int = 0,
                out_stats: Optional[torch.Tensor] = None, out_stats_c0: int = 0, sums: Optional[torch.Tensor] = None,
                sums_c0: int = 0, seed_step: Optional[torch.Tensor] = None):
    """Backward of ``gn_silu``: returns (dx, sums) with sums double [B, channels, 2] = per-sample
    (sum du, sum du*xhat), i.e. dbeta = sums[..., 0].sum(0), dgamma = sums[..., 1].sum(0).
    dx = GroupNorm/SiLU/dropout backward of dy [+ add]; ``out_stats`` accumulates (sum, sumsq) of dx."""
    b, voxels = _gn_common(x, channels, stats, gamma, beta, "gn_silu_bwd")
    _planar_ok(dy, "gn_silu_bwd dy")
    if out is None:
        out = torch.empty((b, channels // 8) + tuple(x.shape[2:]), dtype=torch.bfloat16, device=x.device)
    _planar_ok(out, "gn_silu_bwd out")
    if sums is None:
        sums = torch.zeros((b, channels, 2), dtype=torch.float64, device=x.device)
    _need(sums.dtype == torch.float64 and sums.is_contiguous() and sums.dim() == 3 and sums.shape[0] == b and
          sums.shape[2] == 2 and sums_c0 + channels <= sums.shape[1], "gn_silu_bwd: sums must be a zeroed double [B, >= channels, 2]")
    vx, vg, vo = _view(x, x_plane0), _view(dy, dy_plane0), _view(out, out_plane0)
    lib = _C.lib()
    rc = lib.vdm_gn_silu_bwd_reduce(ctypes.byref(vx), ctypes.byref(vg), b, voxels, channels, groups, stats.data_ptr(),
                                    gamma.data_ptr(), beta.data_ptr(), eps, dropout_p, seed, _ptr(seed_step), layer_tag,
                                    sums.data_ptr(), sums.shape[1], sums_c0, _stream())
    _C.check(rc, "vdm_gn_silu_bwd_reduce")
    va = None
    if add is not None:
        _planar_ok(add, "gn_silu_bwd add")
        va = ctypes.byref(_view(add, add_plane0))
    rc = lib.vdm_gn_silu_bwd_apply(ctypes.byref(vx), ctypes.byref(vg), va, ctypes.byref(vo), b, voxels, channels, groups,
                                   stats.data_ptr(), gamma.data_ptr(), beta.data_ptr(), eps, dropout_p, seed, _ptr(seed_step),
                                   layer_tag, sums.data_ptr(), sums.shape[1], sums_c0, _ptr(out_stats),
                                   0 if out_stats is None else out_stats.shape[1], out_stats_c0, _stream())
    _C.check(rc, "vdm_gn_silu_bwd_apply")
    _launched(2)
    return out, sums


def avgpool2_bwd(dy: torch.Tensor, channels: int, dx: torch.Tensor, *, dy_plane0: int = 0, dx_plane0: int = 0,
                 accumulate: bool = False, stats: Optional[torch.Tensor] = None, stats_c0: int = 0) -> torch.Tensor:
    """dx[window] = (dx[window] if accumulate else 0) + upsample(dy)/8; dx is on the fine grid."""
    _planar_ok(dy, "avgpool2_bwd dy")
    _planar_ok(dx, "avgpool2_bwd dx")
    b, _, d, h, w, _ = dx.shape
    _need(tuple(dy.shape[2:5]) == (d // 2, h // 2, w // 2), "avgpool2_bwd: dy grid must be half the dx grid")
    vg, vx = _view(dy, dy_plane0), _view(dx, dx_plane0)
    rc = _C.lib().vdm_avgpool2_bwd(ctypes.byref(vg), ctypes.byref(vx), b, d, h, w, channels, 1 if accumulate else 0,
                                   _ptr(stats), 0 if stats is None else stats.shape[1], stats_c0, _stream())
    _C.check(rc, "vdm_avgpool2_bwd")
    _launched(1)
    return dx


def upsample2_bwd(dy: torch.Tensor, channels: int, *, dy_plane0: int = 0, out: Optional[torch.Tensor] = None,
                  out_plane0: int = 0, stats: Optional[torch.Tensor] = None, stats_c0: int = 0) -> torch.Tensor:
    """dcoarse = sum over each 2x2x2 block of the fine gradient window dy."""
    _planar_ok(dy, "upsample2_bwd dy")
    b, _, d, h, w, _ = dy.shape
    if out is None:
        out = torch.empty((b, channels // 8, d // 2, h // 2, w // 2, 8), dtype=torch.bfloat16, device=dy.device)
    _planar_ok(out, "upsample2_bwd out")
    vg, vo = _view(dy, dy_plane0), _view(out, out_plane0)
    rc = _C.lib().vdm_upsample2_bwd(ctypes.byref(vg), ctypes.byref(vo), b, d, h, w, channels, _ptr(stats),
                                    0 if stats is None else stats.shape[1], stats_c0, _stream())
    _C.check(rc, "vdm_upsample2_bwd")
    _launched(1)
    return out


def augment_crop(raw: torch.Tensor, crop, anchor, flip, perm, *, alpha: float = 0.0, mean: float = 0.0, std: float = 1.0,
                 do_log: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``vdm_augment_crop``: periodic crop (start ``anchor``, extent ``crop``) of a raw fp32 box (S0, S1, S2), optional
    ``(log10(x + alpha) - mean) / std``, flip of the cropped axes in ``flip`` and ``permute`` by ``perm`` in one pass."""
    _need(raw.is_cuda and raw.dtype == torch.float32 and raw.is_contiguous() and raw.dim() == 3, "augment_crop: raw must be contiguous CUDA fp32 (S0, S1, S2)")
    crop, anchor, flip, perm = [int(v) for v in crop], [int(v) for v in anchor], [int(bool(v)) for v in flip], [int(v) for v in perm]
    n = tuple(crop[perm[d]] for d in range(3))
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=raw.device)
    _need(out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape[-3:]) == n and out.numel() == n[0] * n[1] * n[2],
          "augment_crop: out must be contiguous CUDA fp32 with the permuted crop shape")
    arr = lambda v: (ctypes.c_int32 * 3)(*v)
    rc = _C.lib().vdm_augment_crop(raw.data_ptr(), out.data_ptr(), arr(raw.shape), arr(crop), arr(anchor), arr(flip), arr(perm),
                                   alpha, mean, std, 1 if do_log else 0, _stream())
    _C.check(rc, "vdm_augment_crop")
    _launched(1)
    return out


def log_histogram(fields: torch.Tensor, lo: float, hi: float, nbins: int, add: float = 1.0) -> torch.Tensor:
    """``vdm_log_histogram``: per-field histogram of log10(field + add) on ``nbins`` equal bins of [lo, hi]
    (numpy.histogram semantics).  fields: CUDA fp32 (F, ...) -> int64 (F, nbins)."""
    _need(fields.is_cuda and fields.dtype == torch.float32 and fields.is_contiguous() and fields.dim() >= 2,
          "log_histogram: fields must be contiguous CUDA fp32 (F, ...)")
    f = fields.shape[0]
    counts = torch.zeros((f, nbins), dtype=torch.int64, device=fields.device)
    rc = _C.lib().vdm_log_histogram(fields.data_ptr(), f, fields.numel() // f, add, lo, hi, nbins, counts.data_ptr(), _stream())
    _C.check(rc, "vdm_log_histogram")
    _launched(1)
    return counts


def sumsq(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out (double scalar tensor, accumulated) += sum(x^2) over a flat fp32 buffer."""
    _need(x.is_cuda and x.dtype == torch.float32 and x.is_contiguous(), "sumsq: x must be contiguous CUDA fp32")
    if out is None:
        out = torch.zeros(1, dtype=torch.float64, device=x.device)
    _C.check(_C.lib().vdm_sumsq(x.data_ptr(), x.numel(), out.data_ptr(), _stream()), "vdm_sumsq")
    _launched(1)
    return out


def adamw_step(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, *, lr: float,
               step: int, beta1: float = 0.9, beta2: float = 0.999, eps: float = 1e-8, weight_decay: float = 0.01,
               grad_sumsq: Optional[torch.Tensor] = None, max_norm: float = 0.0, grad_scale: float = 1.0,
               step_ptr: Optional[torch.Tensor] = None) -> None:
    """``vdm_adamw_step`` on flat fp32 buckets (in place); the step number is ``step + *step_ptr`` when a device
    counter is given (CUDA-graph replay)."""
    for t in (param, grad, exp_avg, exp_avg_sq):
        _need(t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.numel() == param.numel(),
              "adamw_step: buckets must be contiguous CUDA fp32 of equal length")
    rc = _C.lib().vdm_adamw_step_dev(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                     param.numel(), lr, beta1, beta2, eps, weight_decay, step, _ptr(step_ptr),
                                     _ptr(grad_sumsq), max_norm, grad_scale, _stream())
    _C.check(rc, "vdm_adamw_step")
    _launched(1)


# ---- sampler ---------------------------------------------------------------------------------------
def sampler_step(z: torch.Tensor, eps_hat: torch.Tensor, coef: torch.Tensor, *, out: Optional[torch.Tensor] = None,
                 step_ptr: Optional[torch.Tensor] = None, seed: int = 0, realisation_id: Optional[torch.Tensor] = None,
                 draw_base: int = 1, noise: Optional[torch.Tensor] = None, cond: Optional[torch.Tensor] = None,
                 packed_out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``vdm_sampler_step``: z_out = out_scale * (w_z z + w_eps eps_hat + noise_scale N(0,1)).

    coef: fp32 [steps, 4] = (w_z, w_eps, noise_scale, out_scale); ``step_ptr`` (device int32) picks the row.
    """
    _need(z.is_cuda and z.dtype == torch.float32 and z.is_contiguous(), "sampler_step: z must be contiguous CUDA fp32")
    _need(eps_hat.dtype == torch.float32 and eps_hat.is_contiguous() and eps_hat.numel() == z.numel(),
          "sampler_step: eps_hat must be fp32 with z's shape")
    _need(coef.is_cuda and coef.dtype == torch.float32 and coef.is_contiguous() and coef.shape[-1] == 4,
          "sampler_step: coef must be fp32 [steps, 4]")
    b = z.shape[0]
    voxels = z.numel() // b
    if out is None:
        out = torch.empty_like(z)
    n_cond = 0 if cond is None else cond.shape[1]
    packed_planes = 0 if packed_out is None else packed_out.shape[1]
    if noise is not None:
        _need(noise.dtype == torch.float32 and noise.is_contiguous() and noise.numel() == z.numel(),
              "sampler_step: injected noise must be fp32 with z's shape")
    rc = _C.lib().vdm_sampler_step(z.data_ptr(), eps_hat.data_ptr(), out.data_ptr(), b, voxels, coef.data_ptr(),
                                   _ptr(step_ptr), seed, _ptr(realisation_id), draw_base, _ptr(noise), _ptr(cond),
                                   n_cond, _ptr(packed_out), packed_planes, _stream())
    _C.check(rc, "vdm_sampler_step")
    _launched(1)
    return out


def philox_normal(shape, seed: int, draw: int, realisation_id: Optional[torch.Tensor] = None,
                  device="cuda") -> torch.Tensor:
    out = torch.empty(shape, dtype=torch.float32, device=device)
    b = shape[0]
    rc = _C.lib().vdm_philox_normal(out.data_ptr(), b, out.numel() // b, seed, _ptr(realisation_id), draw, _stream())
    _C.check(rc, "vdm_philox_normal")
    _launched(1)
    return out


def increment(counter: torch.Tensor) -> None:
    _C.check(_C.lib().vdm_increment(counter.data_ptr(), _stream()), "vdm_increment")
    _launched(1)


# ---- P(k) --------------------------------------------------------------------------------------------
def _pk_shape(fields: torch.Tensor):
    _need(fields.is_cuda and fields.dtype == torch.float32 and fields.is_contiguous() and fields.dim() in (5, 6),
          "pk: fields must be contiguous CUDA fp32 [F, B, C, (n0,) n1, n2]")
    if fields.dim() == 5:
        f, b, c, n1, n2 = fields.shape
        n0 = 1
    else:
        f, b, c, n0, n1, n2 = fields.shape
    return f, b, c, n0, n1, n2


def pk_fields(fields: torch.Tensor, fields2: Optional[torch.Tensor] = None):
    """``vdm_pk``: per field f: power(fields[f], fields2[f]) of src/utils.py:16-83.
    fields: fp32 [F, B, C, n0, n1, n2] (3-D) or [F, B, C, n1, n2] (2-D).  Returns (k, P, N) as
    (double [F, kmax], double [F, kmax], int64 [F, kmax])."""
    f, b, c, n0, n1, n2 = _pk_shape(fields)
    if fields2 is not None:
        _need(fields2.shape == fields.shape and fields2.dtype == torch.float32 and fields2.is_contiguous(),
              "pk: fields2 must match fields")
    lib = _C.lib()
    nbytes = lib.vdm_pk_work_bytes(f, b, c, n0, n1, n2, 0 if fields2 is None else 1)
    work = torch.empty(nbytes, dtype=torch.uint8, device=fields.device)
    kmax = (min(n1, n2) if n0 == 1 else min(n0, n1, n2)) // 2
    k = torch.empty((f, kmax), dtype=torch.float64, device=fields.device)
    p = torch.empty_like(k)
    n = torch.empty((f, kmax), dtype=torch.int64, device=fields.device)
    rc = lib.vdm_pk(fields.data_ptr(), _ptr(fields2), f, b, c, n0, n1, n2, work.data_ptr(), nbytes, k.data_ptr(),
                    p.data_ptr(), n.data_ptr(), _stream())
    _C.check(rc, "vdm_pk")
    _launched(3)
    return k, p, n


def pk_cross3(fields1: torch.Tensor, fields2: torch.Tensor):
    """``vdm_pk_cross3``: (k, P11, P22, P12, N) from two transforms per field pair."""
    f, b, c, n0, n1, n2 = _pk_shape(fields1)
    _need(fields2.shape == fields1.shape and fields2.dtype == torch.float32 and fields2.is_contiguous() and
          fields2.is_cuda, "pk_cross3: fields2 must match fields1")
    lib = _C.lib()
    nbytes = lib.vdm_pk_work_bytes(f, b, c, n0, n1, n2, 1)
    work = torch.empty(nbytes, dtype=torch.uint8, device=fields1.device)
    kmax = (min(n1, n2) if n0 == 1 else min(n0, n1, n2)) // 2
    k = torch.empty((f, kmax), dtype=torch.float64, device=fields1.device)
    p11, p22, p12 = torch.empty_like(k), torch.empty_like(k), torch.empty_like(k)
    n = torch.empty((f, kmax), dtype=torch.int64, device=fields1.device)
    rc = lib.vdm_pk_cross3(fields1.data_ptr(), fields2.data_ptr(), f, b, c, n0, n1, n2, work.data_ptr(), nbytes,
                           k.data_ptr(), p11.data_ptr(), p22.data_ptr(), p12.data_ptr(), n.data_ptr(), _stream())
    _C.check(rc, "vdm_pk_cross3")
    _launched(3)
    return k, p11, p22, p12, n
