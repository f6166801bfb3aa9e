"""``CUNet``: the 3-D conditional UNet denoiser of vdm4cdm, B200-native.

Mirrors the interface the reference imports as ``mltools.networks.networks.CUNet`` (constructor call
sites: trainVDM3D128_c_c_from_field_name_thick_lowbatch.py:116-127, src/utils.py:451-462;
``forward(x, t, s_conditioning, v_conditionings)`` and the ``downs`` loop with ``no_down`` on the last
level: networks.py:259-265 recovered in model_test.ipynb:684; ResNetDown / ResNetBlock structure:
blocks.py:129-170, model_test.ipynb:686-692).

The torch modules below only HOLD the fp32 parameters (so ``state_dict`` keys are the usual
``conv_in.weight``, ``downs.0.resnet_blocks.0.net1.0.weight`` ...); the arithmetic of ``forward`` runs in
the sm_100a kernels behind ``vdm4cdm_b200.ops`` on channel-planar bf16 activations:

    conv_in / every Conv3d : vdm_conv3d   (tcgen05 implicit GEMM; bias + conditioning row, residual
                                            and GroupNorm statistics fused into the epilogue)
    GroupNorm+SiLU(+Dropout): vdm_gn_silu (one read, one write; statistics come from the producer)
    avg_pool3d / upsample   : vdm_avgpool2 / vdm_upsample2 (concat = plane windows of one buffer)

Only the tiny time / parameter embedding MLPs (B x <=256 GEMVs) stay in torch.  There is no PyTorch
fallback for the convolutional path; autograd support lives in ``vdm4cdm_b200.autograd``.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops


def timestep_embedding(t: torch.Tensor, dim: int, scale: float = 1000.0) -> torch.Tensor:
    """[sin(s t f_j), cos(s t f_j)], f_j = 1e4^(-j/half): the sinusoidal features fed to the time MLP."""
    half = dim // 2
    j = torch.arange(half, dtype=torch.float32, device=t.device)
    freqs = torch.exp(-math.log(10000.0) * j / half)
    args = (t.to(torch.float32) * scale)[:, None] * freqs[None, :]
    return torch.cat([torch.sin(args), torch.cos(args)], dim=1)


class ResNetBlock(nn.Module):
    """Parameter holder of a pre-activation residual block (GroupNorm first: blocks.py:129-132)."""

    def __init__(self, ch_in: int, ch_out: int, conditioning_dims: Sequence[int], dropout_prob: float,
                 norm_groups: int, padding_mode: str = "zeros"):
        super().__init__()
        self.ch_in, self.ch_out = ch_in, ch_out
        self.conditioning_dims = list(conditioning_dims)
        self.dropout_prob = dropout_prob
        self.norm_groups = norm_groups
        self.net1 = nn.Sequential(nn.GroupNorm(norm_groups, ch_in), nn.SiLU(),
                                  nn.Conv3d(ch_in, ch_out, 3, padding=1, padding_mode=padding_mode))
        self.cond_projs = nn.ModuleList([nn.Linear(d, ch_out) for d in self.conditioning_dims])
        self.net2 = nn.Sequential(nn.GroupNorm(norm_groups, ch_out), nn.SiLU(), nn.Dropout(dropout_prob),
                                  nn.Conv3d(ch_out, ch_out, 3, padding=1, padding_mode=padding_mode))
        self.skip_conv = nn.Conv3d(ch_in, ch_out, 1) if ch_in != ch_out else None

    def conditioning_row(self, conditionings: Optional[List[torch.Tensor]]) -> torch.Tensor:
        """bias of net1's conv + sum of the conditioning projections: fp32 [..., B, ch_out]."""
        row = self.net1[2].bias
        if conditionings is not None:
            assert len(conditionings) == len(self.conditioning_dims)
            for c, proj in zip(conditionings, self.cond_projs):
                row = row + proj(c)
        return row


class ResNetDown(nn.Module):
    def __init__(self, resnet_blocks: List[ResNetBlock]):
        super().__init__()
        self.resnet_blocks = nn.ModuleList(resnet_blocks)
        self.attention_blocks = None


class ResNetUp(nn.Module):
    def __init__(self, resnet_blocks: List[ResNetBlock]):
        super().__init__()
        self.resnet_blocks = nn.ModuleList(resnet_blocks)


class _Arena:
    """Per-(batch, grid) cache of activation buffers so the steady state allocates nothing."""

    def __init__(self):
        self.bufs: Dict[str, torch.Tensor] = {}

    def get(self, name: str, shape, dtype, device, zero: bool = False) -> torch.Tensor:
        t = self.bufs.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != device:
            t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=device)
            self.bufs[name] = t
        return t


class _PackedFilter:
    """A slot of ``CUNet._packed_cache``: ``buf``, a kernel-layout copy of (part of) ``conv.weight``; the ``key`` of the
    weights it was packed from; the recipe that packs it again.  ``buf`` is allocated once and re-packed in place, so
    captured CUDA graphs keep a valid pointer.  Recipes, ``kind`` (``args``):
      "bf16" (transpose_flip, c0, n): the forward filter, or the dgrad filter of input channels [c0, c0 + n);
      "f32" (): the fp32 forward filter of ``vdm_conv3d_tf32`` (own slots: switching precision does not re-pack);
      "slice" (c0, n): the bf16 forward filter of input channels [c0, c0 + n) (halves of an up block's convs);
      "poly" (c_up, group, n_par): the bf16 polyphase parity group of the first ``c_up`` input channels
          (``ops.polyphase_group``) and its ``taps``; the effective taps are summed in fp32 and rounded to bf16 once."""

    def __init__(self, conv: nn.Conv3d, kind: str, args: tuple):
        self.conv, self.kind, self.args = conv, kind, args
        self.key = self.buf = self.taps = None

    def weights_key(self, epoch: int) -> tuple:
        w = self.conv.weight
        return (w.data_ptr(), w._version, w.device, epoch)

    @torch.no_grad()
    def refresh(self, epoch: int) -> "_PackedFilter":
        """Re-pack ``buf`` if the weights changed since it was packed (``epoch``: ``CUNet.invalidate_packed`` count)."""
        key = self.weights_key(epoch)
        if key == self.key:
            return self
        w = self.conv.weight.detach()
        if self.kind == "poly":
            c_up, group, n_par = self.args
            part, self.taps = ops.polyphase_group(w[:, :c_up], group, n_par)
            packed = ops.pack_conv_weight(part)
            if self._fits(packed.shape, w.device):
                self.buf.copy_(packed)
            else:
                self.buf = packed
        else:
            if self.kind == "slice":
                w = w[:, self.args[0]:self.args[0] + self.args[1]]
            transpose_flip, c0, n = self.args if self.kind == "bf16" else (False, 0, None)
            dtype = torch.float32 if self.kind == "f32" else torch.bfloat16
            shape = ops.packed_weight_shape(w.shape, transpose_flip, n, dtype=dtype)
            if not self._fits(shape, w.device):
                self.buf = torch.empty(shape, dtype=dtype, device=w.device)
            ops.pack_conv_weight_into(w.contiguous(), self.buf, transpose_flip, c0, n)
        self.key = key
        return self

    def _fits(self, shape, device) -> bool:
        return self.buf is not None and tuple(self.buf.shape) == tuple(shape) and self.buf.device == device


class _Forms:
    """The fused forms one ``CUNet.run_packed`` call may use: bf16 inference only (training keeps every intermediate
    for the backward pass; TF32 runs the unfused path).  The ``CUNet`` switches turn them off one by one."""

    def __init__(self, net: "CUNet", tape: Optional[dict], training_dropout: bool):
        fused = tape is None and net.precision == "bf16"
        # GroupNorm + SiLU applied by the consumer conv to its input tiles (ops.conv3d in_norm): no dropout, zero padding
        self.gn = fused and net.fuse_gn and not training_dropout and not net.circular
        self.gn_min_channels = net.fuse_gn_min_channels
        # up blocks read the coarse tensor (see CUNet._run_block); only then is their skip conv tried fused into net2's
        self.read_coarse = fused and net.fuse_upsample
        self.polyphase = self.read_coarse and net.polyphase_up and not net.circular

    def gn_in_conv(self, c_in: int, c_out: int) -> bool:
        """Whether a ``c_in`` -> ``c_out`` conv normalises its own input: layers of at least ``fuse_gn_min_channels``
        outputs (tile kernel, four warps share every halo stage) and the narrow layers of the marching schedule (at most
        32 channels in and out; R4k, 128^3 x 8: 12.40 -> 11.81 ms per step).  In between (the kd-folded TILE schedule) the
        transform's LDS / STS traffic costs more than the HBM pass it replaces (profiles/R2h_transform_ablation.txt)."""
        return self.gn and (c_out >= self.gn_min_channels or (c_in <= 32 and c_out <= 32))


class CUNet(nn.Module):
    def __init__(self, shape=(1, 128, 128, 128), chs=(32, 64, 128, 256), s_conditioning_channels: int = 0,
                 v_conditioning_dims: Sequence[int] = (), t_conditioning: bool = False, norm_groups: int = 8,
                 mid_attn: bool = False, dropout_prob: float = 0.1, conv_padding_mode: str = "zeros",
                 n_attention_heads: int = 4, t_embedding_dim: int = 64, v_embedding_dim: int = 64,
                 out_channels: Optional[int] = None, precision: str = "bf16"):
        super().__init__()
        # Inference precision of the convolutional trunk: "bf16" (bf16 channel-planar activations, bf16 tensor-core convs) or
        # "tf32" (fp32 channel-planar activations, tcgen05 kind::tf32 convs -- the reference's own cuDNN TF32 class of
        # accuracy, for A/B comparisons).  A plain attribute: it may be changed on a loaded model.  TF32 is inference-only
        # and runs the unfused path (no fuse_gn / fuse_upsample / polyphase_up / fused skip conv).
        self.precision = precision
        self._check_precision()
        if len(shape) != 4:
            raise NotImplementedError("vdm4cdm_b200.CUNet covers the 3-D networks (shape=(C, D, H, W)) only")
        if mid_attn:
            raise NotImplementedError("mid_attn=True is used by the reference's 2-D scripts only")
        if conv_padding_mode not in ("zeros", "circular"):
            raise NotImplementedError(f"conv_padding_mode={conv_padding_mode!r}: 'zeros' and 'circular' are supported")
        if shape[0] != 1 or (out_channels not in (None, 1)):
            raise NotImplementedError("single-channel fields only (every 3-D config of the reference)")
        if s_conditioning_channels + 1 > 8:
            raise NotImplementedError("at most 7 spatial conditioning channels")
        for c in chs:
            if c % 16 != 0 or c > 256:
                raise NotImplementedError(f"channel widths must be multiples of 16 and <= 256, got {chs}")
        for n in shape[1:]:
            if n % (2 ** (len(chs) - 1)) != 0:
                raise ValueError(f"grid {shape[1:]} is not divisible by 2^{len(chs) - 1}")
        self.shape = tuple(shape)
        self.circular = conv_padding_mode == "circular"     # the cropsize == 256 models (src/utils.py:460)
        self.fuse_upsample = True       # inference: up blocks read the coarse tensor instead of its up-sampled copy
        # inference: GroupNorm + SiLU in front of a conv is applied by the conv kernel to its input tile (ops.conv3d
        # in_norm) instead of by a separate read + write pass over the tensor, for the layers _Forms.gn_in_conv picks
        self.fuse_gn = True
        self.fuse_gn_min_channels = 64
        # inference, up blocks: conv3x3x3 over the up-sampled half of cat([interpolate(h), skip]) in its polyphase form --
        # eight 2x2x2-tap convolutions of the COARSE tensor, one per output parity (8/27 of the multiply-adds, the
        # up-sampled activations are never written); the skip half is a plain conv that adds them as its residual
        self.polyphase_up = True
        self._fused_skip_ok = {}        # per up block: False once vdm_conv3d declined the fused skip conv
        self.chs = list(chs)
        self.s_conditioning_channels = s_conditioning_channels
        self.v_conditioning_dims = list(v_conditioning_dims)
        self.t_conditioning = t_conditioning
        self.t_embedding_dim = t_embedding_dim
        self.v_embedding_dim = v_embedding_dim
        self.norm_groups = norm_groups
        self.dropout_prob = dropout_prob
        self.n_attention_heads = n_attention_heads
        in_ch = shape[0] + s_conditioning_channels
        pm = conv_padding_mode

        cond_dims = []
        if t_conditioning:
            self.t_embed = nn.Sequential(nn.Linear(t_embedding_dim, 4 * t_embedding_dim), nn.SiLU(),
                                         nn.Linear(4 * t_embedding_dim, t_embedding_dim), nn.SiLU())
            cond_dims.append(t_embedding_dim)
        self.v_embeds = nn.ModuleList()
        for d in self.v_conditioning_dims:
            self.v_embeds.append(nn.Sequential(nn.Linear(d, 4 * v_embedding_dim), nn.SiLU(),
                                               nn.Linear(4 * v_embedding_dim, v_embedding_dim), nn.SiLU()))
            cond_dims.append(v_embedding_dim)
        self.conditioning_dims = cond_dims

        def block(ci, co):
            return ResNetBlock(ci, co, cond_dims, dropout_prob, norm_groups, pm)

        c = self.chs
        self.conv_in = nn.Conv3d(in_ch, c[0], 3, padding=1, padding_mode=pm)
        self.downs = nn.ModuleList([ResNetDown([block(c[max(i - 1, 0)], c[i])]) for i in range(len(c))])
        self.mid1 = block(c[-1], c[-1])
        self.mid2 = block(c[-1], c[-1])
        self.ups = nn.ModuleList([ResNetUp([block(c[i + 1] + c[i], c[i])]) for i in reversed(range(len(c) - 1))])
        self.conv_out = nn.Sequential(nn.GroupNorm(norm_groups, c[0]), nn.SiLU(),
                                      nn.Conv3d(c[0], 1, 3, padding=1, padding_mode=pm))
        self._arena = _Arena()
        self._train_arena = _Arena()
        self._packed_cache: Dict[str, _PackedFilter] = {}
        self._pack_tables: Dict[tuple, torch.Tensor] = {}
        self._weights_epoch = 0
        self.dropout_seed = 0
        self._dropout_calls = 0
        # device-side training-step counter added to the dropout seed (a captured CUDA graph draws new masks)
        self.register_buffer("drop_counter", torch.zeros(1, dtype=torch.int32), persistent=False)

    PRECISIONS = ("bf16", "tf32")

    def _check_precision(self) -> bool:
        """True in TF32 mode; ValueError for an unknown ``precision``."""
        if self.precision not in self.PRECISIONS:
            raise ValueError(f"CUNet.precision must be one of {self.PRECISIONS}, got {self.precision!r}")
        return self.precision == "tf32"

    def _lanes(self) -> int:
        """Channels per plane of the trunk's planar activations: 8 (bf16) or 4 (TF32 mode, fp32)."""
        return 4 if self.precision == "tf32" else 8

    def _planar(self, ar: "_Arena", name: str, b: int, ch: int, grid, dev) -> torch.Tensor:
        """Arena buffer of a ``ch``-channel planar activation on ``grid`` in the trunk's precision: bf16 [b, ch/8, *grid, 8]
        or (TF32) fp32 [b, ch/4, *grid, 4]."""
        lanes = self._lanes()
        if lanes == 4:       # own buffers: a CUDA graph captured in the other precision keeps valid pointers
            return ar.get("f32." + name, (b, ch // 4) + tuple(grid) + (4,), torch.float32, dev)
        return ar.get(name, (b, ch // 8) + tuple(grid) + (8,), torch.bfloat16, dev)

    def input_channels_pad(self) -> int:
        """Channels of the packed network input (``ops.pack_input``'s ``c_pad``): 16 bf16 or 8 fp32 = two planes."""
        return 8 if self.precision == "tf32" else 16

    # ---- conditioning (tiny fp32 MLPs, torch) -------------------------------------------------
    def conditionings(self, batch: int, t, v_conditionings, device) -> Optional[List[torch.Tensor]]:
        """List of fp32 [..., B, dim] embeddings (time first, then one per parameter vector).

        ``t`` may be (B,), a scalar, or (S, B) for S pre-computed sampler steps."""
        out = []
        if self.t_conditioning:
            tt = torch.as_tensor(t, dtype=torch.float32, device=device)
            if tt.dim() == 0 or tt.numel() == 1:
                tt = tt.reshape(1).expand(batch)
            lead = tt.shape[:-1]
            emb = self.t_embed(timestep_embedding(tt.reshape(-1), self.t_embedding_dim))
            out.append(emb.reshape(*lead, batch, -1))
        v_conditionings = [] if v_conditionings is None else v_conditionings
        assert len(v_conditionings) == len(self.v_embeds)
        for v, emb in zip(v_conditionings, self.v_embeds):
            out.append(emb(v.to(torch.float32)))
        return out if len(out) else None

    # ---- packed weights (kernel layout), re-packed in place when the fp32 parameter changes ------------
    def invalidate_packed(self) -> None:
        """Tell the weight caches that the fp32 parameters changed behind torch's back (the fused
        optimizer kernel writes through raw pointers, which does not bump ``Tensor._version``)."""
        self._weights_epoch += 1

    def _slot(self, slot: str, conv: nn.Conv3d, kind: str, *args) -> _PackedFilter:
        """Cache slot ``slot`` (recipe ``kind``, ``args`` of ``_PackedFilter``), packed on first use, up to date."""
        f = self._packed_cache.get(slot)
        if f is None:
            f = self._packed_cache[slot] = _PackedFilter(conv, kind, args)
        return f.refresh(self._weights_epoch)

    def _packed(self, name: str, conv: nn.Conv3d) -> torch.Tensor:
        """Forward filter of ``conv`` in the trunk's precision: bf16, or in TF32 mode the fp32 filter of ``vdm_conv3d_tf32``."""
        if self.precision == "tf32":
            return self._slot(name + ".f32", conv, "f32").buf
        return self._slot(name, conv, "bf16", False, 0, conv.in_channels).buf

    def _packed_dgrad(self, name: str, conv: nn.Conv3d, c0: int, n: int) -> torch.Tensor:
        """bf16 dgrad filter (roles of Cin/Cout exchanged, taps mirrored) for input channels [c0, c0+n)."""
        return self._slot(f"{name}.dgrad.{c0}.{n}", conv, "bf16", True, c0, n).buf

    def repack_all(self) -> None:
        """Re-pack every stale whole-weight bf16 filter the trunk has used so far (forward and dgrad variants) in one
        ``vdm_pack_conv_weight_batched`` launch -- the training step does this after each optimizer update instead of
        letting ~56 lazy single-filter launches happen."""
        e = self._weights_epoch
        stale = [(slot, f) for slot, f in self._packed_cache.items() if f.kind == "bf16" and f.conv.weight.is_cuda and
                 f.conv.weight.is_contiguous() and f.buf.device == f.conv.weight.device and f.key != f.weights_key(e)]
        if not stale:
            return
        tkey = tuple((slot, f.conv.weight.data_ptr(), f.buf.data_ptr()) for slot, f in stale)
        table = self._pack_tables.get(tkey)
        if table is None:
            self._pack_tables.clear()
            table = ops.pack_job_table([(f.conv.weight.detach(), f.buf, *f.args) for _, f in stale], stale[0][1].buf.device)
            self._pack_tables[tkey] = table
        with torch.no_grad():
            ops.pack_conv_weights_batched(table, len(stale))
        for _, f in stale:
            f.key = f.weights_key(e)

    def refresh_packed(self, training: bool = False) -> None:
        """Re-pack (in place) every cached filter whose fp32 parameter changed since it was packed, and pack the trunk's
        forward filters in the current precision if missing: the whole-weight bf16 filters in one batched launch
        (``repack_all``), every other slot by its own recipe.  A captured sampler graph reads the slots without packing
        lazily, so ``SamplerSession.reset`` calls this.  ``training=True`` (every training forward) skips the slots that
        only inference reads (fp32, slices, polyphase groups): they are re-packed when next used."""
        self.repack_all()
        for name, conv in self._convs():
            self._packed(name, conv)
        if not training:
            for f in self._packed_cache.values():
                f.refresh(self._weights_epoch)

    def trunk_parameters(self):
        """(name, parameter) of everything the convolutional trunk differentiates itself: conv filters and
        GroupNorm affines, named as ``vdm4cdm_b200.autograd`` records their gradients.  (Conv biases and the
        embedding MLPs get theirs through the conditioning rows under torch autograd.)"""
        gn = self.conv_out[0]
        out = [("conv_in.weight", self.conv_in.weight), ("conv_out.weight", self.conv_out[2].weight),
               ("conv_out.gn.weight", gn.weight), ("conv_out.gn.bias", gn.bias)]
        for name, blk in self._blocks():
            out += [(name + ".net1.weight", blk.net1[2].weight), (name + ".net2.weight", blk.net2[3].weight),
                    (name + ".gn1.weight", blk.net1[0].weight), (name + ".gn1.bias", blk.net1[0].bias),
                    (name + ".gn2.weight", blk.net2[0].weight), (name + ".gn2.bias", blk.net2[0].bias)]
            if blk.skip_conv is not None:
                out.append((name + ".skip.weight", blk.skip_conv.weight))
        return out

    def _convs(self):
        out = [("conv_in", self.conv_in), ("conv_out", self.conv_out[2])]
        for name, blk in self._blocks():
            out += [(name + ".net1", blk.net1[2]), (name + ".net2", blk.net2[3])]
            if blk.skip_conv is not None:
                out.append((name + ".skip", blk.skip_conv))
        return out

    def conv_flops_per_sample(self) -> float:
        """Algorithmic conv FLOPs of one forward for one sample: sum of 2 k^3 Cin Cout D H W over the
        Conv3d modules (SURVEY.md section 8d), with the real (un-padded) channel counts."""
        nl = len(self.chs)
        vox = [math.prod(n >> i for n in self.shape[1:]) for i in range(nl)]
        level = {"conv_in": 0, "conv_out": 0, "mid1": nl - 1, "mid2": nl - 1}
        for i in range(nl):
            level[f"downs.{i}.resnet_blocks.0"] = i
        for k, i in enumerate(reversed(range(nl - 1))):
            level[f"ups.{k}.resnet_blocks.0"] = i
        total = 0.0
        for name, conv in self._convs():
            base = name if name in level else name.rsplit(".", 1)[0]
            k3 = conv.kernel_size[0] * conv.kernel_size[1] * conv.kernel_size[2]
            total += 2.0 * k3 * conv.in_channels * conv.out_channels * vox[level[base]]
        return total

    def _blocks(self):
        """(name, block) in execution order."""
        out = []
        for i, down in enumerate(self.downs):
            out.append((f"downs.{i}.resnet_blocks.0", down.resnet_blocks[0]))
        out += [("mid1", self.mid1), ("mid2", self.mid2)]
        for i, up in enumerate(self.ups):
            out.append((f"ups.{i}.resnet_blocks.0", up.resnet_blocks[0]))
        return out

    def chan_add_rows(self, batch: int, t, v_conditionings, device) -> Dict[str, torch.Tensor]:
        """Every per-channel row the conv epilogues add: bias (+ conditioning projections for net1).

        Shapes are [B, c] or, when ``t`` is (S, B), [S, B, c] for the block convs that see the time."""
        conds = self.conditionings(batch, t, v_conditionings, device)
        rows = {"conv_in": self.conv_in.bias.expand(batch, -1).contiguous(),
                "conv_out": self.conv_out[2].bias.expand(batch, -1).contiguous()}
        for name, blk in self._blocks():
            row = blk.conditioning_row(conds)
            if row.dim() == 1:
                row = row.expand(batch, -1)
            rows[name + ".net1"] = row.contiguous().float()
            rows[name + ".net2"] = blk.net2[3].bias.expand(batch, -1).contiguous()
            if blk.skip_conv is not None:
                rows[name + ".skip"] = blk.skip_conv.bias.expand(batch, -1).contiguous()
        return rows

    # ---- the convolutional trunk on channel-planar buffers --------------------------------------
    def _run_block(self, name, blk: ResNetBlock, forms: _Forms, x, x_plane0, x_stats, rows, step_ptr, out, out_plane0,
                   out_stats, out_stats_c0, grid, training_dropout, tape=None, up_from=None):
        """out[window] = block(x[window]).  x_stats: double [B, ch_in, 2] of x.  With a ``tape`` (training)
        every intermediate gets its own buffer and is recorded for the backward pass.

        ``up_from = (coarse, plane0, c_up)`` (inference, up blocks): the first ``c_up`` channels of the block input are
        ``interpolate(coarse)`` and have NOT been written to ``x``.  Nearest up-sampling commutes with pointwise
        operations and with 1x1x1 convs and keeps per-channel means / variances, so the block reads the coarse tensor
        instead: net1's GroupNorm+SiLU up-samples while it normalises, and the skip conv becomes
        ``conv(x[c_up:]) + interpolate(conv(coarse))`` -- the concatenated up-sampled tensor (2/3 of the block input)
        is never materialised, which removes one write and two reads of it per up block (r02f)."""
        b = x.shape[0]
        dev = x.device
        ar = self._arena if tape is None else self._train_arena
        ci, co, g = blk.ch_in, blk.ch_out, blk.norm_groups
        tag = f"{b}x{grid[0]}"
        own = "" if tape is None else name + "."
        n1 = blk.net1[0]
        voxels = grid[0] * grid[1] * grid[2]
        p_drop = blk.dropout_prob if training_dropout else 0.0
        xc, xc_plane0, c_up = up_from or (None, 0, 0)
        c_sk = ci - c_up                            # channels of the block input held by x
        h = self._planar(ar, f"{own}h.{co}.{tag}", b, co, grid, dev)
        h_stats = self._stats(f"{name}.h", b, co, dev)
        net1_kw = dict(out=h, chan_add=rows[name + ".net1"], step_ptr=step_ptr if rows[name + ".net1"].dim() == 3 else None,
                       stats=h_stats, circular=self.circular)
        if up_from is None and forms.gn_in_conv(ci, co):
            coef1 = ops.gn_coef(x_stats, n1.weight, n1.bias, g, voxels, n1.eps,
                                out=ar.get(f"coef1.{name}.{b}", (b, ci, 2), torch.float32, dev))
            ops.conv3d(x, self._packed(name + ".net1", blk.net1[2]), co, x_plane0=x_plane0, c_in=ci, in_norm=coef1, **net1_kw)
        elif up_from is not None and forms.polyphase:
            cgrid = tuple(n // 2 for n in grid)
            # silu(gn(.)) of the coarse channels at the COARSE resolution (statistics of the fine concat)
            ac = ar.get(f"ac.{c_up}.{b}x{cgrid[0]}", (b, c_up // 8) + cgrid + (8,), torch.bfloat16, dev)
            ops.gn_silu_view(xc, c_up, 0, ci, g, x_stats, n1.weight, n1.bias, n1.eps, ac, x_plane0=xc_plane0, upsample="coarse")
            # the eight parity convolutions (2x2x2 taps each on the coarse grid) -> parity-planar partial sums [8 x co
            # channels], n_par parities per launch stacked along N (N = n_par * co <= 256)
            part = ar.get(f"poly.{co}.{b}x{cgrid[0]}", (b, co) + cgrid + (8,), torch.bfloat16, dev)
            # (measured at 128^3 x 8, R2t: N = 128 per launch where the layer is narrow -- 32 channels: 4 parities, 1.17 ms
            #  in 2 launches vs 1.53 in 8; 64 channels: 2 parities, 0.42 ms in 4 launches vs 0.64 in 8 / 0.56 in 2; 128
            #  channels: 2 parities (N = 256), 0.25 ms in 4 launches vs 0.30 in 8)
            n_par = 4 if co <= 32 else 2
            for grp in range(8 // n_par):
                poly = self._slot(f"{name}.net1.poly.{n_par}.{grp}", blk.net1[2], "poly", c_up, grp, n_par)
                ops.conv3d(ac, poly.buf, n_par * co, taps=poly.taps, out=part, out_plane0=grp * n_par * (co // 8))
            # the skip channels at the fine resolution; the partial sums come in through the depth-to-space residual
            w_sk = self._slot(name + ".net1.skiphalf", blk.net1[2], "slice", c_up, c_sk).buf
            if forms.gn_in_conv(c_sk, co):
                # GroupNorm + SiLU of the skip channels applied by the conv to its input tiles: (a, b) of all ci channels of
                # the concat norm (groups straddle the two halves), the skip channels' rows handed to the conv
                coef = ops.gn_coef(x_stats, n1.weight, n1.bias, g, voxels, n1.eps,
                                   out=ar.get(f"coef1.{name}.{b}", (b, ci, 2), torch.float32, dev))
                coef_s = ar.get(f"coef1s.{name}.{b}", (b, c_sk, 2), torch.float32, dev)
                coef_s.copy_(coef[:, c_up:])
                ops.conv3d(x, w_sk, co, x_plane0=x_plane0 + c_up // 8, c_in=c_sk, residual=part, residual_upsample="d2s",
                           in_norm=coef_s, **net1_kw)
            else:
                a_s = ar.get(f"as.{c_sk}.{tag}", (b, c_sk // 8) + grid + (8,), torch.bfloat16, dev)
                ops.gn_silu_view(x, c_sk, c_up, ci, g, x_stats, n1.weight, n1.bias, n1.eps, a_s, x_plane0=x_plane0 + c_up // 8)
                ops.conv3d(a_s, w_sk, co, residual=part, residual_upsample="d2s", **net1_kw)
        else:
            a1 = self._planar(ar, f"{own}a.{ci}.{tag}", b, ci, grid, dev)
            if up_from is None:
                ops.gn_silu(x, ci, g, x_stats, n1.weight, n1.bias, n1.eps, x_plane0=x_plane0, out=a1)
            else:
                ops.gn_silu_view(xc, c_up, 0, ci, g, x_stats, n1.weight, n1.bias, n1.eps, a1, x_plane0=xc_plane0,
                                 out_plane0=0, upsample=True)
                ops.gn_silu_view(x, c_sk, c_up, ci, g, x_stats, n1.weight, n1.bias, n1.eps, a1,
                                 x_plane0=x_plane0 + c_up // 8, out_plane0=c_up // 8)
            a1c, _ = self._conv_input(a1, ci, 0, name + ".a1p", tape)
            ops.conv3d(a1c, self._packed(name + ".net1", blk.net1[2]), co, **net1_kw)
        if p_drop > 0.0:
            self._dropout_calls += 1
        n2 = blk.net2[0]
        if forms.gn_in_conv(co, co):
            # net2's conv reads h itself; (a, b) per (sample, channel) from h's statistics
            a2c = h
            in_norm2 = ops.gn_coef(h_stats, n2.weight, n2.bias, g, voxels, n2.eps,
                                   out=ar.get(f"coef2.{name}.{b}", (b, co, 2), torch.float32, dev))
        else:
            in_norm2 = None
            a2 = self._planar(ar, f"{own}a2.{co}.{tag}" if tape is not None else f"a.{co}.{tag}", b, co, grid, dev)
            ops.gn_silu(h, co, g, h_stats, n2.weight, n2.bias, n2.eps, out=a2, dropout_p=p_drop,
                        seed=self.dropout_seed, layer_tag=self._dropout_calls,
                        seed_step=self.drop_counter if p_drop > 0.0 else None)
            a2c, _ = self._conv_input(a2, co, 0, name + ".a2p", tape)
        if tape is not None:
            tape[name] = dict(x=x, x_plane0=x_plane0, x_stats=x_stats, a1=a1c, h=h, h_stats=h_stats, a2=a2c, grid=grid,
                              p_drop=p_drop, drop_tag=self._dropout_calls, drop_seed=self.dropout_seed)
        if blk.skip_conv is None:
            res, res_plane0 = x, x_plane0
        elif up_from is not None:
            # coarse half of the skip conv (with the skip conv's bias): a small 1x1x1 conv on the half-resolution grid
            rc = ar.get(f"rc.{co}.{b}x{grid[0] // 2}", (b, co // 8) + tuple(n // 2 for n in grid) + (8,), torch.bfloat16, dev)
            ops.conv3d(xc, self._slot(name + ".skip.up", blk.skip_conv, "slice", 0, c_up).buf, co, taps=ops.TAPS_1X1X1,
                       x_plane0=xc_plane0, c_in=c_up, out=rc, chan_add=rows[name + ".skip"])
            w_skip = self._slot(name + ".skip.skip", blk.skip_conv, "slice", c_up, c_sk).buf
            if self._fused_skip_ok.get(name, True):
                # fine half fused into net2's conv as one more channel chunk (centre tap only): no separate 1x1x1 launch,
                # and the residual the epilogue reads is the coarse tensor (1/8 of the bytes)
                try:
                    ops.conv3d(a2c, self._packed(name + ".net2", blk.net2[3]), co, out=out, out_plane0=out_plane0,
                               chan_add=rows[name + ".net2"], residual=rc, residual_upsample=True, stats=out_stats,
                               stats_c0=out_stats_c0, skip_x=x, skip_w=w_skip, skip_plane0=x_plane0 + c_up // 8,
                               circular=self.circular, in_norm=in_norm2)
                    return
                except ops.UnsupportedFusion:
                    self._fused_skip_ok[name] = False          # wide layer: keep the skip conv as its own launch
            res = self._planar(ar, f"{own}r.{co}.{tag}", b, co, grid, dev)
            ops.conv3d(x, w_skip, co, taps=ops.TAPS_1X1X1, x_plane0=x_plane0 + c_up // 8, c_in=c_sk, out=res,
                       residual=rc, residual_upsample=True)
            res_plane0 = 0
        else:
            res = self._planar(ar, f"{own}r.{co}.{tag}", b, co, grid, dev)
            ops.conv3d(x, self._packed(name + ".skip", blk.skip_conv), co, taps=ops.TAPS_1X1X1, x_plane0=x_plane0, c_in=ci,
                       out=res, chan_add=rows[name + ".skip"])
            res_plane0 = 0
        ops.conv3d(a2c, self._packed(name + ".net2", blk.net2[3]), co, out=out, out_plane0=out_plane0,
                   chan_add=rows[name + ".net2"], residual=res, residual_plane0=res_plane0, stats=out_stats,
                   stats_c0=out_stats_c0, circular=self.circular, in_norm=in_norm2)

    def _conv_input(self, x, ch, x_plane0, slot, tape):
        """The tensor a 3x3x3 conv reads: ``x`` itself (zero padding is the TMA unit's out-of-bounds fill) or, for
        circular padding, a copy with a one-voxel periodic halo (``vdm_pad_circular``)."""
        if not self.circular:
            return x, x_plane0
        b = x.shape[0]
        d, h, w = x.shape[2:5]
        ar = self._arena if tape is None else self._train_arena
        name = (slot if tape is not None else "pad") + f".{ch}.{b}x{d}"
        buf = self._planar(ar, name, b, ch, (d + 2, h + 2, w + 2), x.device)
        ops.pad_circular(x, ch, x_plane0=x_plane0, out=buf)
        return buf, 0

    def _stats(self, name: str, b: int, c: int, dev) -> torch.Tensor:
        """A zeroed double [B, c, 2] slice of the per-forward statistics arena."""
        off = self._stats_off
        n = b * c * 2
        self._stats_off += n
        if self._stats_off > self._stats_arena.numel():
            raise RuntimeError("statistics arena too small")  # sized generously in run_packed
        return self._stats_arena[off:off + n].view(b, c, 2)

    def run_packed(self, packed: torch.Tensor, rows: Dict[str, torch.Tensor], step_ptr: Optional[torch.Tensor] = None,
                   out: Optional[torch.Tensor] = None, training_dropout: bool = False, tape: Optional[dict] = None) -> torch.Tensor:
        """eps_hat fp32 (B, 1, D, H, W) from the packed network input (``ops.pack_input``).

        ``tape`` (a dict, training only): intermediates live in a separate arena, nothing is shared between
        layers, and every tensor the backward pass needs is recorded in it (``vdm4cdm_b200.autograd``).
        In TF32 mode ``packed`` is the fp32 planar input and ``tape`` is refused (the mode is inference-only)."""
        if self._check_precision() and tape is not None:
            raise NotImplementedError("CUNet precision='tf32' is inference-only (no training tape)")
        forms = _Forms(self, tape, training_dropout)
        lanes = self._lanes()
        b = packed.shape[0]
        dev = packed.device
        c = self.chs
        nl = len(c)
        grids = [tuple(n >> i for n in self.shape[1:]) for i in range(nl)]
        ar = self._arena if tape is None else self._train_arena
        self._stats_arena = ar.get(f"stats.{b}", (b * 2 * (16 * sum(c) + 64),), torch.float64, dev)
        self._stats_arena.zero_()
        self._stats_off = 0
        self._dropout_calls = 0

        def buf(name, ch, lvl):
            return self._planar(ar, f"{name}.{b}", b, ch, grids[lvl], dev)

        # conv_in
        h = buf("h_in", c[0], 0)
        h_stats = self._stats("conv_in", b, c[0], dev)
        packed_c, _ = self._conv_input(packed, self.input_channels_pad(), 0, "conv_in.xp", tape)
        ops.conv3d(packed_c, self._packed("conv_in", self.conv_in), c[0], out=h, chan_add=rows["conv_in"], stats=h_stats,
                   circular=self.circular)
        x, x_plane0, x_stats = h, 0, h_stats
        # down path: the block output of level i < last lands in the concat buffer of the matching up level
        cats, cat_stats = {}, {}
        for i in range(nl):
            blk = self.downs[i].resnet_blocks[0]
            name = f"downs.{i}.resnet_blocks.0"
            if i < nl - 1:
                cat = buf(f"cat{i}", c[i + 1] + c[i], i)
                cst = self._stats(f"cat{i}", b, c[i + 1] + c[i], dev)
                cats[i], cat_stats[i] = cat, cst
                self._run_block(name, blk, forms, x, x_plane0, x_stats, rows, step_ptr, cat, c[i + 1] // lanes, cst, c[i + 1],
                                grids[i], training_dropout, tape)
                pooled = buf(f"pool{i}", c[i], i + 1)
                pst = self._stats(f"pool{i}", b, c[i], dev)
                ops.avgpool2(cat, c[i], x_plane0=c[i + 1] // lanes, out=pooled, stats=pst)
                x, x_plane0, x_stats = pooled, 0, pst
            else:
                o = buf("bottom0", c[i], i)
                ost = self._stats("bottom0", b, c[i], dev)
                self._run_block(name, blk, forms, x, x_plane0, x_stats, rows, step_ptr, o, 0, ost, 0, grids[i], training_dropout,
                                tape)
                x, x_plane0, x_stats = o, 0, ost
        for j, (name, blk) in enumerate((("mid1", self.mid1), ("mid2", self.mid2))):
            o = buf(f"bottom{1 + j}", c[-1], nl - 1)
            ost = self._stats(name + ".out", b, c[-1], dev)
            self._run_block(name, blk, forms, x, x_plane0, x_stats, rows, step_ptr, o, 0, ost, 0, grids[-1], training_dropout,
                            tape)
            x, x_plane0, x_stats = o, 0, ost
        for k, i in enumerate(reversed(range(nl - 1))):
            blk = self.ups[k].resnet_blocks[0]
            name = f"ups.{k}.resnet_blocks.0"
            cat, cst = cats[i], cat_stats[i]
            o = buf(f"up{i}", c[i], i)
            ost = self._stats(name + ".out", b, c[i], dev)
            if forms.read_coarse and blk.skip_conv is not None:
                # the up-sampled channels are never written (see _run_block); their sums are 8x the coarse tensor's
                torch.mul(x_stats, 8.0, out=cst[:, :c[i + 1]])
                self._run_block(name, blk, forms, cat, 0, cst, rows, step_ptr, o, 0, ost, 0, grids[i], training_dropout, tape,
                                up_from=(x, x_plane0, c[i + 1]))
            else:
                ops.upsample2(x, c[i + 1], cat, coarse_plane0=x_plane0, out_plane0=0, stats=cst, stats_c0=0)
                self._run_block(name, blk, forms, cat, 0, cst, rows, step_ptr, o, 0, ost, 0, grids[i], training_dropout, tape)
            x, x_plane0, x_stats = o, 0, ost
        gn = self.conv_out[0]
        if out is None:
            out = torch.empty((b, 1) + grids[0], dtype=torch.float32, device=dev)
        if forms.gn_in_conv(c[0], 1):
            coef = ops.gn_coef(x_stats, gn.weight, gn.bias, gn.num_groups, grids[0][0] * grids[0][1] * grids[0][2], gn.eps,
                               out=ar.get(f"coef.conv_out.{b}", (b, c[0], 2), torch.float32, dev))
            ops.conv3d(x, self._packed("conv_out", self.conv_out[2]), 1, x_plane0=x_plane0, c_in=c[0], out=out, out_fp32=True,
                       chan_add=rows["conv_out"], in_norm=coef)
            return out
        a = self._planar(ar, ("conv_out." if tape is not None else "") + f"a.{c[0]}.{b}x{grids[0][0]}", b, c[0], grids[0], dev)
        ops.gn_silu(x, c[0], gn.num_groups, x_stats, gn.weight, gn.bias, gn.eps, out=a)
        a_c, _ = self._conv_input(a, c[0], 0, "conv_out.ap", tape)
        if tape is not None:
            tape["trunk"] = dict(packed=packed_c, h_in=h, cats=cats, grids=grids, out_x=x, out_x_stats=x_stats, out_a=a_c)
        ops.conv3d(a_c, self._packed("conv_out", self.conv_out[2]), 1, out=out, out_fp32=True, chan_add=rows["conv_out"],
                   circular=self.circular)
        return out

    def forward(self, x, t=None, s_conditioning=None, v_conditionings=None):
        """eps_hat / v_hat (B, 1, D, H, W) fp32.  Under ``torch.no_grad()`` this is the inference path; with
        gradients enabled it goes through ``vdm4cdm_b200.autograd.unet_forward`` (dropout active iff
        ``self.training``)."""
        tf32 = self._check_precision()
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            if tf32:
                raise NotImplementedError("CUNet precision='tf32' is inference-only: run it under torch.no_grad()")
            from .autograd import unet_forward
            return unet_forward(self, x, t, s_conditioning, v_conditionings)
        with torch.no_grad():
            b = x.shape[0]
            rows = self.chan_add_rows(b, t, v_conditionings, x.device)
            cond = None if s_conditioning is None else s_conditioning.contiguous().float()
            packed = ops.pack_input(x.contiguous().float(), cond, self.input_channels_pad(),
                                    out=self._planar(self._arena, f"packed.{b}", b, self.input_channels_pad(), self.shape[1:],
                                                     x.device))
            return self.run_packed(packed, rows)
