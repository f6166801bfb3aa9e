"""Training path of the CUNet: forward with a tape + hand-scheduled backward on the sm_100a kernels.

Stands in for what autograd records and replays for ``LightVDM.training_step`` / ``LightSFM.training_step``
(trainVDM3D128_c_c_from_field_name_thick_lowbatch.py:128-160 and trainSFM3D160_...:124-150 drive them through
``lightning.Trainer.fit``): cuDNN conv3d backward-data / backward-filter, native_group_norm_backward,
silu_backward, the dropout mask multiply, avg_pool3d_backward, upsample_nearest3d_backward and the
``cat`` split.  Here the whole trunk is ONE ``torch.autograd.Function``:

  forward   ``CUNet.run_packed(..., tape=...)``: same kernels as inference, every intermediate kept
  backward  per ResNet block (y = conv2(drop(silu(gn2(h)))) + skip(x), h = conv1(silu(gn1(x))) + row):
              dW2 = wgrad(a2, dy)            d_a2 = dgrad(dy, W2)            (tcgen05)
              dh  = gn_silu_bwd(h, d_a2)     dgamma2/dbeta2, d_row1 = sum_v dh
              dW1 = wgrad(a1, dh)            d_a1 = dgrad(dh, W1)
              dx  = gn_silu_bwd(x, d_a1) + (dy | dgrad_1x1(dy, Wskip))       dgamma1/dbeta1
            concat split = plane windows of the gradient buffer; the skip gradient and the pooled
            gradient meet by accumulating ``avgpool2_bwd`` in place.
Gradients are bf16 channel-planar (fp32 accumulation inside every kernel); weight gradients are fp32.
Only the tiny embedding MLPs, the bias/conditioning rows and the scalar loss glue run under torch autograd.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch

from . import ops


def _chunks(c: int, limit: int = 256) -> List[tuple]:
    """Split c dgrad output channels into launches of <= limit (256 = the UMMA N limit), multiples of 8."""
    n = -(-c // limit)
    while c % n != 0 or (c // n) % 8 != 0:
        n += 1
    step = c // n
    return [(i * step, step) for i in range(n)]


class _Backward:
    """One backward pass over the tape of one forward."""

    def __init__(self, net, tape: dict, names: List[str]):
        self.net, self.tape = net, tape
        self.ar = net._train_arena
        self.b = tape["trunk"]["h_in"].shape[0]
        self.dev = tape["trunk"]["h_in"].device
        self.grads: Dict[str, Optional[torch.Tensor]] = {}      # parameter / row name -> gradient (None: already in .grad)
        self.params = dict(net.trunk_parameters())
        # ONE double [B][total][2] table holds every per-channel reduction of the pass (gradient channel sums =
        # bias / conditioning-row gradients, GroupNorm (sum du, sum du*xhat)); converted with two torch ops at the end.
        self.tab_channels = 40 * sum(net.chs) + 512
        self.tab = self.ar.get(f"gtab.{self.b}", (self.b, self.tab_channels, 2), torch.float64, self.dev)
        self.tab.zero_()
        self._c_off = 0
        self._rows: List[tuple] = []       # (grad name, c0, channels)
        self._gns: List[tuple] = []        # (gn name, c0, channels)

    # ---- helpers ------------------------------------------------------------------------------------------
    def chan(self, c: int) -> int:
        """Reserve c channels of the reduction table; returns the first channel."""
        c0 = self._c_off
        self._c_off += c
        if self._c_off > self.tab_channels:
            raise RuntimeError("gradient reduction table too small")
        return c0

    def buf(self, name: str, ch: int, grid) -> torch.Tensor:
        return self.ar.get(f"g.{name}.{self.b}x{grid[0]}", (self.b, ch // 8) + tuple(grid) + (8,), torch.bfloat16, self.dev)

    def pad(self, g, g_plane0, g_ch):
        """Periodic one-voxel halo around a gradient window (circular convs only): the dgrad of a circular conv is a
        circular conv of the padded gradient, and the narrow-layer wgrad reads w-shifted gradient tiles."""
        d, h, w = g.shape[2:5]
        gp = self.ar.get(f"g.pad.{g_ch}.{self.b}x{d}", (self.b, g_ch // 8, d + 2, h + 2, w + 2, 8), torch.bfloat16, self.dev)
        return ops.pad_circular(g, g_ch, x_plane0=g_plane0, out=gp)

    def dgrad(self, name: str, conv, g, g_plane0, g_ch, out, out_plane0=0, g_pad=None):
        """out[window] = conv^T(g): one launch per <=256 input channels of the conv."""
        ci = conv.in_channels
        taps = ops.TAPS_3X3X3 if conv.kernel_size[0] == 3 else ops.TAPS_1X1X1
        circ = self.net.circular and conv.kernel_size[0] == 3
        if circ:
            g, g_plane0 = (g_pad if g_pad is not None else self.pad(g, g_plane0, g_ch)), 0
        ops.set_profile_tag("dgrad ")
        # a 3x3x3 dgrad with <= 32 gradient channels runs on the kd-folded schedule when its N is <= 32: three
        # 32-wide launches beat one N = 96 launch on the generic schedule (r01r: 0.94 ms vs 3 x 0.21 ms)
        limit = 32 if (conv.kernel_size[0] == 3 and g_ch in (16, 32) and ci > 32 and ci % 32 == 0) else 256
        for c0, n in _chunks(ci, limit):
            wp = self.net._packed_dgrad(name, conv, c0, n)
            ops.conv3d(g, wp, n, taps=taps, x_plane0=g_plane0, c_in=g_ch, out=out, out_plane0=out_plane0 + c0 // 8,
                       circular=circ)
        ops.set_profile_tag("")

    def wgrad(self, name: str, conv, a, a_plane0, a_ch, g, g_plane0, g_pad=None):
        """Filter gradient, accumulated by the kernel straight into ``weight.grad`` when it exists (the Trainer's
        flat gradient bucket), else into a fresh tensor handed back to autograd."""
        k = conv.kernel_size[0]
        w = self.params[name + ".weight"]
        if w.grad is not None and w.grad.is_contiguous() and w.grad.dtype == torch.float32:
            target, ret = w.grad, None
        else:
            target = ret = torch.zeros_like(w, memory_format=torch.contiguous_format)
        circ = self.net.circular and k == 3
        if circ:
            g, g_plane0 = (g_pad if g_pad is not None else self.pad(g, g_plane0, -(-conv.out_channels // 16) * 16)), 0
        ops.conv3d_wgrad(a, g, a_ch, conv.out_channels, k, a_plane0=a_plane0, g_plane0=g_plane0, grad_out=target,
                         a_padded=circ, g_padded=circ)
        self.grads[name + ".weight"] = ret

    def row_grad(self, name: str, c0: int, c: int):
        self._rows.append(("row." + name, c0, c))

    def gn_bwd(self, name: str, gn, x, x_plane0, x_stats, dy, ch, **kw):
        c0 = self.chan(ch)
        self._gns.append((name, c0, ch))
        ops.gn_silu_bwd(x, dy, ch, gn.num_groups, x_stats, gn.weight, gn.bias, gn.eps, x_plane0=x_plane0, sums=self.tab,
                        sums_c0=c0, **kw)

    def finish(self):
        """Turn the reduction table into the row / GroupNorm gradients (views of two small tensors)."""
        per_sample = self.tab[:, :self._c_off, 0].float()                 # [B, total]
        over_batch = self.tab[:, :self._c_off].sum(dim=0).float()         # [total, 2]
        for name, c0, c in self._rows:
            self.grads[name] = per_sample[:, c0:c0 + c]
        for name, c0, c in self._gns:
            self.grads[name + ".weight"] = over_batch[c0:c0 + c, 1]
            self.grads[name + ".bias"] = over_batch[c0:c0 + c, 0]

    # ---- one residual block ---------------------------------------------------------------------------------
    def block(self, name: str, blk, dy, dy_plane0, dy_c0, dx, dx_plane0, dx_c0):
        """Backward of ``CUNet._run_block``: consumes dy[window] (its per-sample channel sums live at channel
        ``dy_c0`` of the reduction table), writes dx[window] (sums at ``dx_c0``), records every parameter gradient."""
        rec = self.tape[name]
        ci, co, grid = blk.ch_in, blk.ch_out, rec["grid"]
        gn1, conv1, gn2, conv2 = blk.net1[0], blk.net1[2], blk.net2[0], blk.net2[3]
        drop = dict(dropout_p=rec["p_drop"], seed=rec["drop_seed"], layer_tag=rec["drop_tag"],
                    seed_step=self.net.drop_counter if rec["p_drop"] > 0.0 else None)
        # net2: conv -> dropout/silu/gn
        dy_pad = self.pad(dy, dy_plane0, co) if self.net.circular else None
        self.wgrad(name + ".net2", conv2, rec["a2"], 0, co, dy, dy_plane0, g_pad=dy_pad)
        self.row_grad(name + ".net2", dy_c0, co)
        d_a2 = self.buf(f"a.{co}", co, grid)
        self.dgrad(name + ".net2", conv2, dy, dy_plane0, co, d_a2, g_pad=dy_pad)
        dh = self.buf(f"h.{co}", co, grid)
        dh_c0 = self.chan(co)
        self.gn_bwd(name + ".gn2", gn2, rec["h"], 0, rec["h_stats"], d_a2, co, out=dh, out_stats=self.tab,
                    out_stats_c0=dh_c0, **drop)
        # net1: conv (+ conditioning row) -> silu/gn
        dh_pad = self.pad(dh, 0, co) if self.net.circular else None
        self.wgrad(name + ".net1", conv1, rec["a1"], 0, ci, dh, 0, g_pad=dh_pad)
        self.row_grad(name + ".net1", dh_c0, co)
        d_a1 = self.buf(f"a.{ci}", ci, grid)
        self.dgrad(name + ".net1", conv1, dh, 0, co, d_a1, g_pad=dh_pad)
        # skip path
        if blk.skip_conv is None:
            add, add_plane0 = dy, dy_plane0
        else:
            self.wgrad(name + ".skip", blk.skip_conv, rec["x"], rec["x_plane0"], ci, dy, dy_plane0)
            self.row_grad(name + ".skip", dy_c0, co)
            add, add_plane0 = self.buf(f"s.{ci}", ci, grid), 0
            self.dgrad(name + ".skip", blk.skip_conv, dy, dy_plane0, co, add)
        self.gn_bwd(name + ".gn1", gn1, rec["x"], rec["x_plane0"], rec["x_stats"], d_a1, ci, add=add, add_plane0=add_plane0,
                    out=dx, out_plane0=dx_plane0, out_stats=self.tab, out_stats_c0=dx_c0)

    # ---- the whole trunk ---------------------------------------------------------------------------------------
    def run(self, d_out: torch.Tensor, need_dx: bool) -> Optional[torch.Tensor]:
        net, tr = self.net, self.tape["trunk"]
        c, nl, grids, b = net.chs, len(net.chs), tr["grids"], self.b
        # conv_out: fp32 (B,1,D,H,W) gradient -> channel 0 of a 16-channel planar tensor
        g_out = self.ar.get(f"g.out.{b}", (b, 2) + tuple(grids[0]) + (8,), torch.bfloat16, self.dev)
        ops.pack_input(d_out.contiguous().float(), None, 16, out=g_out)
        conv_out, gn_out = net.conv_out[2], net.conv_out[0]
        g_out_pad = self.pad(g_out, 0, 16) if net.circular else None
        self.wgrad("conv_out", conv_out, tr["out_a"], 0, c[0], g_out, 0, g_pad=g_out_pad)
        self.grads["row.conv_out"] = d_out.reshape(b, -1).sum(dim=1, keepdim=True).float()
        d_a = self.buf(f"a.{c[0]}", c[0], grids[0])
        self.dgrad("conv_out", conv_out, g_out, 0, 16, d_a, g_pad=g_out_pad)
        dy = self.buf(f"y.{c[0]}", c[0], grids[0])
        dy_c0 = self.chan(c[0])
        self.gn_bwd("conv_out.gn", gn_out, tr["out_x"], 0, tr["out_x_stats"], d_a, c[0], out=dy, out_stats=self.tab,
                    out_stats_c0=dy_c0)
        # up path, finest level first (reverse execution order)
        d_cats = {}
        for k, i in reversed(list(enumerate(reversed(range(nl - 1))))):
            name = f"ups.{k}.resnet_blocks.0"
            cc = c[i + 1] + c[i]
            d_cat = self.buf(f"cat{i}", cc, grids[i])
            self.block(name, net.ups[k].resnet_blocks[0], dy, 0, dy_c0, d_cat, 0, self.chan(cc))
            d_cats[i] = d_cat
            # gradient of the up-sampled half goes down one level
            dy = self.buf(f"y.{c[i + 1]}", c[i + 1], grids[i + 1])
            dy_c0 = self.chan(c[i + 1])
            ops.upsample2_bwd(d_cat, c[i + 1], dy_plane0=0, out=dy, stats=self.tab, stats_c0=dy_c0)
        # bottom: mid2, mid1, last down block
        for name, blk in (("mid2", net.mid2), ("mid1", net.mid1),
                          (f"downs.{nl - 1}.resnet_blocks.0", net.downs[nl - 1].resnet_blocks[0])):
            ci = blk.ch_in
            dx = self.buf(f"x.{name}", ci, grids[nl - 1])
            dx_c0 = self.chan(ci)
            self.block(name, blk, dy, 0, dy_c0, dx, 0, dx_c0)
            dy, dy_c0 = dx, dx_c0
        # down path: d(block output) = skip half of d_cat + avg-pool backward of the coarser gradient
        for i in reversed(range(nl - 1)):
            name = f"downs.{i}.resnet_blocks.0"
            blk = net.downs[i].resnet_blocks[0]
            d_cat, p0 = d_cats[i], c[i + 1] // 8
            tot_c0 = self.chan(c[i])
            ops.avgpool2_bwd(dy, c[i], d_cat, dx_plane0=p0, accumulate=True, stats=self.tab, stats_c0=tot_c0)
            ci = blk.ch_in
            dx = self.buf(f"x.{name}", ci, grids[i])
            dx_c0 = self.chan(ci)
            self.block(name, blk, d_cat, p0, tot_c0, dx, 0, dx_c0)
            dy, dy_c0 = dx, dx_c0
        # conv_in
        dy_pad = self.pad(dy, 0, c[0]) if net.circular else None
        self.wgrad("conv_in", net.conv_in, tr["packed"], 0, 16, dy, 0, g_pad=dy_pad)
        self.row_grad("conv_in", dy_c0, c[0])
        self.finish()
        if not need_dx:
            return None
        wp = net._packed_dgrad("conv_in", net.conv_in, 0, 1)
        dz = torch.empty((b, 1) + tuple(grids[0]), dtype=torch.float32, device=self.dev)
        if net.circular:
            dy = dy_pad
        ops.set_profile_tag("dgrad ")
        ops.conv3d(dy, wp, 1, out=dz, out_fp32=True, circular=net.circular)
        ops.set_profile_tag("")
        return dz


class _UNetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, s_conditioning, row_names, param_names, x, *tensors):
        b = x.shape[0]
        rows = dict(zip(row_names, tensors[:len(row_names)]))
        rows = {k: v.detach().contiguous() for k, v in rows.items()}
        cond = None if s_conditioning is None else s_conditioning.detach().contiguous().float()
        ar = net._train_arena
        packed = ops.pack_input(x.detach().contiguous().float(), cond, 16,
                                out=ar.get(f"packed.{b}", (b, 2) + tuple(net.shape[1:]) + (8,), torch.bfloat16, x.device))
        tape: dict = {}
        net.refresh_packed(training=True)
        out = net.run_packed(packed, rows, training_dropout=net.training and net.dropout_prob > 0.0, tape=tape)
        ctx.net, ctx.tape, ctx.row_names, ctx.param_names = net, tape, row_names, param_names
        ctx.need_dx = x.requires_grad
        return out

    @staticmethod
    def backward(ctx, d_out):
        net = ctx.net
        bw = _Backward(net, ctx.tape, ctx.row_names)
        dz = bw.run(d_out, ctx.need_dx)
        g = bw.grads
        out = [None, None, None, None, dz]
        out += [g["row." + n] for n in ctx.row_names]
        out += [g[n] for n in ctx.param_names]
        ctx.tape = None
        return tuple(out)


def unet_forward(net, x, t=None, s_conditioning=None, v_conditionings=None):
    """``CUNet.forward`` with gradients: eps_hat / v_hat (B, 1, D, H, W) fp32, differentiable w.r.t. every
    parameter of ``net`` and w.r.t. ``x``."""
    b = x.shape[0]
    rows = net.chan_add_rows(b, t, v_conditionings, x.device)       # torch autograd: biases + embedding MLPs
    row_names = list(rows.keys())
    params = net.trunk_parameters()
    param_names = [n for n, _ in params]
    if net.training and net.dropout_prob > 0.0:
        ops.increment(net.drop_counter)          # new dropout masks every training forward (device counter: graph-safe)
    net.dropout_seed = int(getattr(net, "dropout_base_seed", 0)) << 32
    return _UNetFn.apply(net, s_conditioning, row_names, param_names, x, *[rows[n] for n in row_names],
                         *[p for _, p in params])
