"""TF32 inference mode (CUNet(precision="tf32")): fp32 channel-planar activations and tcgen05 kind::tf32 convs.

Integer inputs (|x| <= 8, |w| <= 4) are exact TF32 operands and their sums are exact in fp32, so the convs must reproduce
fp64 F.conv3d bit for bit; on normal inputs a conv must stay within 2e-3 relative L2 of fp64, and the whole network
within 5e-3 of the fp32 CPU oracle and at most half the error of the bf16 path on the same input."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.dirname(__file__))

CONV_RTOL = 2e-3
NET_RTOL = 5e-3


def _rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


def _ref_conv(x, w, k, circular):
    """fp64 reference conv of (B, C, D, H, W) x with torch weight w."""
    if k == 1:
        return F.conv3d(x, w)
    if circular:
        return F.conv3d(F.pad(x, (1, 1, 1, 1, 1, 1), mode="circular"), w)
    return F.conv3d(x, w, padding=1)


def _run_conv(xd, wd, *, k, circular, x_extra=0, x_plane0=0, y_extra=0, y_plane0=0, out_fp32=False,
              bias=None, residual=None, stats=False):
    """vdm_conv3d_tf32 of fp64 (B, Ci, D, H, W) x; returns (y fp64 (B, Co, D, H, W), stats or None)."""
    from vdm4cdm_b200 import ops
    b, ci = xd.shape[:2]
    co = wd.shape[0]
    dev = "cuda"
    taps = ops.TAPS_3X3X3 if k == 3 else ops.TAPS_1X1X1
    xp = ops.to_planar(xd.float(), 8, dtype=torch.float32)
    if x_extra:                                    # x read from a plane window of a wider buffer
        buf = torch.randn((b, xp.shape[1] + x_extra) + tuple(xp.shape[2:]), dtype=torch.float32)
        buf[:, x_plane0:x_plane0 + xp.shape[1]] = xp
        xp = buf
    xp = xp.cuda()
    if circular:
        xp = ops.pad_circular(xp, ci, x_plane0=x_plane0)
        x_plane0 = 0
    wp = torch.empty(ops.packed_weight_shape(wd.shape, dtype=torch.float32), dtype=torch.float32, device=dev)
    ops.pack_conv_weight_into(wd.float().cuda().contiguous(), wp)
    kw = dict(taps=taps, x_plane0=x_plane0, c_in=ci, circular=circular)
    step = None
    if bias is not None:
        step = torch.tensor([1], dtype=torch.int32, device=dev)
        kw.update(chan_add=bias.float().cuda().contiguous(), step_ptr=step)
    st = None
    if stats:
        st = torch.zeros((b, co + 8, 2), dtype=torch.float64, device=dev)
        kw.update(stats=st, stats_c0=8)
    grid = tuple(xd.shape[2:])
    if out_fp32:
        y = ops.conv3d(xp, wp, co, out_fp32=True, **kw)
        return y.double().cpu(), None
    if residual is not None:
        kw.update(residual=ops.to_planar(residual.float(), 8, dtype=torch.float32).cuda())
    out = torch.full((b, co // 4 + y_extra) + grid + (4,), float("nan"), dtype=torch.float32, device=dev)
    ops.conv3d(xp, wp, co, out=out, out_plane0=y_plane0, **kw)
    if y_extra:
        keep = torch.ones(out.shape[1], dtype=torch.bool)
        keep[y_plane0:y_plane0 + co // 4] = False
        assert torch.isnan(out[:, keep]).all(), "planes outside the output window were written"
    y = ops.from_planar(out[:, y_plane0:y_plane0 + co // 4].contiguous()).double().cpu()
    return y, (None if st is None else st[:, 8:].cpu())


CASES = [  # (c_in, c_out, grid, batch, k, circular, x window (extra, plane0), y window (extra, plane0), out_fp32)
    (16, 32, (12, 20, 24), 2, 3, False, (0, 0), (0, 0), False),
    (32, 32, (16, 16, 16), 2, 3, False, (0, 0), (0, 0), False),
    (64, 64, (16, 16, 16), 1, 3, False, (6, 4), (4, 2), False),
    (96, 32, (16, 16, 16), 2, 3, False, (8, 8), (0, 0), False),    # a concat window of a 128-channel buffer
    (128, 256, (8, 8, 8), 1, 3, False, (0, 0), (0, 0), False),     # few tiles: the planner splits N over CTAs
    (256, 256, (16, 16, 16), 1, 3, False, (0, 0), (0, 0), False),
    (64, 32, (16, 16, 16), 2, 1, False, (0, 0), (0, 0), False),
    (32, 1, (16, 16, 16), 2, 3, False, (0, 0), (0, 0), True),
    (32, 32, (16, 16, 16), 2, 3, True, (0, 0), (0, 0), False),
]


@pytest.mark.parametrize("ci,co,grid,b,k,circ,xw,yw,out_fp32", CASES)
def test_tf32_conv_bit_exact_on_integers(ci, co, grid, b, k, circ, xw, yw, out_fp32):
    g = torch.Generator().manual_seed(ci * 1000 + co)
    x = torch.randint(-8, 9, (b, ci) + grid, generator=g).double()
    w = torch.randint(-4, 5, (co, ci, k, k, k), generator=g).double()
    bias = torch.randint(-50, 51, (3, b, co), generator=g).double()      # row block 1 is selected through step_ptr
    want = _ref_conv(x, w, k, circ) + bias[1][:, :, None, None, None]
    res = None
    if not out_fp32:
        res = torch.randint(-100, 101, (b, co) + grid, generator=g).double()
        want = want + res
    got, st = _run_conv(x, w, k=k, circular=circ, x_extra=xw[0], x_plane0=xw[1], y_extra=yw[0], y_plane0=yw[1],
                        out_fp32=out_fp32, bias=bias, residual=res, stats=not out_fp32)
    assert torch.equal(got, want), (got - want).abs().max().item()
    if st is not None:
        # the statistics are of the stored fp32 values, accumulated as fp32 per tile and fp64 across tiles: exact up to the
        # fp32 partial sums of these large integers
        s1 = want.sum(dim=(2, 3, 4))
        s2 = (want * want).sum(dim=(2, 3, 4))
        scale = want.abs().sum(dim=(2, 3, 4))
        assert ((st[..., 0] - s1).abs() <= 1e-6 * scale).all(), ((st[..., 0] - s1).abs() / scale).max().item()
        assert ((st[..., 1] - s2).abs() <= 1e-6 * s2).all(), ((st[..., 1] - s2).abs() / s2).max().item()


@pytest.mark.parametrize("ci,co,grid,b,k,circ,xw,yw,out_fp32", CASES)
def test_tf32_conv_normal_inputs(ci, co, grid, b, k, circ, xw, yw, out_fp32):
    g = torch.Generator().manual_seed(ci + co)
    x = torch.randn((b, ci) + grid, generator=g).double()
    w = (torch.randn((co, ci, k, k, k), generator=g) / (ci * k ** 3) ** 0.5).double()
    want = _ref_conv(x, w, k, circ)
    got, _ = _run_conv(x, w, k=k, circular=circ, x_extra=xw[0], x_plane0=xw[1], y_extra=yw[0], y_plane0=yw[1],
                       out_fp32=out_fp32)
    err = _rel_l2(got, want)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = True
    try:
        cudnn = _ref_conv(x.float().cuda(), w.float().cuda(), k, circ).double().cpu()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    print(f"tf32 conv {ci}->{co} k={k} {grid}: relative L2 {err:.3e} (cuDNN TF32 on the same inputs: {_rel_l2(cudnn, want):.3e})")
    assert err <= CONV_RTOL, err


def test_tf32_elementwise_kernels():
    from vdm4cdm_b200 import ops
    g = torch.Generator().manual_seed(5)
    b, c, grid = 2, 32, (8, 12, 16)
    x = torch.randn((b, c) + grid, generator=g).double()
    xp = ops.to_planar(x.float(), 8, dtype=torch.float32).cuda()
    xf = ops.from_planar(xp.cpu()).double()                       # == x rounded to fp32
    # gn_silu (exp-based SiLU)
    stats = torch.stack([xf.sum(dim=(2, 3, 4)), (xf * xf).sum(dim=(2, 3, 4))], dim=-1).contiguous()
    gamma, beta = torch.randn(c, generator=g), torch.randn(c, generator=g)
    y = ops.gn_silu(xp, c, 8, stats.cuda(), gamma.cuda(), beta.cuda(), 1e-5)
    want = F.silu(F.group_norm(xf, 8, gamma.double(), beta.double(), 1e-5))
    assert y.dtype == torch.float32 and _rel_l2(ops.from_planar(y.cpu()), want) <= 1e-6
    # avgpool2 with statistics
    st = torch.zeros((b, c, 2), dtype=torch.float64, device="cuda")
    p = ops.avgpool2(xp, c, stats=st)
    want = F.avg_pool3d(xf, 2)
    assert _rel_l2(ops.from_planar(p.cpu()), want) <= 1e-6
    assert torch.allclose(st.cpu()[..., 0], want.sum(dim=(2, 3, 4)), rtol=1e-6, atol=1e-5)
    assert torch.allclose(st.cpu()[..., 1], (want * want).sum(dim=(2, 3, 4)), rtol=1e-6)
    # upsample2 into a plane window of a concat buffer, with statistics
    cat = torch.zeros((b, 3 * c // 4) + grid + (4,), dtype=torch.float32, device="cuda")
    st = torch.zeros((b, 3 * c, 2), dtype=torch.float64, device="cuda")
    ops.upsample2(p, c, cat, out_plane0=c // 4, stats=st, stats_c0=c)
    want = F.interpolate(ops.from_planar(p.cpu()).double(), scale_factor=2, mode="nearest")
    assert torch.equal(ops.from_planar(cat[:, c // 4:c // 2].contiguous().cpu()).double(), want)
    assert (cat[:, :c // 4] == 0).all() and (cat[:, c // 2:] == 0).all()
    assert torch.allclose(st.cpu()[:, c:2 * c, 0], want.sum(dim=(2, 3, 4)), rtol=1e-6, atol=1e-5)
    # periodic halo of an fp32 planar tensor
    pad = ops.pad_circular(xp, c)
    assert torch.equal(ops.from_planar(pad.cpu()).double(), F.pad(xf, (1, 1, 1, 1, 1, 1), mode="circular"))
    # packed network input: (z, cond_1..cond_n, 0...) in planes 0, 1
    z = torch.randn((b, 1) + grid, generator=g)
    cond = torch.randn((b, 3) + grid, generator=g)
    pk = ops.pack_input(z.cuda(), cond.cuda(), 8, dtype=torch.float32)
    assert pk.shape == (b, 2) + grid + (4,)
    want = torch.cat([z, cond, torch.zeros((b, 4) + grid)], dim=1)
    assert torch.equal(ops.from_planar(pk.cpu()), want)


def test_tf32_dtype_mix_is_rejected_before_launch():
    from vdm4cdm_b200 import ops
    x32 = torch.zeros((1, 4, 8, 8, 8, 4), device="cuda")
    x16 = torch.zeros((1, 2, 8, 8, 8, 8), dtype=torch.bfloat16, device="cuda")
    w32 = torch.zeros((27, 4, 16, 4), device="cuda")
    w16 = torch.zeros((27, 2, 16, 8), dtype=torch.bfloat16, device="cuda")
    n0 = ops.launch_count()
    with pytest.raises(ValueError):
        ops.conv3d(x32, w16, 16)
    with pytest.raises(ValueError):
        ops.conv3d(x16, w32, 16)
    with pytest.raises(ValueError):
        ops.conv3d(x32, w32, 16, out=torch.zeros((1, 2, 8, 8, 8, 8), dtype=torch.bfloat16, device="cuda"))
    with pytest.raises(ValueError):
        ops.avgpool2(x32, 16, out=torch.zeros((1, 2, 4, 4, 4, 8), dtype=torch.bfloat16, device="cuda"))
    with pytest.raises(ValueError):
        ops.upsample2(x16, 16, torch.zeros((1, 4, 16, 16, 16, 4), device="cuda"))
    with pytest.raises(ValueError):
        ops.pad_circular(x32, 16, out=torch.zeros((1, 2, 10, 10, 10, 8), dtype=torch.bfloat16, device="cuda"))
    assert ops.launch_count() == n0
    with pytest.raises(ops.UnsupportedFusion):
        ops.conv3d(x32, w32, 16, in_norm=torch.zeros((1, 16, 2), device="cuda"))


def _net_pair(shape, chs, padding="zeros"):
    from test_gpu_unet import _models
    return _models(shape, chs, padding=padding)


NET_CASES = [((1, 32, 32, 32), (16, 32, 64, 128), 2, "zeros"),
             ((1, 16, 32, 48), (32, 64), 1, "zeros"),
             ((1, 24, 24, 24), (16, 32, 64), 3, "zeros"),
             ((1, 80, 80, 80), (16, 32, 64), 1, "zeros"),
             ((1, 56, 56, 56), (32, 64), 1, "zeros"),
             ((1, 32, 32, 32), (16, 32, 64), 2, "circular")]


@pytest.mark.parametrize("shape,chs,batch,padding", NET_CASES)
def test_tf32_unet_forward_matches_oracle(shape, chs, batch, padding):
    ref, net = _net_pair(shape, chs, padding)
    g = torch.Generator().manual_seed(1)
    x = torch.randn((batch,) + shape, generator=g)
    cond = 0.7 * x + 0.3 * torch.randn((batch,) + shape, generator=g)
    t = torch.rand(batch, generator=g)
    v = [torch.rand(batch, 6, generator=g)]
    args = (x.cuda(),)
    kw = dict(t=t.cuda(), s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()])
    with torch.no_grad():
        want = ref(x, t=t, s_conditioning=cond, v_conditionings=v)
        got_bf16 = net(*args, **kw).cpu()
        net.precision = "tf32"
        got = net(*args, **kw).cpu()
        net.precision = "bf16"
        again_bf16 = net(*args, **kw).cpu()
    err, err_bf16 = _rel_l2(got, want), _rel_l2(got_bf16, want)
    print(f"unet {shape} {chs} {padding}: tf32 relative L2 {err:.3e}, bf16 {err_bf16:.3e}")
    assert got.dtype == torch.float32 and got.shape == want.shape
    assert err <= NET_RTOL and err <= 0.5 * err_bf16, (err, err_bf16)
    assert torch.equal(again_bf16, got_bf16) or _rel_l2(again_bf16, got_bf16) < 1e-3    # switching back is harmless


def test_tf32_sampler_step_graph_cfg_and_ddnm():
    from oracle.vdm_ref import VDM as RefVDM
    from vdm4cdm_b200 import utils
    from vdm4cdm_b200.vdm_model import VDM, LightVDM
    shape, chs, b = (1, 16, 16, 16), (16, 32), 2
    ref, net = _net_pair(shape, chs)
    g = torch.Generator().manual_seed(3)
    cond = torch.randn((b,) + shape, generator=g)
    v = [torch.rand(b, 6, generator=g)]
    noises = [torch.randn((b,) + shape, generator=g) for _ in range(8)]
    kw = dict(s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()])
    vdm, ref_vdm = VDM(net).cuda().eval(), RefVDM(ref).eval()
    # one reverse step with injected noise against the oracle, bf16 and tf32 on the same input
    with torch.no_grad():
        want = ref_vdm.sample(b, 1, "cpu", noise_fn=lambda d, s: noises[d], s_conditioning=cond, v_conditionings=v)
    errs = {}
    for prec in ("bf16", "tf32"):
        net.precision = prec
        got = vdm.sample(b, 1, "cuda:0", noise_fn=lambda d, s: noises[d].cuda(), **kw).cpu()
        errs[prec] = _rel_l2(got, want)
    print(f"one reverse step: tf32 relative L2 {errs['tf32']:.3e}, bf16 {errs['bf16']:.3e}")
    assert errs["tf32"] <= NET_RTOL and errs["tf32"] <= 0.5 * errs["bf16"], errs
    # the CUDA-graph replayed chain equals the eager chain bit for bit
    net.precision = "tf32"
    chains = []
    for graph in (False, True):
        vdm.use_cuda_graph = graph
        chains.append(vdm.sample(b, 5, "cuda:0", seed=11, **kw).cpu())
    vdm.use_cuda_graph = True
    assert torch.equal(chains[0], chains[1])
    # classifier-free guidance and DDNM go through CUNet.forward
    cfg = VDM(net, w_cfg=1.5).cuda().eval()
    xs = cfg.sample(b, 2, "cuda:0", seed=3, **kw)
    assert xs.shape == (b,) + shape and torch.isfinite(xs).all()
    mask = (torch.rand((1,) + shape, generator=g) > 0.5).float().cuda()
    y = mask * noises[0].cuda()
    dd = utils.get_ddnm_result(LightVDM(net).cuda().eval(), y, lambda x: mask * x, lambda x: mask * x, n_sampling_steps=3, l=[0, 1, 1], **kw)
    assert dd.shape == (b,) + shape and torch.isfinite(dd).all()
    net.precision = "bf16"
