"""GPU parity of the training kernels (wgrad, dgrad, GroupNorm/SiLU/pool/upsample backward, AdamW)
against torch autograd on the same inputs.

Integer-valued inputs make the conv gradients exact in fp32 (bit-exact comparison); the elementwise
backward kernels are compared with fp32 autograd of the same bf16-rounded inputs at bf16 output tolerance.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _ops():
    from vdm4cdm_b200 import ops
    return ops


def _int_tensor(shape, lo, hi, gen, device):
    return torch.randint(lo, hi + 1, shape, generator=gen, device="cpu").float().to(device)


WGRAD_CASES = [
    # B, Cin, Cout, D, H, W, k
    (1, 32, 32, 4, 16, 8, 3),
    (2, 32, 32, 6, 20, 12, 3),      # ragged grid, several tiles per CTA
    (1, 16, 32, 5, 16, 16, 3),      # conv_in shape (S = 8 slices folded into M)
    (1, 64, 64, 4, 16, 16, 3),
    (1, 96, 32, 4, 16, 16, 3),      # concat input: 3 channel blocks of 32
    (1, 128, 128, 3, 16, 8, 3),
    (1, 256, 256, 2, 16, 8, 3),     # n split over two CTAs
    (1, 384, 128, 2, 16, 8, 3),
    (2, 32, 1, 4, 16, 16, 3),       # conv_out: one real output channel in a 16-channel window
    (1, 96, 32, 4, 16, 16, 1),      # 1x1x1 skip conv
    (1, 32, 64, 3, 9, 7, 1),
]


@pytest.mark.parametrize("case", WGRAD_CASES, ids=lambda c: "x".join(map(str, c)))
def test_wgrad_exact_integers(case):
    ops = _ops()
    b, ci, co, d, h, w, k = case
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(4321 + ci + co)
    a = _int_tensor((b, ci, d, h, w), -2, 2, gen, dev)
    g = _int_tensor((b, co, d, h, w), -2, 2, gen, dev)
    wt = torch.zeros((co, ci, k, k, k), device=dev, dtype=torch.float64, requires_grad=True)
    F.conv3d(a.double(), wt, padding=k // 2).backward(g.double())
    ref = wt.grad.round().float()
    dw = ops.conv3d_wgrad(ops.to_planar(a, 16), ops.to_planar(g, 16), ci, co, k)
    torch.cuda.synchronize()
    got = ops.wgrad_to_torch(dw, k)
    bad = (got != ref).sum().item()
    assert bad == 0, f"{bad} of {ref.numel()} differ; max |diff| = {(got - ref).abs().max().item()}"


def test_wgrad_plane_windows_and_accumulation():
    ops = _ops()
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(8)
    b, ci, co, d, h, w = 2, 32, 32, 4, 16, 16
    a = _int_tensor((b, ci, d, h, w), -2, 2, gen, dev)
    g = _int_tensor((b, co, d, h, w), -2, 2, gen, dev)
    abuf = torch.zeros((b, 7, d, h, w, 8), dtype=torch.bfloat16, device=dev)
    abuf[:, 2:6] = ops.to_planar(a)
    gbuf = torch.zeros((b, 6, d, h, w, 8), dtype=torch.bfloat16, device=dev)
    gbuf[:, 1:5] = ops.to_planar(g)
    wt = torch.zeros((co, ci, 3, 3, 3), device=dev, dtype=torch.float64, requires_grad=True)
    F.conv3d(a.double(), wt, padding=1).backward(g.double())
    ref = wt.grad.round().float()
    dw = ops.conv3d_wgrad(abuf, gbuf, ci, co, 3, a_plane0=2, g_plane0=1)
    ops.conv3d_wgrad(abuf, gbuf, ci, co, 3, a_plane0=2, g_plane0=1, out=dw)      # second micro-batch accumulates
    torch.cuda.synchronize()
    assert torch.equal(ops.wgrad_to_torch(dw, 3), 2 * ref)


def test_wgrad_accumulates_into_a_torch_layout_gradient():
    """The Trainer's path: the kernel adds straight into weight.grad (c_out, c_in_real, k, k, k) inside a flat bucket."""
    ops = _ops()
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(9)
    b, ci_real, ci, co, d, h, w = 2, 2, 16, 32, 4, 16, 16             # conv_in: 2 real channels in a 16-channel tensor
    a = _int_tensor((b, ci_real, d, h, w), -2, 2, gen, dev)
    g = _int_tensor((b, co, d, h, w), -2, 2, gen, dev)
    wt = torch.zeros((co, ci_real, 3, 3, 3), device=dev, dtype=torch.float64, requires_grad=True)
    F.conv3d(a.double(), wt, padding=1).backward(g.double())
    flat = torch.full((co * ci_real * 27 + 8,), 1.0, device=dev)
    grad = flat[4:4 + co * ci_real * 27].view(co, ci_real, 3, 3, 3)
    ops.conv3d_wgrad(ops.to_planar(a, 16), ops.to_planar(g, 16), ci, co, 3, grad_out=grad)
    torch.cuda.synchronize()
    assert torch.equal(grad, wt.grad.round().float() + 1.0)
    assert (flat[:4] == 1).all() and (flat[-4:] == 1).all()


@pytest.mark.parametrize("co,ci,k", [(32, 2, 3), (1, 32, 3), (64, 32, 3), (128, 384, 1), (32, 96, 3)])
def test_pack_conv_weight_kernel_matches_host_packing(co, ci, k):
    ops = _ops()
    dev = torch.device("cuda:0")
    w = torch.randn((co, ci, k, k, k), generator=torch.Generator().manual_seed(co + ci)).to(dev)
    out = torch.empty(ops.packed_weight_shape(w.shape), dtype=torch.bfloat16, device=dev)
    ops.pack_conv_weight_into(w, out)
    assert torch.equal(out, ops.pack_conv_weight(w))
    for c0, n in ((0, ci),) if ci <= 256 else ((0, ci // 2), (ci // 2, ci // 2)):
        outd = torch.empty(ops.packed_weight_shape(w.shape, True, n), dtype=torch.bfloat16, device=dev)
        ops.pack_conv_weight_into(w, outd, True, c0, n)
        assert torch.equal(outd, ops.pack_conv_weight(w[:, c0:c0 + n], transpose_flip=True))
    torch.cuda.synchronize()


def test_batched_pack_equals_the_single_filter_launches():
    """vdm_pack_conv_weight_batched: every filter of a job table (forward and dgrad variants, 3x3x3 and 1x1x1) in one
    launch gives bit for bit what the per-filter launches give; CUNet.repack_all re-packs exactly the stale filters."""
    ops = _ops()
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(11)
    jobs, want = [], []
    for co, ci, k in ((32, 2, 3), (1, 32, 3), (64, 32, 3), (128, 384, 1), (32, 96, 3), (256, 256, 3)):
        w = torch.randn((co, ci, k, k, k), generator=gen).to(dev)
        variants = [(False, 0, ci)] + ([(True, 0, ci)] if ci <= 256 else [(True, 0, ci // 2), (True, ci // 2, ci // 2)])
        for tf, c0, n in variants:
            out = torch.zeros(ops.packed_weight_shape(w.shape, tf, n), dtype=torch.bfloat16, device=dev)
            ref = torch.empty_like(out)
            ops.pack_conv_weight_into(w, ref, tf, c0, n)
            jobs.append((w, out, tf, c0, n))
            want.append(ref)
    table = ops.pack_job_table(jobs, dev)
    ops.pack_conv_weights_batched(table, len(jobs))
    torch.cuda.synchronize()
    for (w, out, tf, c0, n), ref in zip(jobs, want):
        assert torch.equal(out, ref), (tuple(w.shape), tf, c0, n)

    from vdm4cdm_b200.networks import CUNet
    net = CUNet(shape=(1, 16, 16, 16), chs=[16, 32], s_conditioning_channels=1, v_conditioning_dims=[], t_conditioning=True).to(dev)
    net.refresh_packed()
    before = {slot: f.buf.clone() for slot, f in net._packed_cache.items()}
    with torch.no_grad():
        for p_ in net.parameters():
            p_.mul_(1.5)
    net.invalidate_packed()
    launches0 = ops.launch_count()
    net.repack_all()
    assert ops.launch_count() - launches0 == 1
    torch.cuda.synchronize()
    for name, conv in net._convs():
        assert torch.equal(net._packed_cache[name].buf, ops.pack_conv_weight(conv.weight.detach()))
        assert not torch.equal(net._packed_cache[name].buf, before[name])


def test_dgrad_wide_input_in_two_launches():
    """dgrad of a 384 -> 128 conv: 384 output channels exceed one launch (N <= 256) -> two plane windows."""
    ops = _ops()
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(6)
    b, ci, co, d, h, w = 1, 384, 128, 2, 16, 8
    wt = _int_tensor((co, ci, 3, 3, 3), -1, 1, gen, dev)
    dy = _int_tensor((b, co, d, h, w), -1, 1, gen, dev)
    x = torch.zeros((b, ci, d, h, w), device=dev, requires_grad=True)
    F.conv3d(x, wt, padding=1).backward(dy)
    ref = x.grad.to(torch.bfloat16).float()
    out = torch.empty((b, ci // 8, d, h, w, 8), dtype=torch.bfloat16, device=dev)
    dyp = ops.to_planar(dy)
    for c0 in (0, 192):
        wp = ops.pack_conv_weight(wt[:, c0:c0 + 192], transpose_flip=True)
        ops.conv3d(dyp, wp, 192, out=out, out_plane0=c0 // 8)
    torch.cuda.synchronize()
    assert torch.equal(ops.from_planar(out, ci), ref)


@pytest.mark.parametrize("shape,groups,p", [((2, 32, 6, 10, 14), 8, 0.0), ((1, 96, 4, 8, 8), 8, 0.0),
                                            ((2, 16, 4, 6, 6), 8, 0.0), ((2, 64, 4, 8, 8), 8, 0.1)])
def test_gn_silu_backward_matches_autograd(shape, groups, p):
    ops = _ops()
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(12)
    c = shape[1]
    x = (torch.randn(shape, generator=gen) * 1.7 + 0.3).to(dev)
    dy = torch.randn(shape, generator=gen).to(dev)
    add = torch.randn(shape, generator=gen).to(dev)
    gamma = (torch.rand(c, generator=gen) + 0.5).to(dev)
    beta = (torch.randn(c, generator=gen) * 0.2).to(dev)
    xp, dyp, addp = ops.to_planar(x), ops.to_planar(dy), ops.to_planar(add)
    xr, dyr, addr = ops.from_planar(xp), ops.from_planar(dyp), ops.from_planar(addp)
    st = ops.channel_stats(xp, c)
    # forward with the same dropout mask the backward regenerates
    y0 = ops.from_planar(ops.gn_silu(xp, c, groups, st, gamma, beta))
    y1 = ops.from_planar(ops.gn_silu(xp, c, groups, st, gamma, beta, dropout_p=p, seed=9, layer_tag=2))
    mask = torch.ones_like(y0) if p == 0.0 else ((y1 != 0) | (y0 == 0)).float() / (1.0 - p)
    xa = xr.clone().requires_grad_(True)
    ga, ba = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    (F.silu(F.group_norm(xa, groups, ga, ba, 1e-5)) * mask).backward(dyr)
    out_stats = torch.zeros((shape[0], c, 2), dtype=torch.float64, device=dev)
    dx, sums = ops.gn_silu_bwd(xp, dyp, c, groups, st, gamma, beta, 1e-5, add=addp, dropout_p=p, seed=9, layer_tag=2,
                               out_stats=out_stats)
    torch.cuda.synchronize()
    got = ops.from_planar(dx)
    want = xa.grad + addr
    scale = want.abs().max().item()
    assert (got - want).abs().max().item() < 2 ** -7 * scale, (got - want).abs().max().item() / scale
    assert torch.allclose(sums[..., 0].sum(0).float(), ba.grad, rtol=2e-3, atol=2e-3 * ba.grad.abs().max().item())
    assert torch.allclose(sums[..., 1].sum(0).float(), ga.grad, rtol=2e-3, atol=2e-3 * ga.grad.abs().max().item())
    assert torch.allclose(out_stats[..., 0], got.double().sum(dim=(2, 3, 4)), rtol=1e-5, atol=1e-3)


def test_pool_and_upsample_backward():
    ops = _ops()
    dev = torch.device("cuda:0")
    b, c, d, h, w = 2, 32, 4, 8, 12
    gen = torch.Generator().manual_seed(14)
    g_coarse = torch.randn((b, c, d // 2, h // 2, w // 2), generator=gen).to(dev)
    g_fine = torch.randn((b, c, d, h, w), generator=gen).to(dev)
    gcp, gfp = ops.to_planar(g_coarse), ops.to_planar(g_fine)
    gcr, gfr = ops.from_planar(gcp), ops.from_planar(gfp)
    # avg-pool backward, accumulated on top of an existing gradient inside a plane window of a wider buffer
    buf = torch.zeros((b, 6, d, h, w, 8), dtype=torch.bfloat16, device=dev)
    buf[:, 1:5] = gfp
    st = torch.zeros((b, 48, 2), dtype=torch.float64, device=dev)
    ops.avgpool2_bwd(gcp, c, buf, dx_plane0=1, accumulate=True, stats=st, stats_c0=8)
    torch.cuda.synchronize()
    want = (gfr + F.interpolate(gcr, scale_factor=2, mode="nearest") / 8).to(torch.bfloat16).float()
    got = ops.from_planar(buf[:, 1:5].contiguous())
    assert torch.equal(got, want)
    assert buf[:, 0].float().abs().sum().item() == 0 and buf[:, 5].float().abs().sum().item() == 0
    assert torch.allclose(st[:, 8:40, 0], got.double().sum(dim=(2, 3, 4)), rtol=1e-5, atol=1e-3)
    fresh = torch.full((b, 4, d, h, w, 8), 5.0, dtype=torch.bfloat16, device=dev)
    ops.avgpool2_bwd(gcp, c, fresh)
    assert torch.equal(ops.from_planar(fresh), (F.interpolate(gcr, scale_factor=2, mode="nearest") / 8).to(torch.bfloat16).float())
    # nearest-upsample backward = 8 * avg-pool of the fine gradient
    dc = ops.upsample2_bwd(gfp, c)
    torch.cuda.synchronize()
    assert torch.allclose(ops.from_planar(dc), (F.avg_pool3d(gfr, 2) * 8).to(torch.bfloat16).float(), rtol=2 ** -7, atol=1e-6)


def test_adamw_and_sumsq_match_torch():
    ops = _ops()
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(15)
    n = 100003
    p0 = torch.randn(n, generator=gen).to(dev)
    grads = [torch.randn(n, generator=gen).to(dev) * s for s in (1.0, 0.01, 3.0)]
    ref = p0.clone().requires_grad_(True)
    opt = torch.optim.AdamW([ref], lr=3e-4)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    for step, g in enumerate(grads, 1):
        ref.grad = g.clone()
        torch.nn.utils.clip_grad_norm_([ref], 0.5)
        opt.step()
        ss = ops.sumsq(g)
        torch.cuda.synchronize()
        assert abs(ss.item() - g.double().pow(2).sum().item()) < 1e-6 * ss.item()
        ops.adamw_step(p, g, m, v, lr=3e-4, step=step, grad_sumsq=ss, max_norm=0.5)
    torch.cuda.synchronize()
    assert torch.allclose(p, ref.detach(), rtol=1e-5, atol=1e-6), (p - ref.detach()).abs().max()
