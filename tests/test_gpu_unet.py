"""GPU parity of the CUNet trunk and the VDM sampler against the CPU oracle (oracle/unet_ref.py,
oracle/vdm_ref.py: plain PyTorch fp32) on identical weights, inputs and injected noise.

Tolerance: the CUDA path keeps activations in bf16 (fp32 accumulation, fp32 latent z); BASELINE.json's
north_star allows 1e-2 relative for bf16.  It is applied to the relative L2 error of the network output
and of one sampler step; multi-step trajectories are compared per step with the oracle re-started
from the CUDA path's z_t (SURVEY.md section 7: errors compound over an ancestral chain)."""
import pytest
import torch

pytestmark = pytest.mark.gpu

BF16_RTOL = 1e-2


def _models(shape, chs, v_dims=(6,), seed=0, padding="zeros"):
    from oracle.unet_ref import CUNet as RefNet
    from vdm4cdm_b200.networks import CUNet
    torch.manual_seed(seed)
    kw = dict(shape=shape, chs=chs, s_conditioning_channels=1, v_conditioning_dims=list(v_dims), t_conditioning=True,
              norm_groups=8, dropout_prob=0.1, conv_padding_mode=padding)
    ref = RefNet(**kw).eval()
    # give biases / norm affines non-trivial values so that every epilogue term is exercised
    with torch.no_grad():
        for n, p in ref.named_parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    net = CUNet(**kw)
    net.load_state_dict(ref.state_dict(), strict=True)
    return ref, net.cuda().eval()


def _rel_l2(a, b):
    return ((a - b).norm() / b.norm()).item()


def _assert_bf16_parity(err, oracle_call, want):
    """err < 1e-2; where a whole random-init network exceeds that (it sits AT the bf16 noise floor: ~30 conv layers x 3
    roundings of 2^-9 each) the bar is the error torch's OWN bf16 autocast of the oracle makes on the same input, never
    looser than 1.5e-2.  (Ragged-tile arithmetic itself is pinned bit-exactly in tests/test_gpu_conv3d.py.)"""
    if err < BF16_RTOL:
        return
    with torch.no_grad(), torch.autocast("cpu", dtype=torch.bfloat16):
        autocast_err = _rel_l2(oracle_call().float(), want)
    print(f"  torch bf16 autocast of the oracle on the same input: {autocast_err:.3e}")
    assert err < min(max(BF16_RTOL, autocast_err), 1.5e-2), (err, autocast_err)


@pytest.mark.parametrize("shape,chs,batch", [((1, 32, 32, 32), (16, 32, 64, 128), 2),
                                             ((1, 16, 32, 48), (32, 64), 1),
                                             ((1, 24, 24, 24), (16, 32, 64), 3),
                                             # coarse sides 20 and 28: the deepest levels of the 160^3 / 224^3 configs
                                             # (160 -> 80 -> 40 -> 20, 224 -> 112 -> 56 -> 28): ragged 16 x 8 tiles
                                             ((1, 80, 80, 80), (16, 32, 64), 1),
                                             ((1, 56, 56, 56), (32, 64), 1)])
def test_unet_forward_matches_oracle(shape, chs, batch):
    ref, net = _models(shape, chs)
    g = torch.Generator().manual_seed(1)
    x = torch.randn((batch,) + shape, generator=g)
    cond = 0.7 * x + 0.3 * torch.randn((batch,) + shape, generator=g)
    t = torch.rand(batch, generator=g)
    v = [torch.rand(batch, 6, generator=g)]
    with torch.no_grad():
        want = ref(x, t=t, s_conditioning=cond, v_conditionings=v)
        got = net(x.cuda(), t=t.cuda(), s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()]).cpu()
    assert got.shape == want.shape and got.dtype == torch.float32
    err = _rel_l2(got, want)
    print(f"unet {shape} {chs}: relative L2 error {err:.3e}, max abs {((got - want).abs().max() / want.abs().max()).item():.3e}")
    _assert_bf16_parity(err, lambda: ref(x, t=t, s_conditioning=cond, v_conditionings=v), want)
    # no time / parameter conditioning inputs, scalar t
    with torch.no_grad():
        want1 = ref(x[:1], t=torch.tensor(0.3), s_conditioning=cond[:1], v_conditionings=[v[0][:1]])
        got1 = net(x[:1].cuda(), t=torch.tensor(0.3), s_conditioning=cond[:1].cuda(), v_conditionings=[v[0][:1].cuda()]).cpu()
    _assert_bf16_parity(_rel_l2(got1, want1),
                        lambda: ref(x[:1], t=torch.tensor(0.3), s_conditioning=cond[:1], v_conditionings=[v[0][:1]]), want1)


def test_unet_fused_upsampling_equals_the_materialised_concat():
    """Inference reads the coarse tensor in the up blocks (CUNet.fuse_upsample); the result must agree with the path
    that writes interpolate(h) into the concat buffer (the one training uses) to bf16 rounding."""
    shape, chs, batch = (1, 16, 32, 16), (16, 32, 64), 2
    ref, net = _models(shape, chs)
    g = torch.Generator().manual_seed(8)
    x = torch.randn((batch,) + shape, generator=g)
    cond = 0.7 * x + 0.3 * torch.randn((batch,) + shape, generator=g)
    t, v = torch.rand(batch, generator=g), [torch.rand(batch, 6, generator=g)]
    kw = dict(t=t.cuda(), s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()])
    with torch.no_grad():
        want = ref(x, t=t, s_conditioning=cond, v_conditionings=v)
        assert net.fuse_upsample
        fused = net(x.cuda(), **kw).cpu()
        net.fuse_upsample = False
        plain = net(x.cuda(), **kw).cpu()
    print(f"fused vs materialised: {_rel_l2(fused, plain):.3e}; vs oracle: fused {_rel_l2(fused, want):.3e}, "
          f"materialised {_rel_l2(plain, want):.3e}")
    assert _rel_l2(fused, plain) < BF16_RTOL
    assert _rel_l2(fused, want) < 1.2e-2 and _rel_l2(plain, want) < 1.2e-2


def test_unet_fused_groupnorm_equals_the_two_pass_path():
    """Inference applies GroupNorm + SiLU inside the consumer conv (CUNet.fuse_gn, ops.conv3d in_norm); the result must agree
    with the path that runs vdm_gn_silu as its own pass (the one training uses) to bf16 rounding, and both with the oracle."""
    shape, chs, batch = (1, 16, 32, 16), (16, 32, 64), 2
    ref, net = _models(shape, chs)
    g = torch.Generator().manual_seed(9)
    x = torch.randn((batch,) + shape, generator=g)
    cond = 0.7 * x + 0.3 * torch.randn((batch,) + shape, generator=g)
    t, v = torch.rand(batch, generator=g), [torch.rand(batch, 6, generator=g)]
    kw = dict(t=t.cuda(), s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()])
    with torch.no_grad():
        want = ref(x, t=t, s_conditioning=cond, v_conditionings=v)
        assert net.fuse_gn
        net.fuse_gn_min_channels = 1            # every layer, also the narrow ones the default policy leaves two-pass
        from vdm4cdm_b200 import ops
        n0 = ops.launch_count()
        fused = net(x.cuda(), **kw).cpu()
        n_fused = ops.launch_count() - n0
        net.fuse_gn = False
        n0 = ops.launch_count()
        plain = net(x.cuda(), **kw).cpu()
        n_plain = ops.launch_count() - n0
    print(f"fused GN vs two-pass: {_rel_l2(fused, plain):.3e}; vs oracle: fused {_rel_l2(fused, want):.3e}, "
          f"two-pass {_rel_l2(plain, want):.3e}; launches {n_fused} vs {n_plain}")
    assert _rel_l2(fused, plain) < BF16_RTOL
    assert _rel_l2(fused, want) < 1.2e-2 and _rel_l2(plain, want) < 1.2e-2


def test_unet_polyphase_up_blocks_equal_the_direct_form():
    """Inference runs the up blocks' conv over the up-sampled channels in polyphase form (CUNet.polyphase_up: eight 2x2x2-tap
    convs of the coarse tensor + a depth-to-space residual); the result must agree with the direct 27-tap conv over
    silu(gn(cat([interpolate(h), skip]))) to bf16 rounding, and both with the oracle."""
    shape, chs, batch = (1, 16, 32, 16), (16, 32, 64), 2
    ref, net = _models(shape, chs)
    g = torch.Generator().manual_seed(10)
    x = torch.randn((batch,) + shape, generator=g)
    cond = 0.7 * x + 0.3 * torch.randn((batch,) + shape, generator=g)
    t, v = torch.rand(batch, generator=g), [torch.rand(batch, 6, generator=g)]
    kw = dict(t=t.cuda(), s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()])
    with torch.no_grad():
        want = ref(x, t=t, s_conditioning=cond, v_conditionings=v)
        assert net.polyphase_up
        poly = net(x.cuda(), **kw).cpu()
        net.polyphase_up = False
        direct = net(x.cuda(), **kw).cpu()
    print(f"polyphase vs direct: {_rel_l2(poly, direct):.3e}; vs oracle: polyphase {_rel_l2(poly, want):.3e}, "
          f"direct {_rel_l2(direct, want):.3e}")
    assert _rel_l2(poly, direct) < BF16_RTOL
    assert _rel_l2(poly, want) < 1.2e-2 and _rel_l2(direct, want) < 1.2e-2


def test_unet_forward_circular_padding_matches_oracle():
    """conv_padding_mode="circular" (the cropsize == 256 registry entries, src/utils.py:460)."""
    shape, chs, batch = (1, 16, 32, 16), (16, 32, 64), 2
    ref, net = _models(shape, chs, padding="circular")
    g = torch.Generator().manual_seed(2)
    x = torch.randn((batch,) + shape, generator=g)
    cond = 0.7 * x + 0.3 * torch.randn((batch,) + shape, generator=g)
    t, v = torch.rand(batch, generator=g), [torch.rand(batch, 6, generator=g)]
    with torch.no_grad():
        want = ref(x, t=t, s_conditioning=cond, v_conditionings=v)
        got = net(x.cuda(), t=t.cuda(), s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()]).cpu()
        zero_pad = _models(shape, chs, padding="zeros")[0](x, t=t, s_conditioning=cond, v_conditionings=v)
    err = _rel_l2(got, want)
    # Tolerance for a whole random-init network: the error torch's own bf16 autocast of the ORACLE makes on this
    # input (measured 1.6e-2 here; circular padding is ~30% noisier than zero padding for torch too, 1.3e-2), and
    # never looser than 2e-2.  A wrong halo anywhere shows up at the 1e-1 level (zero padding: 0.89).
    with torch.no_grad(), torch.autocast("cpu", dtype=torch.bfloat16):
        autocast_err = _rel_l2(ref(x, t=t, s_conditioning=cond, v_conditionings=v).float(), want)
    print(f"circular unet: relative L2 error {err:.3e} (torch bf16 autocast of the oracle: {autocast_err:.3e}; "
          f"zero-padded network differs by {_rel_l2(zero_pad, want):.3e})")
    assert err < min(max(BF16_RTOL, autocast_err), 2e-2), (err, autocast_err)
    # periodic boundaries make the network equivariant under shifts by a multiple of the coarsest cell (4 voxels) -- to the
    # bf16 noise floor: every conv output is bit-for-bit equivariant (tests/test_gpu_conv3d.py::
    # test_conv3d_circular_is_shift_equivariant_bit_for_bit), but the GroupNorm sums are added in an order that depends on
    # the position (per-lane fp32 sums along d in the marching schedule), they move by ~1e-7, a few bf16 roundings of the
    # normalised tensor flip, and a random-init network amplifies single flips to every element within ~3 layers
    # (tools/check_equivariance_per_layer.py: 0.3% of the elements differ after the first block, 16% after the third).
    # The bar is therefore the parity bar; a wrong halo shows up at the 1e-1 level (zero padding: 0.89).
    shift = dict(shifts=(4, 8, 4), dims=(2, 3, 4))
    with torch.no_grad():
        rolled = net(torch.roll(x, **shift).cuda(), t=t.cuda(), s_conditioning=torch.roll(cond, **shift).cuda(),
                     v_conditionings=[v[0].cuda()]).cpu()
    eq = _rel_l2(rolled, torch.roll(got, **shift))
    print(f"circular unet: shift equivariance defect {eq:.3e}")
    assert eq < min(max(BF16_RTOL, autocast_err), 2e-2), eq
    assert _rel_l2(rolled, torch.roll(want, **shift)) < min(max(BF16_RTOL, autocast_err), 2e-2)
    # the sampler works on top of it (packed input is re-padded every step)
    from vdm4cdm_b200.vdm_model import VDM
    xs = VDM(net).cuda().eval().sample(batch, 3, "cuda:0", seed=1, s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()])
    assert torch.isfinite(xs).all()


def test_sampler_chain_matches_oracle_per_step_and_graph_equals_eager():
    from oracle.vdm_ref import VDM as RefVDM
    from vdm4cdm_b200.vdm_model import VDM
    shape, chs, batch, n_steps = (1, 16, 16, 16), (16, 32), 2, 6
    ref_net, net = _models(shape, chs)
    ref_vdm, vdm = RefVDM(ref_net).eval(), VDM(net).cuda().eval()
    g = torch.Generator().manual_seed(3)
    noises = [torch.randn((batch,) + shape, generator=g) for _ in range(n_steps + 1)]
    cond = torch.randn((batch,) + shape, generator=g)
    v = [torch.rand(batch, 6, generator=g)]
    kw_ref = dict(s_conditioning=cond, v_conditionings=v)
    kw = dict(s_conditioning=cond.cuda(), v_conditionings=[v[0].cuda()])
    nf = lambda d, shp: noises[d]
    vdm.use_cuda_graph = True
    traj = vdm.sample(batch, n_steps, "cuda:0", return_all=True, noise_fn=lambda d, s: noises[d].cuda(), **kw).cpu()
    vdm.use_cuda_graph = False
    traj_eager = vdm.sample(batch, n_steps, "cuda:0", return_all=True, noise_fn=lambda d, s: noises[d].cuda(), **kw).cpu()
    # same kernels, same inputs; GroupNorm statistics are accumulated with fp64 atomics whose order is not
    # fixed, so the two runs agree to rounding noise rather than bit for bit
    assert _rel_l2(traj, traj_eager) < 1e-3, _rel_l2(traj, traj_eager)
    assert traj.shape == (n_steps + 1, batch) + shape
    steps = torch.linspace(1.0, 0.0, n_steps + 1)
    z = noises[0]
    worst = 0.0
    with torch.no_grad():
        for i in range(n_steps):
            want = ref_vdm.sample_zs_given_zt(zt=z, t=steps[i], s=steps[i + 1], noise=noises[i + 1], **kw_ref)
            worst = max(worst, _rel_l2(traj[i], want))
            z = traj[i]                              # restart the oracle from the CUDA path's state
    print(f"sampler: worst per-step relative L2 error {worst:.3e}")
    assert worst < BF16_RTOL, worst
    # final map x = z_0 / alpha_0 and the folded variant agree
    x_folded = vdm.sample(batch, n_steps, "cuda:0", noise_fn=lambda d, s: noises[d].cuda(), **kw).cpu()
    assert torch.allclose(x_folded, traj[-1], rtol=1e-5, atol=1e-5)
    # whole-chain comparison against the oracle's own trajectory (errors compound: looser, reported)
    with torch.no_grad():
        full = ref_vdm.sample(batch, n_steps, "cpu", noise_fn=nf, **kw_ref)
    print(f"sampler: end-to-end relative L2 error after {n_steps} steps {_rel_l2(x_folded, full):.3e}")
    assert _rel_l2(x_folded, full) < 5 * BF16_RTOL


def test_graph_replay_after_new_weights_matches_a_fresh_model():
    """A captured sampler graph reads the packed filters without packing lazily, so ``SamplerSession.reset`` must
    re-pack every slot (the up blocks' polyphase and input-channel-slice filters too): after ``load_state_dict`` a
    replayed chain with the same seed and noise equals a fresh VDM with the new weights."""
    from vdm4cdm_b200.vdm_model import VDM
    shape, chs, batch, n_steps = (1, 16, 16, 16), (16, 32), 2, 4
    _, net = _models(shape, chs)
    _, net_new = _models(shape, chs, seed=1)
    vdm, vdm_new = VDM(net).cuda().eval(), VDM(net_new).cuda().eval()
    g = torch.Generator().manual_seed(3)
    noises = [torch.randn((batch,) + shape, generator=g).cuda() for _ in range(n_steps + 1)]
    kw = dict(seed=0, noise_fn=lambda d, s: noises[d], s_conditioning=torch.randn((batch,) + shape, generator=g).cuda(),
              v_conditionings=[torch.rand(batch, 6, generator=g).cuda()])
    vdm.use_cuda_graph = vdm_new.use_cuda_graph = True
    old = vdm.sample(batch, n_steps, "cuda:0", **kw).cpu()          # eager first step, then the graph is captured
    assert vdm._sessions and next(iter(vdm._sessions.values())).graph is not None
    vdm.load_state_dict(vdm_new.state_dict())
    got = vdm.sample(batch, n_steps, "cuda:0", **kw).cpu()          # replays the graph captured above
    want = vdm_new.sample(batch, n_steps, "cuda:0", **kw).cpu()
    assert _rel_l2(old, want) > 1e-2                                # the weights differ enough to tell
    assert _rel_l2(got, want) < 1e-3, _rel_l2(got, want)


def test_philox_sampling_is_batch_independent():
    from vdm4cdm_b200.vdm_model import VDM
    shape, chs = (1, 16, 16, 16), (16, 32)
    _, net = _models(shape, chs, v_dims=())
    vdm = VDM(net).cuda().eval()
    cond = torch.randn((1,) + shape, generator=torch.Generator().manual_seed(5)).cuda()
    both = vdm.sample(2, 4, "cuda:0", seed=77, realisation_ids=[4, 9], s_conditioning=cond.expand(2, -1, -1, -1, -1).contiguous())
    one = vdm.sample(1, 4, "cuda:0", seed=77, realisation_ids=[9], s_conditioning=cond)
    # same (seed, realisation id) -> same noise; the network sees the same sample, so results agree to bf16 noise.
    # Bit equality is not guaranteed: GroupNorm statistics are accumulated with atomics whose partition depends on
    # the batch size, a last-bit change of a scale flips a few bf16 roundings, and those flips propagate (measured
    # max |diff| ~1e-2 of the output range, relative L2 ~1e-3) -- so compare in relative L2 at the bf16 tolerance.
    assert _rel_l2(both[1:2], one) < BF16_RTOL, _rel_l2(both[1:2], one)
    assert _rel_l2(both[0:1], one) > 0.3
