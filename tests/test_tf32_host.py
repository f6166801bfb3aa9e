"""Host-side logic of the TF32 inference mode (no GPU needed): CUNet(precision=...) validation, the inference-only
guard, and the shapes of the fp32 packed filters."""
import pytest
import torch


def _net(**kw):
    from vdm4cdm_b200.networks import CUNet
    return CUNet(shape=(1, 16, 16, 16), chs=(16, 32), s_conditioning_channels=1, v_conditioning_dims=[6],
                 t_conditioning=True, **kw)


def test_precision_default_and_validation():
    assert _net().precision == "bf16"
    assert _net(precision="tf32").precision == "tf32"
    with pytest.raises(ValueError, match="precision"):
        _net(precision="fp16")
    net = _net()
    net.precision = "tf32"                  # a plain attribute, settable on a loaded model
    assert net.input_channels_pad() == 8 and net._lanes() == 4
    net.precision = "bf16"
    assert net.input_channels_pad() == 16 and net._lanes() == 8
    net.precision = "fp64"
    with pytest.raises(ValueError, match="precision"):
        net(torch.zeros(1, 1, 16, 16, 16))


def test_tf32_with_gradients_is_not_implemented():
    net = _net(precision="tf32")
    x = torch.zeros(1, 1, 16, 16, 16)
    with pytest.raises(NotImplementedError, match="inference-only"):
        net(x, t=torch.zeros(1), s_conditioning=x, v_conditionings=[torch.zeros(1, 6)])
    with pytest.raises(NotImplementedError, match="inference-only"):
        net.run_packed(torch.zeros(1, 2, 16, 16, 16, 4), {}, tape={})


@pytest.mark.parametrize("co,ci,k,want", [(32, 16, 3, (27, 4, 32, 4)), (32, 2, 3, (27, 2, 32, 4)),
                                          (1, 32, 3, (27, 8, 16, 4)), (64, 96, 1, (1, 24, 64, 4)),
                                          (256, 256, 3, (27, 64, 256, 4))])
def test_fp32_packed_weight_shapes(co, ci, k, want):
    from vdm4cdm_b200 import ops
    assert ops.packed_weight_shape((co, ci, k, k, k), dtype=torch.float32) == want
    # the bf16 shape is unchanged
    assert ops.packed_weight_shape((co, ci, k, k, k)) == (k ** 3, -(-ci // 16) * 2, -(-co // 16) * 16, 8)
    with pytest.raises(ValueError):
        ops.packed_weight_shape((co, ci, k, k, k), transpose_flip=True, dtype=torch.float32)


def test_fp32_planar_layout_round_trip():
    from vdm4cdm_b200 import ops
    x = torch.randn(2, 5, 3, 4, 6)
    p = ops.to_planar(x, 8, dtype=torch.float32)
    assert p.shape == (2, 2, 3, 4, 6, 4) and p.dtype == torch.float32
    assert torch.equal(ops.from_planar(p, 5), x)
    assert torch.equal(p[0, 1, 2, 3, 4], torch.tensor([x[0, 4, 2, 3, 4], 0.0, 0.0, 0.0]))


def test_ops_reject_mixed_planar_dtypes():
    """The dtype checks run before any device pointer is touched (CPU tensors fail the same checks)."""
    from vdm4cdm_b200 import ops
    with pytest.raises(ValueError):
        ops._same_lanes(4, torch.zeros(1, 2, 4, 4, 4, 8, dtype=torch.bfloat16), "t")
    with pytest.raises(ValueError):
        ops._planar_lanes(torch.zeros(1, 2, 4, 4, 4, 8, dtype=torch.float32), "t")
