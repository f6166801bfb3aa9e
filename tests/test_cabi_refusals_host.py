"""Argument refusals of the elementwise, pack and sampler C entry points, pinned on the host (no GPU needed).

Each case calls one entry point through ``_C.lib()`` with arguments that fail one check, and compares the return code
and the exact ``vdm_last_error_string()`` with ``tests/golden/cabi_refusals.json``.  Every check runs before the entry
point's first CUDA call, so the device pointers are fake.  The module skips on a machine with a GPU: there a case that
slipped past its checks would launch a kernel on those pointers.  Running this file as a script rewrites the golden.
"""
import ctypes
import json
import os

import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cabi_refusals.json")

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="fake device pointers: host-only")

P = 1 << 20             # a fake, 16-byte aligned device address; no case gets far enough to use it
MISALIGNED = P + 8
VDM_E_BADARG = -1


def view(planes=4, plane0=0, data=P):
    from vdm4cdm_b200 import _C
    return _C.Tensor(data, planes, plane0)


# Valid arguments of each entry point, in ABI order (views are built per call).  A case overrides some of them.
_VIEW = object()
_GN = dict(x=_VIEW, y=_VIEW, batch=2, voxels=4096, channels=32, groups=8, stats=P, gamma=P, beta=P, eps=1e-5,
           dropout_p=0.0, seed=0, seed_step=None, layer_tag=0, stream=None)
_POOL = dict(x=_VIEW, y=_VIEW, batch=2, depth=16, height=16, width=16, channels=32, stats=None, stats_channels=0,
             stats_c0=0, stream=None)
_PACK_INPUT = dict(z=P, cond=P, out=_VIEW, batch=2, voxels=4096, n_cond=1, c_pad=16, stream=None)
ARGS = {
    "vdm_gn_silu_step": _GN,
    "vdm_gn_silu": {k: v for k, v in _GN.items() if k != "seed_step"},
    "vdm_gn_silu_f32": {k: (16 if k == "channels" else v) for k, v in _GN.items()
                        if k not in ("dropout_p", "seed", "seed_step", "layer_tag")},
    "vdm_gn_silu_view": dict(x=_VIEW, y=_VIEW, batch=2, depth=16, height=16, width=16, channels=32, c_off=0,
                             channels_total=64, groups=8, stats=P, gamma=P, beta=P, eps=1e-5, upsample=0, stream=None),
    "vdm_avgpool2": _POOL,
    "vdm_avgpool2_f32": dict(_POOL, channels=16),
    "vdm_upsample2": _POOL,
    "vdm_upsample2_f32": dict(_POOL, channels=16),
    "vdm_avgpool2_bwd": dict(x=_VIEW, y=_VIEW, batch=2, depth=16, height=16, width=16, channels=32, accumulate=0,
                             stats=None, stats_channels=0, stats_c0=0, stream=None),
    "vdm_upsample2_bwd": _POOL,
    "vdm_pad_circular": dict(x=_VIEW, y=_VIEW, batch=2, depth=16, height=16, width=16, channels=32, stream=None),
    "vdm_channel_stats": dict(x=_VIEW, batch=2, voxels=4096, channels=32, stats=P, stats_channels=0, stats_c0=0,
                              stream=None),
    "vdm_gn_silu_bwd_reduce": dict(x=_VIEW, dy=_VIEW, batch=2, voxels=4096, channels=32, groups=8, stats=P, gamma=P, beta=P,
                                   eps=1e-5, dropout_p=0.0, seed=0, seed_step=None, layer_tag=0, sums=P, sums_channels=0,
                                   sums_c0=0, stream=None),
    "vdm_gn_silu_bwd_apply": dict(x=_VIEW, dy=_VIEW, add=None, dx=_VIEW, batch=2, voxels=4096, channels=32, groups=8,
                                  stats=P, gamma=P, beta=P, eps=1e-5, dropout_p=0.0, seed=0, seed_step=None, layer_tag=0,
                                  sums=P, sums_channels=0, sums_c0=0, out_stats=None, out_stats_channels=0,
                                  out_stats_c0=0, stream=None),
    "vdm_pack_input": _PACK_INPUT,
    "vdm_pack_input_f32": _PACK_INPUT,
    "vdm_pack_conv_weight": dict(w=P, packed=P, c_out=32, c_in=16, kernel=3, transpose_flip=0, ci0=0, n_ci=16, c_in_pad=16,
                                 c_out_pad=32, stream=None),
    "vdm_pack_conv_weight_f32": dict(w=P, packed=P, c_out=32, c_in=16, kernel=3, c_in_pad=16, c_out_pad=32, stream=None),
}

# A valid dgrad filter: K = 16 conv output channels (c_in_pad 16), N = all 32 conv input channels (c_out_pad 32).
_DGRAD = dict(transpose_flip=1, c_out=16, c_in=32, n_ci=32)

# (entry point, case label, overrides): every case fails exactly one check.  View overrides are view() keyword dicts.
_GRID_CASES = [("x NULL", dict(x=None)), ("y misaligned", dict(y=dict(data=MISALIGNED))),
               ("window past the planes", dict(x=dict(planes=4, plane0=1))), ("batch 0", dict(batch=0)),
               ("65536 (sample, plane) blocks", dict(batch=16384)), ("2^31 voxels", dict(depth=1292, height=1292, width=1292)),
               ("odd depth", dict(depth=15)), ("odd width", dict(width=7)), ("zero height", dict(height=0))]
CASES = (
    [(n, "x NULL", dict(x=None)) for n in ("vdm_gn_silu_step", "vdm_gn_silu", "vdm_gn_silu_f32")] +
    [(n, "y misaligned", dict(y=dict(data=MISALIGNED))) for n in ("vdm_gn_silu_step", "vdm_gn_silu_f32")] +
    [(n, "stats NULL", dict(stats=None)) for n in ("vdm_gn_silu_step", "vdm_gn_silu_f32")] +
    [("vdm_gn_silu_step", "12 channels", dict(channels=12)), ("vdm_gn_silu_f32", "18 channels", dict(channels=18)),
     ("vdm_gn_silu_step", "window past the planes", dict(y=dict(planes=5, plane0=2))),
     ("vdm_gn_silu_f32", "window past the planes", dict(x=dict(planes=3)))] +
    [(n, "voxels 0", dict(voxels=0)) for n in ("vdm_gn_silu_step", "vdm_gn_silu", "vdm_gn_silu_f32")] +
    [(n, "65536 (sample, plane) blocks", dict(batch=16384)) for n in ("vdm_gn_silu_step", "vdm_gn_silu", "vdm_gn_silu_f32")] +
    [(n, "groups 3", dict(groups=3)) for n in ("vdm_gn_silu_step", "vdm_gn_silu", "vdm_gn_silu_f32")] +
    [(n, "groups 0", dict(groups=0)) for n in ("vdm_gn_silu_step", "vdm_gn_silu_f32")] +
    [(n, f"dropout_p {p}", dict(dropout_p=p)) for n in ("vdm_gn_silu_step", "vdm_gn_silu") for p in (1.0, -0.25)] +
    [(n, label, kw) for n in ("vdm_avgpool2", "vdm_avgpool2_f32", "vdm_upsample2", "vdm_upsample2_f32", "vdm_avgpool2_bwd",
                              "vdm_upsample2_bwd") for label, kw in _GRID_CASES] +
    [("vdm_avgpool2", "12 channels", dict(channels=12)), ("vdm_avgpool2_f32", "6 channels", dict(channels=6)),
     ("vdm_upsample2", "12 channels", dict(channels=12)), ("vdm_upsample2_f32", "6 channels", dict(channels=6)),
     ("vdm_avgpool2_f32", "x window past the planes", dict(x=dict(planes=3))),
     ("vdm_upsample2_f32", "y window past the planes", dict(y=dict(planes=3)))] +
    [("vdm_gn_silu_view", label, kw) for label, kw in [
        ("x NULL", dict(x=None)), ("y misaligned", dict(y=dict(data=MISALIGNED))), ("12 channels", dict(channels=12)),
        ("gamma NULL", dict(gamma=None)), ("depth 0", dict(depth=0)), ("batch 0", dict(batch=0)),
        ("65536 (sample, plane) blocks", dict(batch=16384)), ("c_off 4", dict(c_off=4)), ("c_off -8", dict(c_off=-8)),
        ("window past the norm", dict(c_off=40)), ("groups 6", dict(groups=6)), ("groups 0", dict(groups=0)),
        ("2^31 voxels", dict(depth=1291, height=1291, width=1291)),
        ("2^31 voxels, up-sampled", dict(depth=1292, height=1292, width=1292, upsample=1)),
        ("odd fine grid, up-sampled", dict(depth=15, upsample=1)),
        ("odd fine grid, coarse", dict(height=9, upsample=2))]] +
    [("vdm_pad_circular", label, kw) for label, kw in [
        ("x NULL", dict(x=None)), ("12 channels", dict(channels=12)), ("65536 (sample, plane) blocks", dict(batch=16384)),
        ("depth 0", dict(depth=0)), ("2^31 padded voxels", dict(depth=1289, height=1289, width=1289))]] +
    [("vdm_channel_stats", label, kw) for label, kw in [
        ("stats NULL", dict(stats=None)), ("12 channels", dict(channels=12)), ("voxels 0", dict(voxels=0)),
        ("65536 (sample, plane) blocks", dict(batch=16384))]] +
    [(n, label, kw) for n in ("vdm_gn_silu_bwd_reduce", "vdm_gn_silu_bwd_apply") for label, kw in [
        ("sums NULL", dict(sums=None)), ("dy misaligned", dict(dy=dict(data=MISALIGNED))), ("voxels 0", dict(voxels=0)),
        ("65536 (sample, plane) blocks", dict(batch=16384)), ("groups 5", dict(groups=5)),
        ("dropout_p 1.5", dict(dropout_p=1.5))]] +
    [("vdm_gn_silu_bwd_apply", "dx NULL", dict(dx=None)),
     ("vdm_gn_silu_bwd_apply", "add misaligned", dict(add=dict(data=MISALIGNED)))] +
    [(n, label, kw) for n in ("vdm_pack_input", "vdm_pack_input_f32") for label, kw in [
        ("z NULL", dict(z=None)), ("out NULL", dict(out=None)), ("out data NULL", dict(out=dict(data=0))),
        ("batch 0", dict(batch=0)), ("batch 65536", dict(batch=65536)), ("voxels 0", dict(voxels=0)),
        ("c_pad 12", dict(c_pad=12)), ("c_pad 0", dict(c_pad=0)), ("n_cond 8", dict(n_cond=8)),
        ("n_cond -1", dict(n_cond=-1)), ("plane0 -1", dict(out=dict(plane0=-1))),
        ("window past the planes", dict(out=dict(planes=4, plane0=3))), ("cond NULL", dict(cond=None))]] +
    [("vdm_pack_input_f32", "out misaligned", dict(out=dict(data=MISALIGNED)))] +
    [(n, label, kw) for n in ("vdm_pack_conv_weight", "vdm_pack_conv_weight_f32") for label, kw in [
        ("w NULL", dict(w=None)), ("packed NULL", dict(packed=None)), ("c_out 0", dict(c_out=0)),
        ("c_in 0", dict(c_in=0)), ("kernel 4", dict(kernel=4)), ("kernel 0", dict(kernel=0)),
        ("c_in_pad 12", dict(c_in_pad=12)), ("c_in_pad 0", dict(c_in_pad=0)), ("c_out_pad 24", dict(c_out_pad=24)),
        ("packed misaligned", dict(packed=MISALIGNED)), ("c_in above c_in_pad", dict(c_in=17)),
        ("c_out above c_out_pad", dict(c_out=33))]] +
    [("vdm_pack_conv_weight", "c_in_pad 24", dict(c_in_pad=24)),
     ("vdm_pack_conv_weight_f32", "c_in_pad 20", dict(c_in_pad=20))] +
    [("vdm_pack_conv_weight", label, dict(_DGRAD, **kw)) for label, kw in [
        ("dgrad slice past c_in", dict(ci0=8)), ("dgrad slice ci0 -1", dict(ci0=-1)), ("dgrad slice empty", dict(n_ci=0)),
        ("dgrad K above c_in_pad", dict(c_out=17)), ("dgrad N above c_out_pad", dict(c_out_pad=16))]]
)


def _id(case):
    return f"{case[0]}: {case[1]}"


def _refusal(name, overrides):
    """(return code, error string) of one call of entry point ``name``."""
    from vdm4cdm_b200 import _C
    args = []
    for k, v in ARGS[name].items():
        v = overrides.get(k, v)
        if v is _VIEW or isinstance(v, dict):
            v = ctypes.byref(view(**(v if isinstance(v, dict) else {})))
        args.append(v)
    lib = _C.lib()
    rc = getattr(lib, name)(*args)
    return rc, lib.vdm_last_error_string().decode()


def _all():
    return {_id(c): list(_refusal(c[0], c[2])) for c in CASES}


@pytest.mark.parametrize("case", CASES, ids=_id)
def test_refusal_matches_golden(case):
    with open(GOLDEN) as f:
        want = json.load(f)[_id(case)]
    rc, msg = _refusal(case[0], case[2])
    assert rc == VDM_E_BADARG
    assert [rc, msg] == want


def test_every_entry_point_has_cases():
    assert sorted({c[0] for c in CASES}) == sorted(ARGS)
    assert len({_id(c) for c in CASES}) == len(CASES)


def test_pack_input_refuses_a_misaligned_out():
    """The kernel stores 16-byte units: a misaligned ``out`` is an argument error, as it is for the fp32 form."""
    rc, msg = _refusal("vdm_pack_input", dict(out=dict(data=MISALIGNED)))
    assert (rc, msg) == (VDM_E_BADARG, "vdm_pack_input: bad argument")


if __name__ == "__main__":
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    if torch.cuda.is_available():
        sys.exit("fake device pointers: run this on a machine without a GPU")
    golden = _all()
    bad = {k: v for k, v in golden.items() if v[0] != VDM_E_BADARG}
    if bad:
        sys.exit(f"not refused as argument errors: {bad}")
    with open(GOLDEN, "w") as f:
        json.dump(golden, f, indent=1)
        f.write("\n")
    print(f"wrote {GOLDEN}: {len(golden)} cases")
