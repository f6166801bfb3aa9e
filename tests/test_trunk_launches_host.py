"""The CUNet trunk's launch sequence, pinned on the host (no GPU needed).

Every ``ops`` function the trunk and ``vdm4cdm_b200.autograd`` call is replaced by a recorder that logs the function
and its arguments (bound to the signature, defaults dropped) and hands back the ``out`` the caller passed.  Tensors are
written as ``#<first-seen ordinal>:<dtype>[shape]``, ordinals keyed by data pointer, so which buffer every launch reads
and writes is pinned too.  The recorder declines the fused skip conv (``skip_x``) for layers wider than 32 channels, so
both outcomes of that fusion are exercised.  ``tests/golden/trunk_launches.json`` holds the expected logs; running this
file as a script rewrites it.

A second test checks that ``CUNet.refresh_packed`` brings every slot of the packed-filter cache up to date after the
parameters change in place: a captured sampler graph reads those slots and never packs lazily again.
"""
import inspect
import json
import os

import pytest
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "trunk_launches.json")

RECORDED = ("conv3d", "conv3d_wgrad", "gn_coef", "gn_silu", "gn_silu_view", "gn_silu_bwd", "avgpool2", "avgpool2_bwd",
            "upsample2", "upsample2_bwd", "pad_circular", "pack_input", "pack_conv_weight_into", "pack_job_table",
            "pack_conv_weights_batched", "increment", "set_profile_tag")
OUT_ARGS = ("out", "grad_out", "dx")        # the argument a recorder hands back


class Recorder:
    def __init__(self, pack=None):
        self.log = []
        self.ordinal = {}
        self.alive = []          # every logged tensor stays referenced, so a data pointer is never reused in one log
        self.pack = pack         # optional host stand-in for pack_conv_weight_into that writes ``out``

    def fmt(self, v):
        from vdm4cdm_b200 import ops
        if isinstance(v, torch.Tensor):
            if v.data_ptr() not in self.ordinal:
                self.ordinal[v.data_ptr()] = len(self.ordinal)
                self.alive.append(v)
            dt = str(v.dtype).replace("torch.", "").replace("bfloat16", "bf16")
            return f"#{self.ordinal[v.data_ptr()]}:{dt}{list(v.shape)}"
        if isinstance(v, (tuple, list)):
            if tuple(v) == ops.TAPS_3X3X3:
                return "3x3x3"
            if tuple(v) == ops.TAPS_1X1X1:
                return "1x1x1"
            return "(" + ", ".join(self.fmt(e) for e in v) + ")"
        if isinstance(v, torch.device):
            return v.type
        return repr(v)

    def wrap(self, name, fn):
        sig = inspect.signature(fn)

        def rec(*args, **kwargs):
            from vdm4cdm_b200 import ops
            bound = sig.bind(*args, **kwargs)
            shown = [f"{k}={self.fmt(v)}" for k, v in bound.arguments.items()
                     if not (sig.parameters[k].default is not inspect.Parameter.empty and _same(v, sig.parameters[k].default))]
            self.log.append(f"{name}({', '.join(shown)})")
            a = bound.arguments
            if name == "conv3d" and a.get("skip_x") is not None and a["c_out"] > 32:
                self.log[-1] += " -> UnsupportedFusion"
                raise ops.UnsupportedFusion("recorder: fused skip conv declined for layers wider than 32 channels")
            if name == "pack_conv_weight_into" and self.pack is not None:
                self.pack(*args, **kwargs)
            if name == "pack_job_table":
                return torch.zeros(len(a["jobs"]), dtype=torch.uint8)
            for k in OUT_ARGS:
                if a.get(k) is not None:
                    return a[k]
            return None
        return rec

    def __enter__(self):
        from vdm4cdm_b200 import ops
        self.saved = {n: getattr(ops, n) for n in RECORDED}
        for n, fn in self.saved.items():
            setattr(ops, n, self.wrap(n, fn))
        return self

    def __exit__(self, *exc):
        from vdm4cdm_b200 import ops
        for n, fn in self.saved.items():
            setattr(ops, n, fn)


def _same(v, default):
    if isinstance(v, torch.Tensor) or isinstance(default, torch.Tensor):
        return v is default
    return v == default


def _net(chs, grid, **kw):
    from vdm4cdm_b200.networks import CUNet
    torch.manual_seed(0)
    return CUNet(shape=(1, grid, grid, grid), chs=chs, s_conditioning_channels=1, v_conditioning_dims=[3],
                 t_conditioning=True, **kw)


def _inputs(b, grid, requires_grad=False):
    g = torch.Generator().manual_seed(1)
    x = torch.randn((b, 1, grid, grid, grid), generator=g).requires_grad_(requires_grad)
    return dict(x=x, t=torch.rand(b, generator=g), s_conditioning=torch.randn((b, 1, grid, grid, grid), generator=g),
                v_conditionings=[torch.rand(b, 3, generator=g)])


def _inference(padding="zeros", precision="bf16", **switches):
    """One no_grad forward at 32^3, B = 2, chs = (16, 32, 64, 128): sets the given CUNet attributes first."""
    def run():
        net = _net((16, 32, 64, 128), 32, conv_padding_mode=padding, precision=precision).eval()
        for k, v in switches.items():
            setattr(net, k, v)
        with Recorder() as r, torch.no_grad():
            net(**_inputs(2, 32))
        return r.log
    return run


def _training(padding):
    """At 16^3, B = 2, chs = (16, 32, 64), dropout on: an inference forward (it leaves derived filter slots in the
    cache), then two training forward + backward passes with an in-place parameter update in between."""
    def run():
        net = _net((16, 32, 64), 16, conv_padding_mode=padding, dropout_prob=0.1)
        with Recorder() as r:
            with torch.no_grad():
                net.eval()(**_inputs(2, 16))
            net.train()
            for _ in range(2):
                net(**_inputs(2, 16, requires_grad=True)).sum().backward()
                with torch.no_grad():
                    for p in net.parameters():
                        p.add_(0.01)
        return r.log
    return run


CASES = {
    "infer_bf16_zeros": _inference(),
    "infer_bf16_circular": _inference("circular"),
    "infer_tf32_zeros": _inference(precision="tf32"),
    "infer_tf32_circular": _inference("circular", precision="tf32"),
    "infer_bf16_fuse_gn_min_channels_1": _inference(fuse_gn_min_channels=1),
    "infer_bf16_no_fuse_gn": _inference(fuse_gn=False),
    "infer_bf16_no_fuse_upsample": _inference(fuse_upsample=False),
    "infer_bf16_no_polyphase_up": _inference(polyphase_up=False),
    "train_zeros": _training("zeros"),
    "train_circular": _training("circular"),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_trunk_launch_sequence_matches_golden(case):
    with open(GOLDEN) as f:
        want = json.load(f)[case]
    got = CASES[case]()
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, f"call {i}"


def _pack_on_host(w, out, transpose_flip=False, ci0=0, n_ci=None):
    """Host stand-in for ``ops.pack_conv_weight_into``: writes the packed filter into ``out`` in the kernel layout."""
    from vdm4cdm_b200 import ops
    n_ci = w.shape[1] if n_ci is None else n_ci
    if out.dtype == torch.bfloat16:
        out.copy_(ops.pack_conv_weight(w[:, ci0:ci0 + n_ci], transpose_flip=transpose_flip))
        return out
    k3, planes, cop = out.shape[0], out.shape[1], out.shape[2]          # fp32 [k^3, Cin_pad/4, Cout_pad, 4]
    t = w.permute(2, 3, 4, 1, 0).reshape(k3, w.shape[1], w.shape[0])
    full = t.new_zeros(k3, planes * 4, cop)
    full[:, :w.shape[1], :w.shape[0]] = t
    out.copy_(full.reshape(k3, planes, 4, cop).permute(0, 1, 3, 2))
    return out


def _fill_cache(net):
    """Every kind of cache slot: bf16 and fp32 forward filters, dgrad filters, input-channel slices, polyphase groups."""
    net.train()
    net(**_inputs(2, 16, requires_grad=True)).sum().backward()
    net.eval()
    with torch.no_grad():
        for precision in ("tf32", "bf16"):
            net.precision = precision
            net(**_inputs(2, 16))


def _slot_buffers(net):
    return {slot: entry.buf for slot, entry in net._packed_cache.items()}


def test_refresh_packed_repacks_every_stale_slot():
    """After an in-place parameter change, refresh_packed() leaves every cached filter equal to a fresh pack of the new
    weights -- also the up blocks' polyphase and input-channel-slice filters, which a captured sampler graph reads."""
    net = _net((16, 32, 64), 16)
    with Recorder(pack=_pack_on_host):
        _fill_cache(net)
        with torch.no_grad():
            for p in net.parameters():
                p.add_(0.01)
        net.refresh_packed()
        got = _slot_buffers(net)
        fresh = _net((16, 32, 64), 16)
        fresh.load_state_dict(net.state_dict())
        _fill_cache(fresh)
        want = _slot_buffers(fresh)
    assert sorted(got) == sorted(want)
    stale = [slot for slot in want if not torch.equal(got[slot], want[slot])]
    assert not stale, stale


if __name__ == "__main__":
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    golden = {case: run() for case, run in sorted(CASES.items())}
    with open(GOLDEN, "w") as f:
        json.dump(golden, f, indent=1)
        f.write("\n")
    print(f"wrote {GOLDEN}: " + ", ".join(f"{k} {len(v)} calls" for k, v in golden.items()))
