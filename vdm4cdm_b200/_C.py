"""ctypes binding of ``libvdm4cdm_b200.so`` (the C ABI declared in ``include/vdm4cdm_b200.h``).

There is deliberately no fallback: if the shared library is missing or a call fails, a
``RuntimeError`` is raised.  ``lib()`` only loads the library (possible on a CPU-only box, used by
the symbol-export test); every compute entry point needs an sm_100 GPU.
"""
from __future__ import annotations

import ctypes
import os
import re
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int8, c_int32, c_int64, c_size_t, \
    c_uint32, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# VDM4CDM_BRINGUP=1 selects the bring-up build (`make -C vdm4cdm_b200/csrc bringup`: ablation branches + vdm_debug_set);
# tools/bench_epilogue.py and tools/bench_conv.py set it, nothing else does.
BRINGUP = os.environ.get("VDM4CDM_BRINGUP", "0") == "1"
LIB_PATH = os.path.join(_HERE, "lib", "libvdm4cdm_b200_bringup.so" if BRINGUP else "libvdm4cdm_b200.so")
HEADER_PATH = os.path.join(_HERE, "..", "include", "vdm4cdm_b200.h")
MAX_TAPS = 27


class ConvDesc(Structure):
    _fields_ = [
        ("batch", c_int32), ("depth", c_int32), ("height", c_int32), ("width", c_int32),
        ("c_in", c_int32), ("c_out", c_int32), ("c_out_pad", c_int32), ("n_taps", c_int32),
        ("tap_offset", (c_int8 * 3) * MAX_TAPS),
        ("circular", c_int32), ("out_fp32", c_int32),
        ("x_planes", c_int32), ("x_plane0", c_int32),
        ("y_planes", c_int32), ("y_plane0", c_int32),
        ("r_planes", c_int32), ("r_plane0", c_int32),
    ]


class PackJob(Structure):
    _fields_ = [
        ("w", c_void_p), ("packed", c_void_p),
        ("c_out", c_int32), ("c_in", c_int32), ("k3", c_int32), ("transpose_flip", c_int32),
        ("ci0", c_int32), ("n_ci", c_int32), ("c_in_pad", c_int32), ("c_out_pad", c_int32),
    ]


class ConvEpilogue(Structure):
    _fields_ = [
        ("chan_add", c_void_p), ("step_ptr", c_void_p), ("chan_add_step_stride", c_int64),
        ("residual", c_void_p), ("stats", c_void_p), ("stats_channels", c_int32), ("stats_c0", c_int32),
        ("residual_upsample", c_int32), ("reserved", c_int32),
        ("skip_x", c_void_p), ("skip_w", c_void_p), ("skip_c_in", c_int32), ("skip_planes", c_int32),
        ("skip_plane0", c_int32), ("reserved2", c_int32),
        ("in_norm", c_void_p),
    ]


class WgradDesc(Structure):
    _fields_ = [
        ("batch", c_int32), ("depth", c_int32), ("height", c_int32), ("width", c_int32),
        ("c_in", c_int32), ("c_out", c_int32), ("kernel", c_int32),
        ("a_planes", c_int32), ("a_plane0", c_int32), ("g_planes", c_int32), ("g_plane0", c_int32),
        ("dw_stride_tap", c_int64), ("dw_stride_ci", c_int64), ("dw_stride_co", c_int64), ("c_in_real", c_int32),
        ("a_padded", c_int32), ("g_padded", c_int32),
    ]


class Tensor(Structure):
    """VdmTensor: a window of planes inside a channel-planar buffer."""
    _fields_ = [("data", c_void_p), ("planes", c_int32), ("plane0", c_int32)]


_T = POINTER(Tensor)

_SIGNATURES = {
    "vdm_version": (c_int, []),
    "vdm_last_error_string": (c_char_p, []),
    "vdm_device_supported": (c_int, [c_int]),
    "vdm_conv3d": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, POINTER(ConvEpilogue), c_void_p]),
    "vdm_conv3d_tf32": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, POINTER(ConvEpilogue), c_void_p]),
    "vdm_pack_conv_weight_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vdm_gn_silu_f32": (c_int, [_T, _T, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_float, c_void_p]),
    "vdm_avgpool2_f32": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "vdm_upsample2_f32": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "vdm_pack_input_f32": (c_int, [c_void_p, c_void_p, _T, c_int, c_int64, c_int, c_int, c_void_p]),
    "vdm_conv3d_wgrad": (c_int, [POINTER(WgradDesc), c_void_p, c_void_p, c_void_p, c_void_p]),
    "vdm_pack_conv_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vdm_pack_conv_weight_batched": (c_int, [c_void_p, c_int, c_void_p]),
    "vdm_gn_silu_step": (c_int, [_T, _T, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                 c_float, c_float, c_uint64, c_void_p, c_uint32, c_void_p]),
    "vdm_gn_silu_bwd_reduce": (c_int, [_T, _T, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_float,
                                       c_float, c_uint64, c_void_p, c_uint32, c_void_p, c_int, c_int, c_void_p]),
    "vdm_gn_silu_bwd_apply": (c_int, [_T, _T, _T, _T, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                      c_float, c_float, c_uint64, c_void_p, c_uint32, c_void_p, c_int, c_int, c_void_p,
                                      c_int, c_int, c_void_p]),
    "vdm_adamw_step_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float,
                                   c_float, c_int, c_void_p, c_void_p, c_float, c_float, c_void_p]),
    "vdm_loss_zt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int64, c_void_p]),
    "vdm_loss_zt_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                c_int64, c_void_p]),
    "vdm_loss_terms": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_double, c_void_p, c_void_p,
                               c_int, c_int64, c_void_p]),
    "vdm_loss_dpred": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "vdm_avgpool2_bwd": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "vdm_upsample2_bwd": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "vdm_augment_crop": (c_int, [c_void_p, c_void_p, POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), POINTER(c_int32),
                                 POINTER(c_int32), c_float, c_float, c_float, c_int, c_void_p]),
    "vdm_log_histogram": (c_int, [c_void_p, c_int, c_int64, c_float, c_double, c_double, c_int, c_void_p, c_void_p]),
    "vdm_sumsq": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "vdm_adamw_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_float,
                               c_float, c_int, c_void_p, c_float, c_float, c_void_p]),
    "vdm_channel_stats": (c_int, [_T, c_int, c_int64, c_int, c_void_p, c_int, c_int, c_void_p]),
    "vdm_gn_silu": (c_int, [_T, _T, c_int, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p,
                            c_float, c_float, c_uint64, c_uint32, c_void_p]),
    "vdm_gn_coef": (c_int, [c_void_p, c_int, c_int, c_int, c_int64, c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "vdm_gn_silu_view": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                 c_void_p, c_float, c_int, c_void_p]),
    "vdm_avgpool2": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "vdm_upsample2": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "vdm_pad_circular": (c_int, [_T, _T, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "vdm_pack_input": (c_int, [c_void_p, c_void_p, _T, c_int, c_int64, c_int, c_int, c_void_p]),
    "vdm_sampler_step": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_uint64,
                                 c_void_p, c_int32, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "vdm_philox_normal": (c_int, [c_void_p, c_int, c_int64, c_uint64, c_void_p, c_int32, c_void_p]),
    "vdm_increment": (c_int, [c_void_p, c_void_p]),
    "vdm_pk_work_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int, c_int, c_int]),
    "vdm_pk": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p,
                       c_void_p, c_void_p, c_void_p]),
    "vdm_pk_cross3": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
}

if BRINGUP:
    _SIGNATURES["vdm_debug_set"] = (c_int, [c_int, c_int])

_lib = None


def declared_symbols(header_path: str = HEADER_PATH):
    """Names of every function the public header declares (used by the export test)."""
    text = open(header_path).read()
    return sorted(set(re.findall(r"VDM_API[^;(]*?\b(vdm_\w+)\s*\(", text)))


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C vdm4cdm_b200/csrc`). vdm4cdm_b200 has no CPU or PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(handle, name)   # AttributeError here == the library is stale
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


E_UNSUPPORTED = -2          # VDM_E_UNSUPPORTED


class UnsupportedFusion(RuntimeError):
    """An optional fused form was requested for a layer that cannot take it (VDM_E_UNSUPPORTED); the caller runs the
    unfused launches instead."""


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().vdm_last_error_string().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
