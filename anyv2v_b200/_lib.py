"""ctypes loader for the C-ABI library (include/anyv2v_b200.h).

There is deliberately no fallback: if ``libanyv2v_b200.so`` is missing or a call fails, the product path raises.
Build it with ``python -c "import __graft_entry__ as g; g.build()"`` (nvcc, sm_100a).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_longlong, POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AV2V_LIB") or os.path.join(_HERE, "lib", "libanyv2v_b200.so")  # AV2V_LIB: bring-up builds

AV2V_OK, AV2V_EINVAL, AV2V_EALIGN, AV2V_ECUDA, AV2V_ENOSUP = 0, -1, -2, -3, -4
A_LINEAR, A_CONV3X3, A_TCONV3 = 0, 1, 2
SEQ_ROWS, SEQ_FRAMES = 0, 1


class DdimArgs(Structure):
    _fields_ = [("x", c_void_p), ("v_neg", c_void_p), ("v_edit", c_void_p), ("out", c_void_p), ("n", c_int64),
                ("guidance", c_float), ("ca", c_float), ("cb", c_float), ("cc", c_float), ("cd", c_float),
                ("coef_dev", c_void_p)]


class GroupNormArgs(Structure):
    _fields_ = [("x", c_void_p), ("y", c_void_p), ("gamma", c_void_p), ("beta", c_void_p), ("workspace", c_void_p),
                ("n_samples", c_int32), ("rows", c_int32), ("C", c_int32), ("groups", c_int32), ("eps", c_float),
                ("silu", c_int32), ("x2", c_void_p), ("C1", c_int32)]


class GemmArgs(Structure):
    _fields_ = [("mode", c_int32), ("a", c_void_p), ("w", c_void_p), ("M", c_int32), ("N", c_int32), ("K", c_int32),
                ("lda", c_int32), ("NF", c_int32), ("H", c_int32), ("W", c_int32), ("Cin", c_int32), ("B", c_int32),
                ("rows_per_clip", c_int32), ("HW", c_int32), ("bias", c_void_p), ("rowbias", c_void_p),
                ("rows_per_rowbias", c_int32), ("residual", c_void_p), ("out", c_void_p), ("ldo", c_int32),
                ("n_slots", c_int32), ("slot_stride", c_int64), ("geglu", c_int32), ("stride", c_int32), ("a_channels", c_int32),
                ("a2", c_void_p), ("k_split", c_int32), ("lda2", c_int32), ("up2_phase", c_int32)]


class ConvPlan(Structure):
    _fields_ = [("box_w", c_int32), ("box_h", c_int32), ("frames_per_tile", c_int32), ("tiles_per_frame", c_int32),
                ("m_tiles", c_int32)]


class LayerNormArgs(Structure):
    _fields_ = [("x", c_void_p), ("y", c_void_p), ("gamma", c_void_p), ("beta", c_void_p), ("rows", c_int64),
                ("C", c_int32), ("eps", c_float)]


class AttnArgs(Structure):
    _fields_ = [("seq_mode", c_int32), ("q", c_void_p), ("k", c_void_p), ("v", c_void_p), ("o", c_void_p),
                ("ldq", c_int32), ("ldk", c_int32), ("ldv", c_int32), ("ldo", c_int32), ("batch", c_int32),
                ("seq", c_int32), ("heads", c_int32), ("HW", c_int32), ("n_v", c_int32),
                ("v_branch_stride", c_int64), ("o_branch_stride", c_int64), ("scale", c_float), ("seq_kv", c_int32),
                ("kv_batch_div", c_int32)]


class TAttnFusedArgs(Structure):
    _fields_ = [("x", c_void_p), ("wqkv", c_void_p), ("o", c_void_p), ("ldx", c_int32), ("ldo", c_int32), ("clips", c_int32),
                ("F", c_int32), ("HW", c_int32), ("heads", c_int32), ("Cx", c_int32), ("scale", c_float), ("n_v", c_int32)]


#: every symbol include/anyv2v_b200.h declares -> (restype, argtypes)
EXPORTS = {
    "av2v_abi_version": (c_int, []),
    "av2v_last_error": (c_char_p, []),
    "av2v_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "av2v_ddim_step_cfg_f16": (c_int, [POINTER(DdimArgs), c_void_p]),
    "av2v_ddim_inverse_step_f16": (c_int, [POINTER(DdimArgs), c_void_p]),
    "av2v_groupnorm_workspace_floats": (c_int, [c_int, c_int]),
    "av2v_groupnorm_silu_f16": (c_int, [POINTER(GroupNormArgs), c_void_p]),
    "av2v_gemm_f16": (c_int, [POINTER(GemmArgs), c_void_p]),
    "av2v_conv3x3_plan": (c_int, [POINTER(GemmArgs), POINTER(ConvPlan)]),
    "av2v_layernorm_f16": (c_int, [POINTER(LayerNormArgs), c_void_p]),
    "av2v_attn_pnp_f16": (c_int, [POINTER(AttnArgs), c_void_p]),
    "av2v_tattn_fused_f16": (c_int, [POINTER(TAttnFusedArgs), c_void_p]),
    "av2v_gemm_debug_timers": (c_int, [c_void_p]),  # diagnostics
    "av2v_tmap_cache_stats": (c_int, [POINTER(c_longlong), POINTER(c_longlong), POINTER(c_int)]),  # diagnostics
}

_lib = None


class Av2vError(RuntimeError):
    """Non-zero return code from the C ABI (SURVEY 8b: shims translate codes into RuntimeError)."""


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Av2vError(
                f"{LIB_PATH} not found: the CUDA extension is not built. anyv2v_b200 has no CPU / PyTorch fallback; "
                "run __graft_entry__.build() (needs nvcc).")
        _lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(_lib, name)  # AttributeError if the build lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
    return _lib


def check(rc: int, what: str) -> None:
    if rc != AV2V_OK:
        msg = lib().av2v_last_error()
        raise Av2vError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")
