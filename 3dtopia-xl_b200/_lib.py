"""ctypes binding of libtpx_b200.so (include/tpx.h).  No fallback: if the library or a B200 is missing the
product path raises."""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtpx_b200.so")
_lock = threading.Lock()
_lib = None

DTYPE_F32, DTYPE_F16 = 0, 1
_vp, _i, _f, _sz, _i64 = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_int64


class DitConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("seq_length", "in_channels", "out_channels", "condition_channels", "hidden_size", "depth",
                                         "num_heads", "mlp_hidden")]


class VaeConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("latent_channels", "out_channels", "ch_mid", "ch_out", "attn_heads")]


class VaeEncoderConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("in_channels", "latent_channels", "ch0", "ch1", "attn_heads")]


class SamplerCoefs(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("sqrt_ab", "sqrt_1mab", "sqrt_recip_ab", "sqrt_recipm1_ab", "c_x0", "c_eps", "sigma", "nonzero",
                                         "coef1", "coef2", "min_log", "max_log")] + [("clip", C.c_int32)]


# name -> (restype, argtypes); mirrors include/tpx.h one to one (tests/test_abi.py checks the header against this table)
SIGNATURES = {
    "tpx_version": (_i, []),
    "tpx_last_error": (C.c_char_p, []),
    "tpx_device_check": (_i, []),
    "tpx_launch_count": (_i64, []),
    "tpx_profile_begin": (_i, []),
    "tpx_profile_end": (_i, [C.POINTER(C.c_float), C.POINTER(_i64)]),
    "tpx_dit_create": (_i, [C.POINTER(DitConfig), C.POINTER(_vp)]),
    "tpx_dit_destroy": (None, [_vp]),
    "tpx_dit_set_weight": (_i, [_vp, C.c_char_p, _vp, _i, C.POINTER(_i64), _i, _vp]),
    "tpx_dit_get_weight": (_i, [_vp, C.c_char_p, _vp, _i, _vp]),
    "tpx_dit_finalize": (_i, [_vp, _vp]),
    "tpx_dit_cond_bytes": (_sz, [_vp, _i, _i]),
    "tpx_dit_workspace_bytes": (_sz, [_vp, _i]),
    "tpx_dit_set_cond": (_i, [_vp, _vp, _i, _i, _vp, _sz, _vp]),
    "tpx_dit_forward": (_i, [_vp, _vp, _vp, _i, _i, _f, _vp, _vp, _sz, _vp]),
    "tpx_dit_timesteps_bytes": (_sz, [_vp, _i]),
    "tpx_dit_set_timesteps": (_i, [_vp, C.POINTER(_i64), _i, _vp, _sz, _vp]),
    "tpx_dit_forward_step": (_i, [_vp, _vp, _i64, _i, _i, _f, _vp, _vp, _sz, _vp]),
    "tpx_dit_debug_residual": (_i, [_vp, _vp, _i, _vp, _vp]),
    "tpx_sampler_step": (_i, [_i, _vp, _vp, _i, _vp, _i64, _i, C.POINTER(SamplerCoefs), _vp, _vp, _vp]),
    "tpx_latent_split": (_i, [_vp, _vp, _vp, _f, _i64, _i, _vp, _vp, _vp]),
    "tpx_primvolume_pack": (_i, [_vp, _vp, _i, _i64, _i, _i, _i, _vp, _vp]),
    "tpx_vae_create": (_i, [C.POINTER(VaeConfig), C.POINTER(_vp)]),
    "tpx_vae_destroy": (None, [_vp]),
    "tpx_vae_set_weight": (_i, [_vp, C.c_char_p, _vp, _i, C.POINTER(_i64), _i, _vp]),
    "tpx_vae_finalize": (_i, [_vp, _vp]),
    "tpx_vae_workspace_bytes": (_sz, [_vp, _i]),
    "tpx_vae_decode": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _sz, _vp]),
    "tpx_vae_encoder_create": (_i, [C.POINTER(VaeEncoderConfig), C.POINTER(_vp)]),
    "tpx_vae_encoder_destroy": (None, [_vp]),
    "tpx_vae_encoder_set_weight": (_i, [_vp, C.c_char_p, _vp, _i, C.POINTER(_i64), _i, _vp]),
    "tpx_vae_encoder_finalize": (_i, [_vp, _vp]),
    "tpx_vae_encoder_workspace_bytes": (_sz, [_vp, _i]),
    "tpx_vae_encode": (_i, [_vp, _vp, _i, _vp, _i, _i, _vp, _sz, _vp]),
    "tpx_vae_encode_stage": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "tpx_vae_posterior": (_i, [_vp, _i, _i64, _i64, _i, _vp, _vp, _vp, _vp]),
    "tpx_linear": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _vp]),
    "tpx_linear_gated": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    "tpx_linear_heads": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _i, _vp]),
    "tpx_ln_modulate": (_i, [_vp, _i, _i, _f, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _vp]),
    "tpx_attention": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "tpx_attention_tc": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "tpx_attention_tc_debug": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp, _vp]),
    "tpx_debug_gemm_timeline": (_i, [_vp]),
    "tpx_cfg_combine": (_i, [_vp, _i64, _f, _vp, _vp]),
    "tpx_gelu_erf": (_i, [_vp, _i64, _vp]),
    "tpx_primsdf_query": (_i, [_vp, _vp, _vp, _i64, _i, _i, _i, _i, _vp, _vp]),
    "tpx_raymarch_preview": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _f, _f, _f, _vp, _vp]),
    "tpx_primsdf_grid_bytes": (_sz, [_i64]),
    "tpx_primsdf_grid_build": (_i, [_vp, _i, _vp, _sz, _vp]),
    "tpx_primsdf_query_grid": (_i, [_vp, _vp, _vp, _vp, _sz, _i64, _i, _i, _i, _i, _vp, _vp]),
    "tpx_groupnorm_silu": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp, _vp]),
    "tpx_conv3d_k3": (_i, [_vp, _vp, _vp, _vp, _f, _vp, _i, _i, _i, _i, _vp]),
    "tpx_conv3d_k3_s2": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
}


class TpxError(RuntimeError):
    pass


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen the library and bind every prototype.  Works without a GPU (no compute is issued)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        override = os.environ.get("TPX_LIB_PATH")       # tuning aid: A/B an older build of the library (symbols it lacks are skipped)
        p = path or override or LIB_PATH
        if not os.path.exists(p):
            raise TpxError(f"{p} not found: build it with `python 3dtopia-xl_b200/build.py` (there is no fallback path)")
        lib = C.CDLL(p)
        for name, (res, args) in SIGNATURES.items():
            if override and not path and not hasattr(lib, name):
                continue
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
        return lib


def lib() -> C.CDLL:
    """Library for the compute path: requires CUDA and an sm_100 device."""
    if not torch.cuda.is_available():
        raise TpxError("3dtopia-xl_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
    return load_library()


def check(rc: int, what: str = "") -> int:
    if rc < 0:
        msg = load_library().tpx_last_error()
        raise TpxError(f"{what or 'libtpx_b200'} failed ({rc}): {msg.decode() if msg else ''}")
    return rc


def ptr(t: torch.Tensor | None) -> int | None:
    return None if t is None else t.data_ptr()


def stream_ptr() -> int:
    return torch.cuda.current_stream().cuda_stream


def dtype_tag(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return DTYPE_F32
    if t.dtype == torch.float16:
        return DTYPE_F16
    raise TpxError(f"unsupported tensor dtype {t.dtype} (fp32 / fp16 only)")
