"""ctypes binding of libmedimgen_b200.so (the C ABI declared in include/medimgen_b200.h).

There is NO fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
PyTorch is only used by the callers for device memory and streams; pointers cross as integers.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmedimgen_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "medimgen_b200.h")

F32, BF16 = 0, 1
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TC = 0, 1, 2


class ConvGeom(C.Structure):
    _fields_ = [("N", C.c_int32), ("in_dims", C.c_int32 * 3), ("out_dims", C.c_int32 * 3), ("Cin", C.c_int32),
                ("Cout", C.c_int32), ("ksize", C.c_int32 * 3), ("stride", C.c_int32 * 3), ("pad", C.c_int32 * 3)]


class GemmDesc(C.Structure):
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("batch_outer", C.c_int32),
                ("batch_inner", C.c_int32),
                ("a_m", C.c_int64), ("a_k", C.c_int64), ("a_outer", C.c_int64), ("a_inner", C.c_int64),
                ("b_k", C.c_int64), ("b_n", C.c_int64), ("b_outer", C.c_int64), ("b_inner", C.c_int64),
                ("c_m", C.c_int64), ("c_n", C.c_int64), ("c_outer", C.c_int64), ("c_inner", C.c_int64),
                ("alpha", C.c_float), ("accumulate", C.c_int32)]


_p, _i, _l, _f = C.c_void_p, C.c_int32, C.c_int64, C.c_float
_I3 = C.c_int32 * 3

# name -> argtypes (restype is int unless listed in _RESTYPES)
_SIGNATURES = {
    "mig_last_error": [],
    "mig_abi_version": [],
    "mig_has_tcgen05": [],
    "mig_conv_fwd": [C.POINTER(ConvGeom), _i, _p, _p, _p, _p, _p, _p, _i, _p, _l, _p],
    "mig_conv_fwd_stats": [C.POINTER(ConvGeom), _i, _p, _p, _p, _p, _p, _p, _p, _i, _i, _p, _l, _p],
    "mig_conv_fwd_stats_in_epilogue": [C.POINTER(ConvGeom), _i, _i, _i, _l],
    "mig_conv_dgrad": [C.POINTER(ConvGeom), _i, _p, _p, _p, _i, _p, _l, _p],
    "mig_conv_wgrad": [C.POINTER(ConvGeom), _i, _p, _p, _p, _p, _i, _p, _l, _p],
    "mig_conv_workspace_bytes": [C.POINTER(ConvGeom), _i, _i, _i],
    "mig_gemm_strided": [C.POINTER(GemmDesc), _i, _i, _p, _p, _p, _i, _p],
    "mig_flash_attention_fwd": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p],
    "mig_flash_attention_fwd_ld": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _l, _l, _l, _f, _p],
    "mig_flash_attention_bwd": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _f, _p],
    "mig_groupnorm_fwd": [_i, _p, _p, _p, _p, _p, _p, _i, _l, _i, _i, _f, _i, _p, _l, _p],
    "mig_groupnorm_bwd": [_i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i, _i, _l, _i, _i, _i, _p, _l, _p],
    "mig_groupnorm_can_split": [_i, _i, _l, _i, _i],
    "mig_groupnorm_stats": [_i, _p, _p, _i, _l, _i, _i, _p],
    "mig_groupnorm_apply": [_i, _p, _p, _p, _p, _p, _p, _p, _i, _l, _i, _i, _f, _i, _p],
    "mig_groupnorm_workspace_bytes": [_i, _l, _i, _i],
    "mig_layernorm_fwd": [_i, _p, _p, _p, _p, _p, _p, _l, _i, _f, _p],
    "mig_layernorm_bwd": [_i, _p, _p, _p, _p, _p, _p, _p, _p, _l, _i, _p],
    "mig_silu_fwd": [_i, _p, _p, _l, _p],
    "mig_silu_bwd": [_i, _p, _p, _p, _l, _p],
    "mig_add": [_i, _p, _p, _p, _l, _p],
    "mig_scale": [_i, _p, _p, _f, _l, _p],
    "mig_mul": [_i, _p, _p, _p, _l, _p],
    "mig_addcmul": [_i, _p, _p, _p, _p, _l, _p],
    "mig_cast": [_i, _i, _p, _p, _l, _p],
    "mig_geglu_fwd": [_i, _p, _p, _l, _i, _p],
    "mig_geglu_bwd": [_i, _p, _p, _p, _l, _i, _p],
    "mig_concat_channels": [_i, _p, _p, _p, _l, _i, _i, _p],
    "mig_split_channels": [_i, _p, _p, _p, _l, _i, _i, _p],
    "mig_upsample_nearest_fwd": [_i, _p, _p, _i, _I3, _I3, _i, _p],
    "mig_upsample_nearest_bwd": [_i, _p, _p, _i, _I3, _I3, _i, _p],
    "mig_avgpool_fwd": [_i, _p, _p, _i, _I3, _I3, _I3, _i, _p],
    "mig_avgpool_bwd": [_i, _p, _p, _i, _I3, _I3, _I3, _i, _p],
    "mig_nchw_to_nhwc": [_i, _i, _p, _p, _i, _i, _l, _p],
    "mig_nhwc_to_nchw": [_i, _i, _p, _p, _i, _i, _l, _p],
    "mig_colsum": [_i, _p, _p, _l, _i, _i, _p],
    "mig_add_channel_bias": [_i, _p, _p, _p, _l, _i, _p],
    "mig_chan_bias_bwd": [_i, _p, _p, _i, _l, _i, _p],
    "mig_softmax_fwd": [_i, _i, _p, _p, _l, _i, _f, _p],
    "mig_softmax_bwd": [_i, _i, _p, _p, _p, _l, _i, _f, _p],
    "mig_softmax_bwd_narrow": [_p, _p, _p, _l, _i, _f, _p],
    "mig_temb_proj_all_fwd": [_p, _p, _p, _p, _p, _i, _i, _i, _p],
    "mig_temb_proj_all_bwd": [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p],
    "mig_timestep_embedding": [_p, _p, _i, _i, _i, _f, _p],
    "mig_ddpm_add_noise": [_i, _p, _p, _p, _p, _p, _i, _l, _i, _i, _p],
    "mig_ddpm_step": [_i, _p, _p, _p, _p, _p, _l, _f, _f, _f, _f, _f, _i, _i, _p],
    "mig_ddim_step": [_i, _p, _p, _p, _p, _p, _l, _f, _f, _f, _f, _f, _i, _i, _p],
    "mig_mse_fwd": [_i, _p, _p, _p, _p, _l, _i, _p],
    "mig_mse_bwd": [_i, _p, _p, _p, _p, _l, _i, _p],
    "mig_kl_fwd": [_i, _p, _p, _p, _p, _l, _i, _p],
    "mig_kl_bwd": [_i, _p, _p, _p, _p, _p, _l, _i, _p],
    "mig_vae_sample_fwd": [_i, _p, _p, _p, _p, _p, _l, _p],
    "mig_vae_sample_bwd": [_i, _p, _p, _p, _p, _p, _p, _p, _l, _p],
    "mig_sumsq": [_p, _p, _p, _l, _p],
    "mig_adamw_step": [_p, _p, _p, _p, _l, _f, _f, _f, _f, _f, _i, _p, _f, _p, _p, _p],
    "mig_sumsq_strided": [_p, _p, _p, _l, _l, _l, _p],
    "mig_adamw_step_strided": [_p, _p, _p, _p, _l, _l, _l, _f, _f, _f, _f, _f, _i, _p, _f, _p, _p, _p],
    "mig_patch_gather": [_p, _p, _p, _i, _i, _i, _I3, _i, _i, _f, _f, _f, _p],
    "mig_patch_stats": [_p, _p, _p, _i, _l, _p, _l, _p],
    "mig_patch_stats_workspace_bytes": [_i],
    "mig_patch_intensity": [_p, _p, _i, _p, _p, _p, _i, _i, _l, _i, _f, _f, _p],
    "mig_upconv_folded_elems": [_i, _i, _I3, _I3, _I3, _i],
    "mig_upconv_fold_filter": [_p, _p, _i, _i, _I3, _I3, _I3, _i, _p],
    "mig_upconv_fwd_direct_ok": [_i, _I3, _i, _i],
    "mig_upconv_fwd": [_p, _p, _p, _p, _i, _I3, _i, _i, _I3, _I3, _I3, _p],
    "mig_upconv_unfold_wgrad": [_p, _p, _i, _i, _I3, _I3, _I3, _p],
    "mig_class_interleave": [_i, _p, _p, _i, _I3, _I3, _i, _i, _p],
}
_RESTYPES = {"mig_last_error": C.c_char_p, "mig_conv_workspace_bytes": C.c_int64,
             "mig_groupnorm_workspace_bytes": C.c_int64, "mig_patch_stats_workspace_bytes": C.c_int64,
             "mig_upconv_folded_elems": C.c_int64}

_lib = None


def declared_symbols() -> list[str]:
    """Every function name declared in include/medimgen_b200.h."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mig_[a-z0-9_]+)\s*\(", text)) - {"mig_conv_geom", "mig_gemm_desc", "mig_patch_desc"})


def load():
    """Load (once) and type the shared library. Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built. Run "
            "`python -m medical_image_generation_b200.build` (there is no CPU / PyTorch fallback).")
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.argtypes = argtypes
        fn.restype = _RESTYPES.get(name, C.c_int)
    if lib.mig_abi_version() != 4:
        raise RuntimeError("libmedimgen_b200.so ABI version mismatch")
    _lib = lib
    return lib


launch_count = 0  # kernels-launching ABI calls made through `call` (bench.py reports it)


def call(name: str, *args):
    """Invoke an int-status entry point; raise RuntimeError(mig_last_error()) on failure."""
    global launch_count
    lib = load()
    rc = getattr(lib, name)(*args)
    launch_count += 1
    if rc != 0:
        raise RuntimeError(f"{name} failed ({rc}): {lib.mig_last_error().decode()}")


def conv_geom(N, in_dims, out_dims, Cin, Cout, ksize, stride, pad) -> ConvGeom:
    g = ConvGeom()
    g.N, g.Cin, g.Cout = N, Cin, Cout
    g.in_dims, g.out_dims = _I3(*in_dims), _I3(*out_dims)
    g.ksize, g.stride, g.pad = _I3(*ksize), _I3(*stride), _I3(*pad)
    return g
