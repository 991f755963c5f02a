"""ctypes binding of the C ABI declared in include/sdb200.h (the drop-in boundary).

The library is loaded from the in-tree build (csrc/libsdb200.so). There is NO fallback: if the library is
missing, importing the ops fails loudly.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_LIB_PATH = Path(__file__).resolve().parent / "csrc" / "libsdb200.so"

ACT_NONE, ACT_GEGLU, ACT_QUICK_GELU, ACT_SILU = 0, 1, 2, 3


class GemmDesc(C.Structure):
    _fields_ = [
        ("a0", C.c_void_p), ("a1", C.c_void_p), ("a2", C.c_void_p), ("a3", C.c_void_p),
        ("c0", C.c_int32), ("c1", C.c_int32), ("c2", C.c_int32), ("c3", C.c_int32),
        ("nb", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
        ("taps", C.c_int32),
        ("b", C.c_void_p),
        ("n", C.c_int32),
        ("alpha", C.c_float),
        ("bias", C.c_void_p),
        ("film", C.c_void_p),
        ("ldf", C.c_int32),
        ("rows_per_sample", C.c_int32),
        ("residual", C.c_void_p),
        ("ldr", C.c_int32),
        ("act", C.c_int32),
        ("out_f16", C.c_void_p),
        ("out_f16_lo", C.c_void_p),
        ("out_f32", C.c_void_p),
        ("ldo", C.c_int32),
        ("block_n", C.c_int32),
        ("splits", C.c_int32),
        ("workspace", C.c_void_p),
        ("workspace_floats", C.c_int64),
        ("stats_out", C.c_void_p),
        ("b_dynamic", C.c_int32),
        ("conv_stride", C.c_int32),
        ("conv_shift", C.c_int32),
        ("in_h", C.c_int32),
        ("in_w", C.c_int32),
        ("pair", C.c_int32),
        ("splitk_mode", C.c_int32),
        ("stats_group", C.c_int32),
    ]


class AttnDesc(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("vt", C.c_void_p), ("out", C.c_void_p),
        ("batch", C.c_int32), ("heads", C.c_int32), ("nq", C.c_int32), ("nkv", C.c_int32),
        ("d", C.c_int32), ("dpad", C.c_int32),
        ("ldq", C.c_int32), ("ldk", C.c_int32), ("ldvt", C.c_int32), ("ldo", C.c_int32),
        ("q_batch_stride", C.c_int64), ("k_batch_stride", C.c_int64),
        ("vt_batch_stride", C.c_int64), ("o_batch_stride", C.c_int64),
        ("scale", C.c_float), ("causal", C.c_int32),
    ]


class PlmsDesc(C.Structure):
    _fields_ = [
        ("unet", C.c_void_p), ("x", C.c_void_p), ("x_out", C.c_void_p), ("pred_x0_out", C.c_void_p), ("work", C.c_void_p),
        ("batch", C.c_int32), ("n_steps", C.c_int32), ("guided", C.c_int32), ("scale", C.c_float),
        ("timesteps", C.POINTER(C.c_float)), ("alphas", C.POINTER(C.c_float)), ("alphas_prev", C.POINTER(C.c_float)),
        ("sqrt_one_minus_alphas", C.POINTER(C.c_float)), ("sigmas", C.POINTER(C.c_float)),
    ]


_P, _I, _L, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float

# name -> argtypes; every symbol declared in include/sdb200.h must appear here (tests check both ways).
SIGNATURES = {
    "sdb_last_error": ([], C.c_char_p),
    "sdb_version": ([], C.c_int),
    "sdb_sm_count": ([], C.c_int),
    "sdb_launch_count": ([], C.c_longlong),
    "sdb_debug_trace": ([_P, _L], C.c_longlong),
    "sdb_gemm": ([C.POINTER(GemmDesc), _P], C.c_int),
    "sdb_gemm_plan": ([C.POINTER(GemmDesc), C.POINTER(C.c_int32)], C.c_int),
    "sdb_attention": ([C.POINTER(AttnDesc), _P], C.c_int),
    "sdb_groupnorm": ([_P, _P, _I, _I, _I, _I, _I, _P, _P, _F, _I, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _P], C.c_int),
    "sdb_layernorm": ([_P, _I, _I, _P, _P, _F, _P, _P, _P], C.c_int),
    "sdb_softmax_rows": ([_P, _I, _I, _F, _P, _P], C.c_int),
    "sdb_nchw_to_nhwc": ([_P, _I, _I, _I, _P, _P, _P], C.c_int),
    "sdb_nhwc_to_nchw": ([_P, _I, _I, _I, _P, _P], C.c_int),
    "sdb_im2col3x3": ([_P, _I, _I, _I, _I, _I, _P, _P], C.c_int),
    "sdb_upsample2x": ([_P, _I, _I, _I, _I, _P, _P], C.c_int),
    "sdb_cast_f16": ([_P, _L, _P, _P], C.c_int),
    "sdb_transpose_f16": ([_P, _I, _I, _I, _I, _P, _I, _P], C.c_int),
    "sdb_timestep_embedding_f32": ([_P, _I, _I, _F, _P, _P], C.c_int),
    "sdb_linear_small": ([_P, _I, _I, _P, _I, _P, _I, _P, _P, _P], C.c_int),
    "sdb_sampler_step": ([_P, _P, _P, _I, _F, _I, _P, _P, _P, _P, _F, _F, _F, _F, _L, _P, _P, _P, _P, _P], C.c_int),
    "sdb_vae_sample": ([_P, _P, _I, _I, _F, _P, _P], C.c_int),
    "sdb_to_uint8": ([_P, _L, _P, _P], C.c_int),
    "sdb_axpby": ([_P, _F, _F, _L, _P, _P], C.c_int),
    "sdb_pointwise_small": ([_P, _L, _I, _I, _P, _P, _F, _P, _P], C.c_int),
    "sdb_embed_tokens": ([_P, _I, _I, _I, _I, _P, _P, _P, _P], C.c_int),
    "sdb_dpm_solver_step": ([_P, _P, _P, _I, _F, _F, _F, _I, _P, _F, _F, _F, _L, _P, _P, _P, _P], C.c_int),
    "sdb_mask_blend": ([_P, _P, _I, _I, _I, _L, _P, _P, _P], C.c_int),
    "sdb_axpby2": ([_P, _P, _F, _F, _L, _P, _P], C.c_int),
    # post-processing (safety.cu)
    "sdb_resample_u8": ([_P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _I, _P, _P], C.c_int),
    "sdb_clip_normalize": ([_P, _I, _I, _I, _I, _F, _F, _F, _F, _F, _F, _P, _P], C.c_int),
    "sdb_patchify": ([_P, _I, _I, _I, _I, _P, _P], C.c_int),
    "sdb_safety_scores": ([_P, _I, _I, _P, _P, _I, _P, _P, _I, _P, _P, _P], C.c_int),
    "sdb_blank_flagged": ([_P, _L, _I, _P, _P], C.c_int),
    "sdb_watermark_dwtdct": ([_P, _I, _I, _I, _P, _I, _F, _P, _P, _P], C.c_int),
    # handle level (plan.cu)
    "sdb_plan_begin": ([C.POINTER(C.c_void_p)], C.c_int),
    "sdb_plan_end": ([_P], C.c_int),
    "sdb_plan_size": ([_P], C.c_int),
    "sdb_plan_launch": ([_P, _P], C.c_int),
    "sdb_plan_destroy": ([_P], C.c_int),
    "sdb_fill_f32": ([_P, _L, _F, _P], C.c_int),
    "sdb_unet_create": ([_P, _P, _P, _P, _I, _I, _I, _I, _I, C.POINTER(C.c_void_p)], C.c_int),
    "sdb_unet_forward": ([_P, _P, _P, _P, _P], C.c_int),
    "sdb_unet_destroy": ([_P], C.c_int),
    "sdb_sample_plms": ([C.POINTER(PlmsDesc), _P], C.c_int),
}

_lib = None


def load() -> C.CDLL:
    """Load libsdb200.so (built by build.py / __graft_entry__.build()). Raises if it is missing."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise RuntimeError(
                f"{_LIB_PATH} is missing: build it with `python stable-diffusion_b200/build.py` "
                "(there is no CPU or PyTorch fallback for the sdb200 kernels)")
        lib = C.CDLL(str(_LIB_PATH))
        for name, (argtypes, restype) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = lib
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().sdb_last_error()
        raise RuntimeError(f"{what} failed ({rc}): {msg.decode() if msg else '?'}")
