"""ctypes binding of libsdxl_b200.so (the C ABI in include/sdxl_b200.h).

There is deliberately no fallback: if the CUDA library is missing the import of the product path
fails loudly (`SdxlLibraryMissing`), it never routes through the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsdxl_b200.so")

SDXL_MAX_LEVELS = 8


class SdxlLibraryMissing(RuntimeError):
    pass


class SdxlError(RuntimeError):
    pass


class UnetCfg(C.Structure):
    _fields_ = [
        ("adm_in_channels", C.c_int32), ("in_channels", C.c_int32), ("out_channels", C.c_int32),
        ("model_channels", C.c_int32), ("n_levels", C.c_int32), ("channel_mults", C.c_int32 * SDXL_MAX_LEVELS),
        ("n_head_channels", C.c_int32), ("transformer_depths", C.c_int32 * SDXL_MAX_LEVELS),
        ("context_dim", C.c_int32), ("is_refiner", C.c_int32), ("n_steps", C.c_int32),
    ]


class Conditioning(C.Structure):
    _fields_ = [
        ("on_host", C.c_int32), ("n_batch", C.c_int32), ("n_ctx", C.c_int32),
        ("context_full", C.c_void_p), ("context_open_clip", C.c_void_p),
        ("unconditional_context_full", C.c_void_p), ("unconditional_context_open_clip", C.c_void_p),
        ("channel_context", C.c_void_p), ("channel_context_refiner", C.c_void_p),
        ("unconditional_channel_context", C.c_void_p), ("unconditional_channel_context_refiner", C.c_void_p),
        ("resolution", C.c_int32 * 2),
    ]


class VaeCfg(C.Structure):
    _fields_ = [
        ("latent_channels", C.c_int32), ("n_blocks", C.c_int32),
        ("block_in", C.c_int32 * SDXL_MAX_LEVELS), ("block_out", C.c_int32 * SDXL_MAX_LEVELS),
        ("n_group", C.c_int32), ("scale_factor", C.c_double),
        ("n_enc_blocks", C.c_int32), ("enc_in", C.c_int32 * SDXL_MAX_LEVELS), ("enc_out", C.c_int32 * SDXL_MAX_LEVELS),
        ("enc_z_channels", C.c_int32),
    ]


class ClipCfg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_vocab", "n_state", "embed_dim", "n_head", "n_ctx", "n_layer", "quick_gelu")]


# name -> (restype, argtypes); every symbol include/sdxl_b200.h declares
P = C.c_void_p
I = C.c_int
PROTOTYPES = {
    "sdxl_ctx_create": (I, [I, P, C.POINTER(P)]),
    "sdxl_ctx_destroy": (None, [P]),
    "sdxl_last_error": (C.c_char_p, [P]),
    "sdxl_ctx_synchronize": (I, [P]),
    "sdxl_ctx_launch_count": (C.c_uint64, [P]),
    "sdxl_unet_load": (I, [P, C.POINTER(UnetCfg), P, C.c_size_t, I, C.POINTER(P)]),
    "sdxl_unet_destroy": (None, [P]),
    "sdxl_unet_set_conditioning": (I, [P, I, I, P, P]),
    "sdxl_unet_forward": (I, [P, I, I, I, P, C.c_int32, P]),
    "sdxl_unet_forward_f32": (I, [P, I, I, I, P, C.c_int32, P]),
    "sdxl_sample_latent": (I, [P, C.POINTER(Conditioning), C.c_double, I, I, P, P, I, C.c_uint64, P, P, P]),
    "sdxl_sampler_begin": (I, [P, C.POINTER(Conditioning), C.c_double]),
    "sdxl_sampler_step": (I, [P, I, I]),
    "sdxl_sampler_step_host": (I, [P, I, I, P]),
    "sdxl_sampler_set_latent": (I, [P, P, I]),
    "sdxl_sampler_get_latent": (I, [P, P, I]),
    "sdxl_unet_alpha": (C.c_double, [P, I]),
    "sdxl_unet_load_broadcast": (I, [P, C.POINTER(UnetCfg), P, C.c_size_t, I, P, I, I, C.POINTER(P)]),
    "sdxl_unet_plan_flops": (C.c_double, [P]),
    "sdxl_unet_plan_num_ops": (I, [P]),
    "sdxl_unet_plan_flops_executed": (C.c_double, [P]),
    "sdxl_unet_profile_plan": (I, [P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "sdxl_unet_profile_dump": (I, [P, C.c_char_p]),
    "sdxl_dbg_igemm_timeline": (I, [P, I, I, I, I, I, C.POINTER(C.c_uint64)]),
    "sdxl_dbg_igemm_gaps": (I, [P, I, I, I, I, I, C.POINTER(C.c_int64)]),
    "sdxl_dbg_attention_timeline": (I, [P, I, I, I, I, C.POINTER(C.c_longlong)]),
    "sdxl_dbg_plan_gemm": (I, [P, I, P, C.c_size_t, I, I, I, I, I, I, P, P, P, I, I, P, P, I, C.POINTER(C.c_int32), I]),
    "sdxl_dbg_plan_group_norm": (I, [P, P, C.c_size_t, P, I, P, I, I, I, I, P, P, P]),
    "sdxl_dbg_plan_attention": (I, [P, I, P, I, I, P, I, I, I, I, I, I, I, P, I, P, I]),
    "sdxl_dbg_plan_vae_attention": (I, [P, P, P, P, I, I, P, P, P, P, C.POINTER(C.c_int32), I]),
    "sdxl_randn": (I, [P, P, C.c_size_t, C.c_uint64, C.c_uint64]),
    "sdxl_qkv_attention": (I, [P, P, P, P, P, I, I, I, I, I, P]),
    "sdxl_op_linear": (I, [P, P, P, P, P, I, I, I, I, I, P]),
    "sdxl_op_conv2d": (I, [P, P, P, P, I, I, I, I, I, I, I, I, P]),
    "sdxl_op_group_norm": (I, [P, P, I, P, I, I, I, I, P, P, C.c_float, I, P]),
    "sdxl_op_layer_norm": (I, [P, P, P, P, C.c_float, I, I, P]),
    "sdxl_op_timestep_embedding": (I, [P, P, I, I, I, P]),
    "sdxl_vae_load": (I, [P, C.POINTER(VaeCfg), P, C.c_size_t, I, C.POINTER(P)]),
    "sdxl_vae_destroy": (None, [P]),
    "sdxl_vae_decode_latent": (I, [P, I, I, I, P, I, P]),
    "sdxl_vae_latent_to_image": (I, [P, I, I, I, P, I, P]),
    "sdxl_vae_encode_image": (I, [P, I, I, I, P, I, P]),
    "sdxl_vae_image_to_latent": (I, [P, I, I, I, P, I, P]),
    "sdxl_vae_encode_plan_flops": (C.c_double, [P]),
    "sdxl_vae_plan_flops": (C.c_double, [P]),
    "sdxl_vae_profile_plan": (I, [P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "sdxl_vae_profile_dump": (I, [P, C.c_char_p]),
    "sdxl_tokenizer_last_error": (C.c_char_p, []),
    "sdxl_tokenizer_create_clip": (I, [C.c_char_p, C.POINTER(P)]),
    "sdxl_tokenizer_create_open_clip": (I, [C.c_char_p, C.c_char_p, C.POINTER(P)]),
    "sdxl_tokenizer_destroy": (None, [P]),
    "sdxl_tokenizer_encode": (I, [P, C.c_char_p, I, I, C.POINTER(C.c_uint32), I, C.POINTER(I)]),
    "sdxl_tokenizer_decode": (I, [P, C.POINTER(C.c_uint32), I, C.c_char_p, I, C.POINTER(I)]),
    "sdxl_tokenize_text": (I, [P, C.c_char_p, I, C.POINTER(C.c_int32)]),
    "sdxl_tokenizer_special": (I, [P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "sdxl_clip_load": (I, [P, C.POINTER(ClipCfg), P, C.c_size_t, I, C.POINTER(P)]),
    "sdxl_clip_destroy": (None, [P]),
    "sdxl_clip_forward_hidden": (I, [P, I, C.POINTER(C.c_int32), I, P, I]),
    "sdxl_clip_forward_hidden_pooled": (I, [P, I, C.POINTER(C.c_int32), I, P, P, I]),
    "sdxl_clip_plan_flops": (C.c_double, [P]),
    "sdxl_make_inpaint_mask": (I, [I, I, I, I, I, I, I, I, I, I, P]),
    "sdxl_mpk_decode_u16": (I, [P, C.c_size_t, C.c_size_t, P, C.POINTER(C.c_size_t)]),
    "sdxl_mpk_encode_u16": (C.c_size_t, [P, C.c_size_t, P]),
}

PROFILE_KINDS = 24   # SDXL_PROFILE_KINDS (include/sdxl_b200.h)
_lib = None


def load() -> C.CDLL:
    """dlopen the library and bind every prototype. Works without a GPU (no CUDA call is made)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SdxlLibraryMissing(
            f"{LIB_PATH} not found: build it with `python stable-diffusion-xl-burn_b200/build.py` "
            "(or __graft_entry__.build()). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
