"""ctypes loader for libpaella_b200.so (the C ABI declared in include/paella_b200.h).

There is no fallback: if the library is missing, or an entry point reports an error, this raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char, c_char_p, c_double, c_float, c_int, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpaella_b200.so")

PB200_MAX_LEVELS = 4

EPI_F16, EPI_F32, EPI_GELU_F16, EPI_RESID_F32, EPI_UNPATCH_F32, EPI_NCHW_F32, EPI_RESID_LN_F32, EPI_F16_LN = range(8)


class GemmEpilogue(ctypes.Structure):
    _fields_ = [
        ("mode", c_int), ("bias", c_void_p), ("out", c_void_p), ("ldo", c_int64), ("resid", c_void_p),
        ("ldr", c_int64), ("alpha", c_float), ("sqsum", c_void_p), ("rows_per_sample", c_int), ("film", c_void_p),
        ("film_ld", c_int64), ("film_off", c_int64), ("remap_in", c_int), ("remap_out", c_int), ("up_h", c_int),
        ("up_w", c_int), ("up_cout", c_int), ("out16", c_void_p), ("ln_stat", c_void_p), ("ln_wsum", c_void_p),
        ("ln_c", c_int), ("ln_shift", c_void_p), ("ln_mean_out", c_void_p), ("a_scale", c_void_p), ("a_scale_ld", c_int64),
    ]


class PaellaConfig(ctypes.Structure):
    _fields_ = [
        ("c_in", c_int), ("c_out", c_int), ("num_labels", c_int), ("c_r", c_int), ("patch_size", c_int),
        ("c_cond", c_int), ("n_levels", c_int), ("c_hidden", c_int * PB200_MAX_LEVELS),
        ("nhead", c_int * PB200_MAX_LEVELS), ("blocks", c_int * PB200_MAX_LEVELS),
        ("level_config", (c_char * 8) * PB200_MAX_LEVELS), ("clip_embd", c_int), ("byt5_embd", c_int),
        ("clip_seq_len", c_int), ("kernel_size", c_int), ("self_attn", c_int),
    ]


class Cond(ctypes.Structure):
    _fields_ = [("byt5", c_void_p), ("byt5_len", c_int), ("clip", c_void_p), ("clip_image", c_void_p),
                ("n_clip_image", c_int)]


class VqganConfig(ctypes.Structure):
    _fields_ = [("levels", c_int), ("bottleneck_blocks", c_int), ("c_hidden", c_int), ("c_latent", c_int),
                ("codebook_size", c_int), ("scale_factor", c_float)]


# name -> (restype, argtypes); mirrors include/paella_b200.h one to one
SIGNATURES = {
    "pb200_last_error": (c_char_p, []),
    "pb200_abi_version": (c_int, []),
    "pb200_device_info": (c_int, [POINTER(c_int), POINTER(c_int)]),
    "pb200_launch_count": (ctypes.c_longlong, []),
    "pb200_profile_enable": (c_int, [c_int]),
    "pb200_profile_report": (c_int, [c_char_p, ctypes.c_longlong]),
    "pb200_philox_offset_increment": (c_int64, [c_int64]),
    "pb200_randint": (c_int, [c_void_p, c_int64, c_int64, c_uint64, c_uint64, c_void_p]),
    "pb200_rand": (c_int, [c_void_p, c_int64, c_uint64, c_uint64, c_void_p]),
    "pb200_multinomial": (c_int, [c_void_p, c_int64, c_int64, c_uint64, c_uint64, c_void_p, c_void_p]),
    "pb200_resample_logits": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_double, c_double, c_int,
                                      c_uint64, c_uint64, c_void_p, c_void_p]),
    "pb200_resample_quant": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_double, c_double, c_void_p, c_int,
                                     c_void_p, c_void_p]),
    "pb200_add_noise": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_uint64, c_uint64, c_void_p,
                                c_void_p, c_void_p]),
    "pb200_vq_nearest": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "pb200_vq_gather": (c_int, [c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "pb200_gemm_f16": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64,
                               POINTER(GemmEpilogue), c_void_p]),
    "pb200_gemm_plan": (c_int, [c_int64, c_int64, c_int64, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "pb200_layernorm": (c_int, [c_void_p, c_int64, c_int, ctypes.c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pb200_nchw_to_nhwc": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "pb200_nhwc_to_nchw": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "pb200_cast_f16": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "pb200_dwconv_ln": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "pb200_grn_f16": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pb200_grn_f32": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pb200_film_apply": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_int64, c_int64, c_void_p]),
    "pb200_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                c_int, c_int, c_void_p]),
    "pb200_paella_create": (c_int, [POINTER(PaellaConfig), POINTER(c_void_p)]),
    "pb200_paella_destroy": (None, [c_void_p]),
    "pb200_paella_weight_bytes": (c_int64, [c_void_p]),
    "pb200_paella_bind_weights": (c_int, [c_void_p, c_void_p]),
    "pb200_paella_num_params": (c_int, [c_void_p]),
    "pb200_paella_param_name": (c_char_p, [c_void_p, c_int]),
    "pb200_paella_param_numel": (c_int64, [c_void_p, c_int]),
    "pb200_paella_load_param": (c_int, [c_void_p, c_char_p, c_void_p, c_int64, c_void_p]),
    "pb200_paella_workspace_bytes": (c_int64, [c_void_p, c_int, c_int, c_int, c_int]),
    "pb200_paella_cond_cache_bytes": (c_int64, [c_void_p, c_int, c_int]),
    "pb200_paella_prepare_cond": (c_int, [c_void_p, POINTER(Cond), c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                          c_int64, c_void_p]),
    "pb200_paella_r_embedding": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "pb200_paella_c_embeddings": (c_int, [c_void_p, POINTER(Cond), c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "pb200_paella_features": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                      c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "pb200_paella_logits": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "pb200_paella_sample_tokens": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_double, c_uint64,
                                           c_uint64, c_void_p, c_void_p, c_int64, c_void_p]),
    "pb200_paella_sample_tokens_masked": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_double, c_uint64,
                                                  c_uint64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "pb200_vqgan_create": (c_int, [POINTER(VqganConfig), POINTER(c_void_p)]),
    "pb200_vqgan_destroy": (None, [c_void_p]),
    "pb200_vqgan_weight_bytes": (c_int64, [c_void_p]),
    "pb200_vqgan_bind_weights": (c_int, [c_void_p, c_void_p]),
    "pb200_vqgan_num_params": (c_int, [c_void_p]),
    "pb200_vqgan_param_name": (c_char_p, [c_void_p, c_int]),
    "pb200_vqgan_param_numel": (c_int64, [c_void_p, c_int]),
    "pb200_vqgan_load_param": (c_int, [c_void_p, c_char_p, c_void_p, c_int64, c_void_p]),
    "pb200_vqgan_workspace_bytes": (c_int64, [c_void_p, c_int, c_int, c_int]),
    "pb200_vqgan_encode": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int64, c_void_p]),
    "pb200_vqgan_decode": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int64,
                                   c_void_p]),
    "pb200_vqgan_decode_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int64,
                                      c_void_p]),
    "pb200_vqgan_decode_composite": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                             c_void_p, c_int64, c_void_p]),
    "pb200_vqgan_sync_params": (c_int, [c_void_p, c_void_p]),
    "pb200_vq_mlp_fused": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p]),
    "pb200_vqgan_resblock_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int]),
    "pb200_vqgan_resblock": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, POINTER(c_float), c_void_p, c_int64, c_void_p]),
}

IMG_F32_NCHW, IMG_F32_NCHW_CLAMP01, IMG_U8_NHWC = range(3)

_lib = None


class PaellaB200Error(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Load the shared library once; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PaellaB200Error(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C paella_b200/csrc`). paella_b200 has no CPU or PyTorch fallback.")
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)        # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        if l.pb200_abi_version() != 2:
            raise PaellaB200Error("libpaella_b200.so ABI version mismatch")
        _lib = l
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().pb200_last_error()
        raise PaellaB200Error(f"{what}: {msg.decode() if msg else 'unknown error'}")


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL).  CPU tensors are refused: no CPU path exists."""
    if t is None:
        return None
    if not t.is_cuda:
        raise PaellaB200Error("paella_b200 runs on CUDA tensors only (got a CPU tensor); there is no CPU fallback")
    if not t.is_contiguous():
        raise PaellaB200Error("paella_b200 expects contiguous tensors at the C boundary")
    return c_void_p(t.data_ptr())


def current_stream():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
