"""ctypes binding of libtld_b200.so (C ABI in include/tld_b200.h).

The library is the product path: if it is missing or cannot be loaded every compute entry point of this
package raises.  There is no PyTorch/CPU fallback anywhere in the package.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtld_b200.so")

_lock = threading.Lock()
_lib = None


class TldConfig(C.Structure):
    """struct tld_config (include/tld_b200.h)"""

    _fields_ = [
        ("image_size", C.c_int32), ("noise_embed_dims", C.c_int32), ("patch_size", C.c_int32),
        ("embed_dim", C.c_int32), ("n_layers", C.c_int32), ("text_emb_size", C.c_int32),
        ("mlp_multiplier", C.c_int32), ("n_channels", C.c_int32), ("dropout", C.c_float),
    ]


# name -> (restype, argtypes); must list every symbol declared in include/tld_b200.h
PROTOTYPES = {
    "tld_last_error": (C.c_char_p, []),
    "tld_version": (C.c_int, []),
    "tld_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "tld_denoiser_create": (C.c_int, [C.POINTER(TldConfig), C.c_int, C.POINTER(C.c_void_p)]),
    "tld_denoiser_destroy": (None, [C.c_void_p]),
    "tld_denoiser_set_param": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "tld_denoiser_set_params_async": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_void_p),
                                                C.POINTER(C.c_int64), C.c_void_p]),
    "tld_denoiser_missing_params": (C.c_int, [C.c_void_p]),
    "tld_forward_serial": (C.c_longlong, [C.c_void_p]),
    "tld_denoiser_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                       C.c_void_p]),
    "tld_sampler_generate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                       C.POINTER(C.c_double), C.c_int, C.c_float, C.c_float, C.c_float, C.c_int,
                                       C.c_void_p]),
    "tld_sampler_edit": (C.c_int, [C.c_void_p] * 6 + [C.c_int, C.POINTER(C.c_double), C.c_int, C.c_int, C.c_float, C.c_int,
                                                    C.c_void_p]),
    "tld_sampler_last_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int64)]),
    "tld_op_gemm": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                              C.c_void_p]),
    "tld_op_gemm_nn": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tld_op_gemm_mn": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tld_op_gemm_xattn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_void_p]),
    "tld_op_gemm_lnfold": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int, C.c_void_p]),
    "tld_op_gemm_bias_resid_lnp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "tld_op_gemm_xattn_lnp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "tld_op_rowstats_cast": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tld_op_ln_fold_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_int, C.c_void_p]),
    "tld_op_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tld_op_self_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_op_ln_xattn_ln": (C.c_int, [C.c_void_p] * 8 + [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tld_op_qkv_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_vae_group_norm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "tld_vae_add_bias": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]),
    "tld_vae_conv3x3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p]),
    "tld_vae_conv3x3_fused": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p]),
    "tld_vae_group_norm_from_conv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                               C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]),
    "tld_vae_attention_core": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_vae_conv_out3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_vae_upsample2x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_latent_quantize": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_float, C.c_void_p]),
    "tld_latent_dequantize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_float, C.c_void_p]),
    "tld_image_grid_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p]),
    "tld_clip_embed": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_clip_causal_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_clip_quick_gelu": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "tld_clip_final": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_void_p]),
    "tld_train_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "tld_train_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "tld_train_get_grad": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "tld_train_grad_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                        C.c_int]),
    "tld_train_prepare": (C.c_int, [C.c_void_p]),
    "tld_train_wait_grad": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "tld_train_grad_offset": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "tld_adam_ema_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_double,
                                    C.c_double, C.c_double, C.c_double, C.c_int64, C.c_double, C.c_double, C.c_void_p]),
    "tld_bwd_cast_transpose": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tld_bwd_colsum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tld_bwd_layernorm": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                    C.c_void_p]),
    "tld_bwd_dwconv_gelu": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_bwd_xattn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                C.c_int, C.c_int, C.c_void_p]),
    "tld_bwd_self_attention": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p]),
    "tld_op_gemm_up_dwconv_gelu": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "tld_op_dwconv_gelu": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p]),
}


class TldError(RuntimeError):
    """Raised when a libtld_b200 call returns a non-zero status."""


def load():
    """Load (once) and return the ctypes handle of libtld_b200.so; raises if it is not built."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise TldError(
                    f"{LIB_PATH} not found: build it with `python -m transformer_latent_diffusion_b200.build` "
                    "(this package has no CPU/PyTorch fallback)")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in PROTOTYPES.items():
                fn = getattr(lib, name)  # AttributeError if the symbol is not exported
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().tld_last_error()
        raise TldError(f"{what}: {msg.decode() if msg else 'unknown error'}")


def ptr(t) -> int:
    """device/host address of a torch tensor (must be contiguous)"""
    assert t.is_contiguous(), "tensor passed to libtld_b200 must be contiguous"
    return t.data_ptr()


def current_stream_ptr(device=None) -> int:
    import torch

    return torch.cuda.current_stream(device).cuda_stream
