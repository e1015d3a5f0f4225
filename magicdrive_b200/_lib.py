"""ctypes binding of the C-ABI shared library (include/magicdrive_b200.h).

The library is the product: there is no Python / torch fallback.  `lib()` raises if the shared object is missing
and every wrapper raises `MdbError` when a call returns a non-zero status.
"""
import ctypes as C
import os
from pathlib import Path

_LIB = None
LIB_PATH = Path(os.environ.get("MDB_LIB_PATH") or Path(__file__).resolve().parent / "lib" / "libmagicdrive_b200.so")  # env: A/B builds


class MdbError(RuntimeError):
    pass


class GemmDesc(C.Structure):
    _fields_ = [
        ("a0", C.c_void_p), ("a1", C.c_void_p),
        ("c0", C.c_int), ("lda0", C.c_int), ("c1", C.c_int), ("lda1", C.c_int),
        ("n_img", C.c_int), ("h_in", C.c_int), ("w_in", C.c_int),
        ("w", C.c_void_p), ("n_out", C.c_int),
        ("taps_h", C.c_int), ("taps_w", C.c_int), ("stride", C.c_int), ("pad_h", C.c_int), ("pad_w", C.c_int),
        ("h_out", C.c_int), ("w_out", C.c_int),
        ("bias", C.c_void_p), ("rowbias", C.c_void_p), ("rowbias_ld", C.c_int),
        ("residual", C.c_void_p), ("ldr", C.c_int),
        ("out", C.c_void_p), ("ldo", C.c_int), ("out_is_f32", C.c_int), ("out_scale", C.c_float),
        ("epi_mode", C.c_int),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("force_block_n", C.c_int), ("force_splits", C.c_int), ("kernel_variant", C.c_int), ("debug_flags", C.c_int), ("trace", C.c_void_p),
        ("ln_stats", C.c_void_p), ("ln_parts", C.c_int), ("ln_eps", C.c_float), ("ln_colsum", C.c_void_p),
        ("stats_out", C.c_void_p),
    ]


# name -> (restype, argtypes); mirrors include/magicdrive_b200.h one to one
_vp, _i, _f, _ll = C.c_void_p, C.c_int, C.c_float, C.c_longlong
SIGNATURES = {
    "mdb_last_error": (C.c_char_p, []),
    "mdb_set_pdl": (_i, [_i]),
    "mdb_version": (_i, []),
    "mdb_device_ok": (_i, []),
    "mdb_gemm_conv": (_i, [C.POINTER(GemmDesc), _vp]),
    "mdb_gemm_conv_launches": (_i, [C.POINTER(GemmDesc)]),
    "mdb_gemm_conv_stats_parts": (_i, [C.POINTER(GemmDesc)]),
    "mdb_conv_direct": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "mdb_groupnorm": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _f, _vp, _vp, _i, _vp, _i, _vp, _vp]),
    "mdb_layernorm": (_i, [_vp, _ll, _i, _i, _vp, _vp, _f, _vp, _i, _vp]),
    "mdb_attention": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _i, _f, _vp]),
    "mdb_attention_multi": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _f, _vp]),
    "mdb_attention_debug_trace": (_i, [_vp]),
    "mdb_add": (_i, [_vp, _vp, _vp, _ll, _vp]),
    "mdb_upsample_nearest": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "mdb_adaptive_avgpool": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _i, _i, _vp]),
    "mdb_linear_small": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _i, _i, _i, _vp, _i, _vp]),
    "mdb_timestep_embedding": (_i, [_vp, _i, _i, _i, _f, _vp, _vp]),
    "mdb_fourier_embed": (_i, [_vp, _ll, _i, _i, _vp, _vp]),
    "mdb_nchw_to_nhwc": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "mdb_nhwc_to_nchw": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp]),
    "mdb_f32_to_bf16": (_i, [_vp, _vp, _ll, _vp]),
    "mdb_bf16_to_f32": (_i, [_vp, _vp, _ll, _vp]),
    "mdb_pack_latents": (_i, [_vp, _i, _ll, _i, _i, _i, _vp, _vp]),
    "mdb_pack_image_patches": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "mdb_latent_dist": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _f, _vp, _vp]),
    "mdb_cfg_ddim_step": (_i, [_vp, _i, _i, _i, _f, _vp, _vp, _ll, _vp]),
    "mdb_softmax_rows": (_i, [_vp, _i, _ll, _i, _vp, _i, _i, _vp]),
    "mdb_pin_views": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _ll, _i, _vp]),
    "mdb_peer_barrier": (_i, [_vp, _i, _i, _i, _i, _vp, _ll, _vp, _vp]),
    "mdb_prepare_boxes": (_i, [_vp, _i, _vp, _vp, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "mdb_camera_param": (_i, [_vp, _vp, _i, _vp, _vp]),
    "mdb_cfg_unipc_step": (_i, [_vp, _i, _i, _i, _f, _vp, _vp, _vp, _vp, _vp, _ll, _vp]),
}


def lib():
    """Load (once) and return the C-ABI library; raises if it has not been built."""
    global _LIB
    if _LIB is None:
        if not LIB_PATH.exists():
            raise MdbError(
                f"{LIB_PATH} is missing: build it with `python -m magicdrive_b200.build` "
                "(there is no CPU / torch fallback for this path)")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the header and the library disagree
            fn.restype = res
            fn.argtypes = args
        _LIB = handle
    return _LIB


def check(status: int, what: str = ""):
    if status != 0:
        msg = lib().mdb_last_error()
        raise MdbError(f"{what} failed ({status}): {msg.decode() if msg else ''}")
