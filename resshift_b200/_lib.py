"""ctypes binding of ``librs_b200.so`` (C ABI in include/resshift_b200.h).

There is no CPU or PyTorch fallback: if the CUDA library is missing, importing this module
fails loudly, and every compute entry point needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("RESSHIFT_B200_LIB", _HERE / "lib" / "librs_b200.so"))

RS_MAX_LEVELS = 8


class RsError(RuntimeError):
    pass


class UNetConfigC(C.Structure):
    """Mirror of ``rs_unet_config``."""
    _fields_ = [
        ("image_size", C.c_int32), ("in_channels", C.c_int32), ("model_channels", C.c_int32),
        ("out_channels", C.c_int32), ("n_levels", C.c_int32),
        ("channel_mult", C.c_int32 * RS_MAX_LEVELS), ("num_res_blocks", C.c_int32 * RS_MAX_LEVELS),
        ("n_attn", C.c_int32), ("attention_resolutions", C.c_int32 * RS_MAX_LEVELS),
        ("swin_depth", C.c_int32), ("swin_embed_dim", C.c_int32), ("swin_heads", C.c_int32),
        ("window_size", C.c_int32), ("mlp_ratio", C.c_float), ("cond_mask", C.c_int32), ("lq_size", C.c_int32),
    ]


class VQConfigC(C.Structure):
    """Mirror of ``rs_vq_config``."""
    _fields_ = [
        ("embed_dim", C.c_int32), ("n_embed", C.c_int32), ("z_channels", C.c_int32), ("in_channels", C.c_int32),
        ("out_ch", C.c_int32), ("ch", C.c_int32), ("n_levels", C.c_int32),
        ("ch_mult", C.c_int32 * RS_MAX_LEVELS), ("num_res_blocks", C.c_int32 * RS_MAX_LEVELS),
    ]


# every symbol include/resshift_b200.h declares: (restype, argtypes)
_P = C.c_void_p
_SIGNATURES = {
    "rs_version": (C.c_int, []),
    "rs_last_error": (C.c_char_p, []),
    "rs_unet_create": (C.c_int, [C.POINTER(UNetConfigC), C.POINTER(_P)]),
    "rs_unet_destroy": (None, [_P]),
    "rs_unet_param_count": (C.c_int, [_P]),
    "rs_unet_param_info": (C.c_int, [_P, C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32)]),
    "rs_unet_arena_bytes": (C.c_size_t, [_P]),
    "rs_unet_set_arena": (C.c_int, [_P, _P]),
    "rs_unet_load_param": (C.c_int, [_P, C.c_char_p, _P, _P]),
    "rs_plan_create": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "rs_plan_destroy": (None, [_P]),
    "rs_plan_workspace_bytes": (C.c_size_t, [_P]),
    "rs_plan_bind": (C.c_int, [_P, _P]),
    "rs_plan_num_launches": (C.c_int, [_P]),
    "rs_plan_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "rs_plan_profile": (C.c_int, [_P, _P, _P, _P, _P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32), _P]),
    "rs_plan_profile_ops": (C.c_int, [_P, _P, _P, _P, _P, C.POINTER(C.c_double), C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_int32), _P]),
    "rs_plan_probe": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32), _P]),
    "rs_sampler_create": (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.c_double, C.POINTER(C.c_int32), C.POINTER(_P)]),
    "rs_sampler_destroy": (None, [_P]),
    "rs_sampler_run": (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int, _P]),
    "rs_sampler_run_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, C.c_size_t, C.c_int, _P]),
    "rs_sampler_staging_bytes": (C.c_size_t, [_P]),
    "rs_sampler_set_taps": (C.c_int, [_P, _P, _P]),
    "rs_p_sample": (C.c_int, [_P, _P, _P, _P, C.c_float, C.c_float, C.c_float, C.c_int, C.c_longlong, _P]),
    "rs_op_pack_conv_weight": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "rs_op_conv2d": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int,
                               C.c_int, _P, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int, _P]),
    "rs_op_conv2d_stats": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int,
                                     C.c_int, _P, C.c_int, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int, C.c_int,
                                     C.POINTER(C.c_int32), _P, _P, C.c_int, _P]),
    "rs_op_conv2d_splitk": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int,
                                      C.c_int, _P, C.c_int, _P, C.c_int, C.c_int, _P, C.c_int, C.c_int, _P,
                                      C.POINTER(C.c_int32), _P, _P, _P]),
    "rs_op_conv2d_timeline": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int,
                                        C.c_int, _P, C.c_int, C.c_int, C.c_int, _P, C.POINTER(C.c_int32), _P, _P]),
    "rs_op_groupnorm": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_longlong, C.c_int,
                                  _P, C.c_int, _P, _P]),
    "rs_op_groupnorm_scratch_floats": (C.c_longlong, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "rs_op_groupnorm_apply": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_longlong, C.c_int,
                                        _P, C.c_int, _P, _P]),
    "rs_op_groupnorm_finalize": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, _P, _P]),
    "rs_op_groupnorm_apply_pairs": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_longlong,
                                              C.c_int, _P, C.c_int, _P, C.c_int, _P]),
    "rs_op_expand_relpos": (C.c_int, [_P, _P, C.c_int, _P]),
    "rs_op_window_attention": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P]),
    "rs_op_swin_attn": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, _P, _P, _P, _P, _P, _P,
                                  _P, _P, _P, _P, _P]),
    "rs_op_vq_attention": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.c_int, _P, _P]),
    "rs_op_mlp": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "rs_debug_tile_config": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int32)]),
    "rs_debug_swin_timeline": (C.c_int, [_P]),
    "rs_op_upsample2x": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "rs_vq_create": (C.c_int, [C.POINTER(VQConfigC), C.POINTER(_P)]),
    "rs_vq_plan_create": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "rs_vq_encode": (C.c_int, [_P, _P, _P, _P]),
    "rs_vq_decode": (C.c_int, [_P, _P, _P, _P, C.c_int, _P]),
    "rs_vq_profile_ops": (C.c_int, [_P, C.POINTER(C.c_double), C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_int32), _P]),
    "rs_op_bicubic_upsample": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "rs_op_ingest_u8": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "rs_op_emit_u8": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P]),
    "rs_op_tile_gather": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
}


def _load():
    if not LIB_PATH.exists():
        raise ImportError(
            f"resshift_b200: CUDA library {LIB_PATH} not found. Build it with "
            f"`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(rc: int) -> None:
    if rc != 0:
        msg = lib.rs_last_error()
        raise RsError(f"librs_b200 error {rc}: {msg.decode(errors='replace') if msg else '?'}")


def declared_symbols():
    return sorted(_SIGNATURES)


def ptr(t) -> int:
    """Device (or host) address of a torch tensor, or None."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def make_config(cfg) -> UNetConfigC:
    c = UNetConfigC()
    c.image_size, c.in_channels, c.model_channels, c.out_channels = cfg.image_size, cfg.in_channels, cfg.model_channels, cfg.out_channels
    c.n_levels = len(cfg.channel_mult)
    for i, v in enumerate(cfg.channel_mult):
        c.channel_mult[i] = int(v)
    for i, v in enumerate(cfg.num_res_blocks):
        c.num_res_blocks[i] = int(v)
    c.n_attn = len(cfg.attention_resolutions)
    for i, v in enumerate(cfg.attention_resolutions):
        c.attention_resolutions[i] = int(v)
    c.swin_depth, c.swin_embed_dim, c.swin_heads = cfg.swin_depth, cfg.swin_embed_dim, cfg.swin_heads
    c.window_size, c.mlp_ratio = cfg.window_size, float(cfg.mlp_ratio)
    c.cond_mask, c.lq_size = int(cfg.cond_mask), cfg.lq_size
    return c


def make_vq_config(cfg) -> VQConfigC:
    c = VQConfigC()
    c.embed_dim, c.n_embed, c.z_channels = cfg.embed_dim, cfg.n_embed, cfg.z_channels
    c.in_channels, c.out_ch, c.ch = cfg.in_channels, cfg.out_ch, cfg.ch
    c.n_levels = len(cfg.ch_mult)
    for i, v in enumerate(cfg.ch_mult):
        c.ch_mult[i] = int(v)
    for i, v in enumerate(cfg.num_res_blocks):
        c.num_res_blocks[i] = int(v)
    return c
