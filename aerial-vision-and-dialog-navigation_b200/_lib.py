"""ctypes binding of ``csrc/libavdn.so`` (the C ABI of ``include/avdn.h``).

Fails loudly: a missing library, a missing symbol or a non-zero status raises;
nothing here ever falls back to a CPU or torch implementation.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libavdn.so")

_lib = None

c_void_p, c_int, c_i64, c_f32, c_f64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double


class ConvItem(C.Structure):
    """``avdn_conv_item`` of include/avdn.h."""
    _fields_ = [("w", C.c_void_p), ("wf", C.c_void_p), ("wd", C.c_void_p), ("dwf", C.c_void_p), ("grad", C.c_void_p),
                ("Cout", C.c_int32), ("Cin", C.c_int32), ("k", C.c_int32), ("stride", C.c_int32),
                ("Cout_p", C.c_int32), ("Cin_p", C.c_int32), ("pairs", C.c_int32), ("pad_", C.c_int32)]


class TileDesc(C.Structure):
    """``avdn_tile_desc`` of include/avdn.h."""
    _fields_ = [("tile8", C.c_void_p), ("H", C.c_int32), ("W", C.c_int32)]


# name -> argtypes ; every function returns int (avdn_status) unless noted
_SIGNATURES = {
    "avdn_pack_tile": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_resize_area_width": [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "avdn_raster_attention": [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_gps_to_pixels": [c_void_p, c_void_p, c_int, c_void_p, c_void_p],
    "avdn_homography_from_corners": [c_void_p, c_int, c_void_p, c_void_p],
    "avdn_render_views": [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                          c_void_p, c_void_p, c_void_p, c_void_p],
    # struct pointers are passed with ctypes.byref(...)
    "avdn_gemm_plan": [c_void_p, c_void_p, C.c_size_t],
    "avdn_gemm_run": [c_void_p, c_void_p],
    "avdn_conv0_fwd": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_conv0_fwd_eval": [c_void_p, c_void_p, c_void_p, c_void_p, c_f32, c_void_p, c_int, c_int, c_int, c_void_p],
    "avdn_conv0_wgrad": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    "avdn_conv0_fwd_stats": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "avdn_conv0_fwd_apply": [c_void_p, c_void_p, c_void_p, c_void_p, c_f32, c_void_p, c_void_p, c_int, c_int, c_int,
                             c_void_p],
    "avdn_conv0_set_tensor_path": [c_int],
    "avdn_conv3x3_thin_fwd": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_conv3x3_thin_supported": [c_int, c_int, c_int, c_int],
    "avdn_conv3x3_thin_dgrad": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "avdn_conv3x3_thin_wgrad": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "avdn_conv0_bwd": [c_void_p] * 8 + [c_f32, c_int, c_int, c_int] + [c_void_p] * 7 + [c_void_p],
    "avdn_bn_stats": [c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_f32, c_f32,
                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "avdn_bn_finalize": [c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_f32, c_f32,
                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "avdn_bn_eval_coeffs": [c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_f32, c_void_p, c_void_p,
                            c_void_p],
    "avdn_bn_set_order": [c_int],
    "avdn_bn_apply": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_f32, c_void_p],
    "avdn_bn_backward": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_int, c_f32,
                         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "avdn_bn_backward_apply": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_int, c_f32,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    "avdn_pack_conv_weight": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "avdn_unpack_conv_wgrad": [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_unpack_conv_wgrad_pairs": [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_pack_conv_weights": [c_void_p, c_int, c_void_p],
    "avdn_unpack_conv_wgrads": [c_void_p, c_int, c_int, c_void_p],
    "avdn_cast_f32_bf16": [c_void_p, c_void_p, c_i64, c_void_p],
    "avdn_nhwc_to_nchw_f32": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    "avdn_nchw_f32_to_nhwc": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    # ---- stage 3: ET
    "avdn_frame_attn_fwd": [c_void_p] * 6 + [c_int, c_int] + [c_void_p] * 4 + [c_void_p],
    "avdn_frame_attn_bwd": [c_void_p] * 5 + [c_int, c_int] + [c_void_p] * 9 + [c_void_p],
    "avdn_frame_attn_bwd_cls": [c_void_p] * 5 + [c_int, c_int] + [c_void_p] * 10 + [c_void_p],
    "avdn_embed_fwd": [c_void_p] * 6 + [c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_embed_dir_bwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "avdn_ln_fwd": [c_void_p] * 4 + [c_i64, c_int, c_f32] + [c_void_p] * 5 + [c_void_p],
    "avdn_ln_bwd": [c_void_p] * 6 + [c_i64, c_int] + [c_void_p] * 4 + [c_void_p],
    "avdn_softmax_fwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    "avdn_softmax_bwd": [c_void_p, c_void_p, c_i64, c_int, c_int, c_f32, c_void_p, c_void_p],
    # train-mode variants: nn.Dropout sites evaluated from a stateless hash of (seed, site, element)
    "avdn_ln_fwd_drop": [c_void_p] * 4 + [c_i64, c_int, c_f32] + [c_void_p] * 5 + [c_f32, C.c_uint64, C.c_uint32, c_void_p],
    "avdn_ln_bwd_drop": [c_void_p] * 6 + [c_i64, c_int] + [c_void_p] * 4 + [c_f32, C.c_uint64, C.c_uint32, c_void_p],
    "avdn_softmax_fwd_drop": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_f32,
                              C.c_uint64, C.c_uint32, c_void_p],
    "avdn_softmax_bwd_drop": [c_void_p, c_void_p, c_i64, c_int, c_int, c_f32, c_void_p, c_f32, C.c_uint64, C.c_uint32,
                              c_void_p],
    "avdn_dropout_bf16": [c_void_p, c_i64, c_f32, C.c_uint64, C.c_uint32, c_void_p],
    "avdn_dropout_f32": [c_void_p, c_void_p, c_i64, c_f32, C.c_uint64, C.c_uint32, c_void_p],
    "avdn_add_dropout_f32": [c_void_p, c_void_p, c_void_p, c_i64, c_f32, C.c_uint64, C.c_uint32, c_void_p],
    "avdn_add_dropout_f32_at": [c_void_p, c_void_p, c_void_p, c_i64, c_i64, c_f32, C.c_uint64, C.c_uint32, c_void_p],
    "avdn_dropout_keep_scale": [c_void_p, c_i64, c_f32, C.c_uint64, C.c_uint32, c_void_p],
    "avdn_heads_fwd_drop": [c_void_p, c_int, c_int, c_int, c_int] + [c_void_p] * 12 + [c_f32, C.c_uint64, C.c_uint32,
                                                                                     c_void_p],
    "avdn_heads_bwd_drop": [c_void_p, c_int, c_int, c_int, c_int] + [c_void_p] * 18 + [c_f32, c_void_p],
    "avdn_attn_decode": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_f32, c_void_p, c_void_p],
    "avdn_bert_embed_ln": [c_void_p] * 6 + [c_int, c_int, c_int, c_f32] + [c_void_p] * 5 + [c_void_p],
    "avdn_bert_embed_bwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    "avdn_gelu_fwd": [c_void_p, c_void_p, c_i64, c_void_p],
    "avdn_gelu_bwd": [c_void_p, c_void_p, c_void_p, c_i64, c_void_p],
    "avdn_linear_f32_bwd": [c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_i64,
                            c_int, c_void_p, c_void_p, c_void_p],
    "avdn_build_masks": [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "avdn_colsum": [c_void_p, c_int, c_i64, c_int, c_i64, c_void_p, c_void_p],
    "avdn_heads_fwd": [c_void_p, c_int, c_int, c_int, c_int] + [c_void_p] * 12 + [c_void_p],
    "avdn_heads_bwd": [c_void_p, c_int, c_int, c_int, c_int] + [c_void_p] * 18 + [c_void_p],
    # ---- config 5: ViT_LSTM step + simulator update
    "avdn_lstm_set_kernels": [c_int],
    "avdn_linear_f32": [c_void_p, c_i64, c_void_p, c_i64, c_void_p, c_void_p, c_i64, c_int, c_int, c_int, c_int, c_int,
                        c_void_p],
    "avdn_lstm_cell": [c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_int, c_int, c_void_p],
    "avdn_direction_embed": [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    "avdn_lang_attn_fwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_i64, c_void_p],
    "avdn_lstm_cell_bwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_int, c_int,
                           c_void_p],
    "avdn_direction_embed_bwd": [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p],
    "avdn_lang_attn_bwd": [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_int, c_int, c_void_p, c_void_p,
                           c_void_p],
    "avdn_waypoint_step": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_f32, c_int, c_void_p, c_void_p,
                           c_void_p, c_void_p],
    # ---- agent slice
    "avdn_teacher_action": [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                            c_void_p],
    "avdn_loss": [c_void_p] * 7 + [c_int, c_f32, c_int, c_f64] + [c_void_p] * 4 + [c_void_p],
    "avdn_upsample_saliency": [c_void_p, c_int, c_void_p, c_void_p],
    "avdn_upsample_saliency_bwd": [c_void_p, c_int, c_void_p, c_void_p],
    "avdn_saliency_metrics": [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p],
    "avdn_postprocess_waypoints": [c_void_p, c_void_p, c_int, c_f32] + [c_void_p] * 5 + [c_void_p],
    "avdn_sumsq": [c_void_p, c_i64, c_void_p, c_void_p],
    "avdn_adamw": [c_void_p] * 4 + [c_i64] + [c_f32] * 5 + [c_int, c_void_p, c_f32, c_f32, c_void_p],
}
_SIZE_T_FUNCS = ["avdn_gemm_plan_bytes"]


def exported_symbols():
    """Every symbol ``include/avdn.h`` declares (used by the CPU-side ABI test)."""
    return (["avdn_last_error_string", "avdn_abi_version", "avdn_device_supported"] + _SIZE_T_FUNCS
            + list(_SIGNATURES))


def register(name, argtypes):
    _SIGNATURES[name] = argtypes
    if _lib is not None:
        fn = getattr(_lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int


def lib():
    """Load (once) and return the ctypes handle; raises if the library is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback.")
        h = C.CDLL(LIB_PATH)
        h.avdn_last_error_string.restype = C.c_char_p
        h.avdn_last_error_string.argtypes = []
        h.avdn_abi_version.restype = C.c_int
        h.avdn_device_supported.restype = C.c_int
        for name in _SIZE_T_FUNCS:
            getattr(h, name).restype = C.c_size_t
            getattr(h, name).argtypes = []
        for name, argtypes in _SIGNATURES.items():
            fn = getattr(h, name)          # AttributeError if the symbol is missing
            fn.argtypes = argtypes
            fn.restype = C.c_int
        _lib = h
    return _lib


def last_error() -> str:
    return lib().avdn_last_error_string().decode()


def check(status: int, what: str = ""):
    if status != 0:
        raise RuntimeError(f"libavdn {what} failed (status {status}): {last_error()}")


def ptr(t):
    """Device pointer of a tensor (``None`` -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# When set to a list, every kernel launch made through call() / GemmPlan.run() is bracketed by
# CUDA events on the launching stream and (name, ev0, ev1, flops, bytes) is appended: the live
# per-kernel breakdown bench.py reports.  None (default) = no instrumentation.
PROFILE = None


def profile_record(name, fn, flops=0, nbytes=0):
    ev0 = torch.cuda.Event(enable_timing=True)
    ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    fn()
    ev1.record()
    PROFILE.append((name, ev0, ev1, flops, nbytes))


def call(name, *args, flops=0):
    """Invoke an ABI function on torch's current stream; raise on error.  ``flops``: algorithmic FLOPs of the call,
    recorded with its CUDA-event time when profiling is on (bench.py's roofline)."""
    fn = getattr(lib(), name)
    if PROFILE is not None:
        profile_record(name, lambda: check(fn(*args, stream_ptr()), name), flops=flops)
        return
    check(fn(*args, stream_ptr()), name)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("libavdn ops take CUDA tensors only (no CPU fallback)")
