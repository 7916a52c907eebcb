"""ctypes binding of libtu_b200.so (C ABI declared in include/tu_b200.h).

There is no fallback: if the shared library is missing or a symbol is absent, importing the engine
raises, and every entry point raises on a non-zero return code with the library's message.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtu_b200.so")

TU_F32, TU_BF16, TU_U8, TU_F16 = 0, 1, 2, 3      # TU_U8 and TU_F16: image input / output only, never a compute dtype
TU_LAYOUT_HWC, TU_LAYOUT_HWC_BGR = 0x100, 0x200      # OR-ed into TU_U8 for interleaved uint8 frames
TU_LAYOUT_NV12 = 0x400                               # OR-ed into TU_U8 for NV12 (4:2:0) video frames, (B, 3H/2, W)
TU_YUV_BT601, TU_YUV_FULL_RANGE = 0x1000, 0x2000     # colour bits of an NV12 code; neither = BT.709 limited range
TU_U16 = 4                                           # 16-bit frame words: valid only with a 16-bit YUV layout (P010, ...)
TU_LAYOUT_P010 = 0x800                               # OR-ed into TU_U16 for P010 (10-bit 4:2:0) video frames, (B, 3H/2, W)
TU_YUV_BT2020 = 0x4000                               # BT.2020 matrix: a colour bit of P010 codes only (not with TU_YUV_BT601)
# OR-ed into TU_U8 for 4-byte pixels with a straight alpha byte, (B, H, W, 4): R G B A / B G R A.  The layout bits 8..11 are an
# enumeration (0 CHW, 1 HWC, 2 HWC_BGR, 3 RGBA, 4 NV12, 5 BGRA, 8 P010): compare whole values, never single bits
TU_LAYOUT_RGBA, TU_LAYOUT_BGRA = 0x300, 0x500
# planar YUV, three planes Y, U, V: yuv420p (TU_U8, (B, 3H/2, W)), yuv444p (TU_U8, (B, 3, H, W)) and yuv444p16 (TU_U16 | TU_LAYOUT_YUV444P,
# (B, 3, H, W) words with the code in the high 10 bits)
TU_LAYOUT_YUV420P, TU_LAYOUT_YUV444P = 0x600, 0x700
# 4:2:2: yuv422p (TU_U8, three planes, (B, 2H, W)) and NV16 (TU_U8) / P210 (TU_U16, code in the high 10 bits): Y then interleaved (U, V) rows
TU_LAYOUT_YUV422P, TU_LAYOUT_NV16 = 0x900, 0xA00
TU_YUV_LSB10 = 0x10000                               # with TU_U16 and a planar layout: yuv420p10le / yuv422p10le / yuv444p10le
# packed 4:2:2, one plane (B, H, W, 2): YUYV (TU_U8: yuyv422 / YUY2 bytes Y0 U Y1 V; TU_U16: y210 words, code in the high 10 bits) and
# UYVY (TU_U8 only: uyvy422 bytes U Y0 V Y1)
TU_LAYOUT_YUYV, TU_LAYOUT_UYVY = 0xB00, 0xC00
TU_ERR_ARG, TU_ERR_SCALE, TU_ERR_TOKENS, TU_ERR_WORKSPACE, TU_ERR_CUDA = -1, -2, -3, -4, -5
MODEL_IDS = {"WindowTransformer": 0, "FastTransformer": 1, "ResidualTransformer": 2}

vp, fp, i32, sz = C.c_void_p, C.c_void_p, C.c_int, C.c_size_t   # float* passed as raw addresses too


class TuBlockWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "ln1_w", "ln1_b", "ln2_w", "ln2_b", "qkv_w", "qkv_b", "proj_w", "proj_b",
        "fc1_w", "fc1_b", "fc2_w", "fc2_b", "rel_bias")]


class TuUpsamplerStage(C.Structure):
    _fields_ = [("w", C.c_void_p), ("b", C.c_void_p), ("r", C.c_int)]


class TuUpFold(C.Structure):
    _fields_ = [("w", C.c_void_p), ("b", C.c_void_p), ("ring_w", C.c_void_p), ("ring_b", C.c_void_p), ("r", C.c_int)]


class TuModelWeights(C.Structure):
    _fields_ = [
        ("model", C.c_int), ("dim", C.c_int), ("heads", C.c_int), ("n_blocks", C.c_int),
        ("conv1_w", C.c_void_p), ("conv1_b", C.c_void_p), ("conv1_w64", C.c_void_p),
        ("conv2_w", C.c_void_p), ("conv2_b", C.c_void_p),
        ("down_w", C.c_void_p), ("down_b", C.c_void_p),
        ("embed_w", C.c_void_p), ("embed_b", C.c_void_p),
        ("pos_embed", C.c_void_p),
        ("blocks", C.POINTER(TuBlockWeights)),
        ("stack_w", C.c_void_p), ("stack_p", C.c_void_p), ("stack_rel", C.c_void_p),
        ("unembed_w", C.c_void_p), ("unembed_b", C.c_void_p),
        ("dec1_w", C.c_void_p), ("dec1_b", C.c_void_p),
        ("dec2_w", C.c_void_p), ("dec2_b", C.c_void_p), ("dec2_w16", C.c_void_p),
        ("dec2_wst", C.c_void_p), ("dec2_b16", C.c_void_p),
        ("up1", (TuUpsamplerStage * 2) * 4),
        ("fin", (TuUpsamplerStage * 2) * 4),
        ("up1conv_w", C.c_void_p), ("up1conv_w16", C.c_void_p), ("up1conv_wst", C.c_void_p), ("up1conv_b16", C.c_void_p),
        ("finconv_w", C.c_void_p), ("finconv_b", C.c_void_p),
        ("upfold", TuUpFold * 4),
        ("host_finconv_wb", C.c_void_p),
    ]


TU_MAX_BLOCKS = 16


class TuNamedTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("numel", C.c_longlong)]


class TuPackedModel(C.Structure):
    _fields_ = [("w", TuModelWeights), ("blocks", TuBlockWeights * TU_MAX_BLOCKS), ("host_finconv_wb", C.c_float * 84),
                ("device_bytes_used", C.c_size_t)]


class TuFramePlanes(C.Structure):
    """one NV12 / P010 frame as two device planes with row pitches in bytes (decoder / encoder surfaces)"""
    _fields_ = [("y", C.c_void_p), ("uv", C.c_void_p), ("y_pitch", C.c_longlong), ("uv_pitch", C.c_longlong)]


class TuFramePlanes3(C.Structure):
    """one planar YUV frame (yuv420p / yuv444p / yuv444p16) as three device planes with row pitches in bytes"""
    _fields_ = [("y", C.c_void_p), ("u", C.c_void_p), ("v", C.c_void_p), ("y_pitch", C.c_longlong), ("u_pitch", C.c_longlong),
                ("v_pitch", C.c_longlong)]


class TuFramePacked(C.Structure):
    """one packed 4:2:2 frame (yuyv422 / uyvy422 / y210) as one device plane with its row pitch in bytes"""
    _fields_ = [("data", C.c_void_p), ("pitch", C.c_longlong)]


# name -> (restype, argtypes); must list every symbol include/tu_b200.h declares
SIGNATURES = {
    "tu_version": (i32, []),
    "tu_last_error": (C.c_char_p, []),
    "tu_bf16_uses_tcgen05": (i32, []),
    "tu_set_bf16_tcgen05": (None, [i32]),
    "tu_debug_set": (i32, [C.c_char_p, i32]),
    "tu_debug_trace": (i32, [vp, C.c_uint]),
    "tu_launch_count": (C.c_longlong, []),
    "tu_profile_enable": (None, [i32]),
    "tu_profile_collect": (i32, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    "tu_profile_report": (i32, [C.c_char_p, sz]),
    "tu_profile_reset": (None, []),
    "tu_packed_weights_bytes": (sz, [i32, i32, i32, i32]),
    "tu_pack_weights": (i32, [i32, C.POINTER(TuNamedTensor), i32, i32, vp, sz, C.POINTER(TuPackedModel), vp]),
    "tu_forward_workspace_bytes": (sz, [i32] * 8),
    "tu_forward_workspace_bytes_for": (sz, [C.POINTER(TuModelWeights)] + [i32] * 7),
    "tu_forward_workspace_bytes_io": (sz, [C.POINTER(TuModelWeights)] + [i32] * 9),
    "tu_forward": (i32, [C.POINTER(TuModelWeights), vp, i32, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp, sz, vp]),
    "tu_forward_planes": (i32, [C.POINTER(TuModelWeights), vp, C.POINTER(TuFramePlanes), i32, vp, C.POINTER(TuFramePlanes), i32,
                                i32, i32, i32, i32, i32, i32, i32, i32, vp, sz, vp]),
    "tu_forward_frames": (i32, [C.POINTER(TuModelWeights), vp, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, i32, i32, vp, sz,
                                vp]),
    "tu_stem_conv": (i32, [vp, i32, fp, vp, fp, vp, i32, i32, i32, i32, vp]),
    "tu_conv3x3_c64": (i32, [vp, vp, fp, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    "tu_conv3x3_c64_to3": (i32, [vp, i32, fp, vp, fp, fp, i32, i32, i32, i32, vp]),
    "tu_conv3x3_c64_to3_stream": (i32, [vp, vp, fp, fp, i32, i32, i32, i32, vp]),
    "tu_conv3x3_c3_ps": (i32, [fp, fp, fp, fp, i32, i32, i32, i32, vp]),
    "tu_final_conv_add": (i32, [fp, fp, fp, fp, vp, i32, i32, i32, i32, i32, vp]),
    "tu_conv12_fused": (i32, [vp, i32, vp, fp, vp, fp, vp, i32, i32, i32, vp]),
    "tu_dec12_fused": (i32, [vp, vp, fp, vp, fp, fp, i32, i32, i32, vp]),
    "tu_upfold_conv": (i32, [vp, C.POINTER(TuUpFold), fp, i32, i32, i32, vp]),
    "tu_subpixel_conv_add": (i32, [fp, fp, fp, i32, vp, fp, vp, i32, i32, i32, i32, i32, vp]),
    "tu_patch_embed": (i32, [vp, i32, vp, fp, fp, fp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    "tu_patch_unembed": (i32, [fp, vp, fp, vp, i32, i32, vp, i32, i32, i32, i32, i32, i32, i32, i32, vp]),
    "tu_block_workspace_bytes": (sz, [i32, i32, i32]),
    "tu_block_workspace_bytes_for": (sz, [i32, i32, i32, i32, i32]),
    "tu_transformer_block": (i32, [fp, C.POINTER(TuBlockWeights), i32, i32, i32, i32, i32, i32, vp, sz, vp]),
    "tu_window_stack": (i32, [fp, C.POINTER(TuModelWeights), i32, vp]),
    "tu_resid_pre": (i32, [fp, vp, C.POINTER(TuModelWeights), i32, i32, vp]),
    "tu_resid_post": (i32, [fp, vp, C.POINTER(TuModelWeights), i32, i32, vp]),
    "tu_global_attention_workspace_bytes": (sz, [i32, i32, i32]),
    "tu_global_attention": (i32, [vp, vp, i32, i32, i32, vp, sz, vp]),
    "tu_window_attention": (i32, [vp, fp, vp, i32, i32, i32, i32, vp]),
    "tu_bicubic_add_clamp": (i32, [vp, i32, i32, i32, fp, i32, i32, vp, i32, i32, i32, i32, i32, vp]),
    "tu_resize_bilinear_aa": (i32, [vp, i32, vp, i32, i32, i32, i32, i32, i32, vp]),
    "tu_resize_bilinear_aa_to": (i32, [vp, i32, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "tu_resize_bilinear_aa_to_alpha": (i32, [vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]),
    "tu_frames_to_planar": (i32, [vp, i32, vp, i32, i32, i32, vp]),
    "tu_resample_alpha": (i32, [vp, i32, vp, i32, i32, i32, i32, i32, vp]),
    "tu_bicubic_row_schedule": (i32, [i32, i32, i32]),
    "tu_nv12_to_rgb": (i32, [vp, i32, vp, i32, i32, i32, vp]),
    "tu_rgb_to_nv12": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "tu_p010_to_rgb": (i32, [vp, i32, vp, i32, i32, i32, vp]),
    "tu_rgb_to_p010": (i32, [vp, vp, i32, i32, i32, i32, vp]),
    "tu_yuv420_planes_to_rgb": (i32, [C.POINTER(TuFramePlanes), i32, vp, i32, i32, i32, vp]),
    "tu_rgb_to_yuv420_planes": (i32, [vp, C.POINTER(TuFramePlanes), i32, i32, i32, i32, vp]),
    "tu_yuvp_to_rgb": (i32, [vp, C.POINTER(TuFramePlanes3), i32, vp, i32, i32, i32, vp]),
    "tu_rgb_to_yuvp": (i32, [vp, vp, C.POINTER(TuFramePlanes3), i32, i32, i32, i32, vp]),
    "tu_yuv422sp_to_rgb": (i32, [vp, C.POINTER(TuFramePlanes), i32, vp, i32, i32, i32, vp]),
    "tu_rgb_to_yuv422sp": (i32, [vp, vp, C.POINTER(TuFramePlanes), i32, i32, i32, i32, vp]),
    "tu_packed422_to_rgb": (i32, [vp, C.POINTER(TuFramePacked), i32, vp, i32, i32, i32, vp]),
    "tu_rgb_to_packed422": (i32, [vp, vp, C.POINTER(TuFramePacked), i32, i32, i32, i32, vp]),
}



def dtype_size(code: int) -> int:
    """bytes per element of an image dtype code (a layout or colour bits do not change it: every uint8 frame is bytes, every P010
    frame 16-bit words)"""
    return {TU_F32: 4, TU_BF16: 2, TU_U8: 1, TU_F16: 2, TU_U16: 2}[code & 0xFF]


_lib = None


def load() -> C.CDLL:
    """Load libtu_b200.so and bind every symbol; raises if anything is missing (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA engine is not built. Run `python -m transformerupscaler_b200.build` "
            "(or __graft_entry__.build()). There is no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def last_error() -> str:
    return load().tu_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Translate a C-ABI return code into the exception the reference would raise."""
    if rc == 0:
        return
    msg = last_error()
    if rc == TU_ERR_SCALE:
        raise ValueError(msg)          # FastTransformer/utils.py:96-97
    raise RuntimeError(msg)
