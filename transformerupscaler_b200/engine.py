"""Forward dispatch into libtu_b200 (registered as the PyTorch custom op ``tu::forward``) and thin
single-op wrappers used by the per-op parity tests.

PyTorch is plumbing here: it owns device memory (inputs, outputs, workspace from the caching
allocator) and the CUDA stream; all arithmetic happens in the library's kernels.  CPU tensors are
rejected — there is no fallback path.
"""
from __future__ import annotations

import ctypes as C
import itertools
import math
import weakref
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from .packing import PackedWeights

_DT = {torch.float32: _lib.TU_F32, torch.bfloat16: _lib.TU_BF16, torch.float16: _lib.TU_F16, torch.uint8: _lib.TU_U8,
       torch.uint16: _lib.TU_U16}
_TORCH_DT = {v: k for k, v in _DT.items()}
# handle -> PackedWeights, WEAK: the owner (EngineModel._tu_cache, or a test) keeps the object alive; a handle whose owner is gone
# simply disappears, so a copied / unpickled module can never release another module's weights and nothing leaks
_REGISTRY: "weakref.WeakValueDictionary[int, PackedWeights]" = weakref.WeakValueDictionary()
_next_handle = itertools.count(1)


def register_weights(pw: PackedWeights) -> int:
    h = next(_next_handle)
    _REGISTRY[h] = pw
    return h


def release_weights(handle: int) -> None:
    _REGISTRY.pop(handle, None)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _require_cuda(*ts: torch.Tensor) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("transformerupscaler_b200 runs on CUDA tensors only (no CPU fallback); got a "
                               f"{t.device} tensor")


def _code(dt: torch.dtype) -> int:
    if dt not in _DT:
        raise TypeError(f"unsupported dtype {dt}; the engine handles float32, bfloat16, float16 and (frames only) uint8 / uint16")
    return _DT[dt]


LAYOUTS = {"chw": 0, "hwc": _lib.TU_LAYOUT_HWC, "hwc_bgr": _lib.TU_LAYOUT_HWC_BGR, "nv12": _lib.TU_LAYOUT_NV12,
           "p010": _lib.TU_LAYOUT_P010, "rgba": _lib.TU_LAYOUT_RGBA, "bgra": _lib.TU_LAYOUT_BGRA,
           "yuv420p": _lib.TU_LAYOUT_YUV420P, "yuv444p": _lib.TU_LAYOUT_YUV444P, "yuv444p16": _lib.TU_LAYOUT_YUV444P,
           "yuv420p10le": _lib.TU_LAYOUT_YUV420P | _lib.TU_YUV_LSB10, "yuv422p": _lib.TU_LAYOUT_YUV422P,
           "yuv422p10le": _lib.TU_LAYOUT_YUV422P | _lib.TU_YUV_LSB10, "yuv444p10le": _lib.TU_LAYOUT_YUV444P | _lib.TU_YUV_LSB10,
           "nv16": _lib.TU_LAYOUT_NV16, "p210": _lib.TU_LAYOUT_NV16, "yuyv422": _lib.TU_LAYOUT_YUYV, "uyvy422": _lib.TU_LAYOUT_UYVY,
           "y210": _lib.TU_LAYOUT_YUYV}
# planar YUV layouts (FFmpeg's pix_fmt names) -> frame dtype; yuv444p and yuv444p16 share the layout bits and differ in the dtype, the
# *p10le layouts carry TU_YUV_LSB10 (the code in the low 10 bits of each word)
PLANAR = {"yuv420p": torch.uint8, "yuv444p": torch.uint8, "yuv444p16": torch.uint16, "yuv420p10le": torch.uint16,
          "yuv422p": torch.uint8, "yuv422p10le": torch.uint16, "yuv444p10le": torch.uint16}
# semi-planar 4:2:2 layouts -> frame dtype (nv16 and p210 share the layout bits and differ in the dtype)
SEMI422 = {"nv16": torch.uint8, "p210": torch.uint16}
# packed 4:2:2 layouts (one plane (B, H, W, 2)) -> frame dtype (yuyv422 and y210 share the layout bits and differ in the dtype)
PACKED422 = {"yuyv422": torch.uint8, "uyvy422": torch.uint8, "y210": torch.uint16}
# every YUV layout, and the ones of 16-bit words (10-bit codes: the only ones BT.2020 is defined for)
YUV_LAYOUTS = ("nv12", "p010", *PLANAR, *SEMI422, *PACKED422)
YUV16_LAYOUTS = ("p010", "yuv444p16", "yuv420p10le", "yuv422p10le", "yuv444p10le", "p210", "y210")
# colour of NV12 and P010 frames: matrix and range
YUV = {"bt709": 0, "bt601": _lib.TU_YUV_BT601, "bt709_full": _lib.TU_YUV_FULL_RANGE,
       "bt601_full": _lib.TU_YUV_BT601 | _lib.TU_YUV_FULL_RANGE}
# BT.2020 (HDR10 / HLG, 10-bit UHD): defined for 10-bit coding, so P010 frames only
YUV_P010 = {"bt2020": _lib.TU_YUV_BT2020, "bt2020_full": _lib.TU_YUV_BT2020 | _lib.TU_YUV_FULL_RANGE}


def layout_code(name: str) -> int:
    if name not in LAYOUTS:
        raise ValueError(f"unknown frame layout {name!r}: use 'chw', 'hwc', 'hwc_bgr', 'rgba', 'bgra', 'nv12', 'p010', 'yuv420p', "
                         "'yuv444p', 'yuv444p16', 'yuv420p10le', 'yuv422p', 'yuv422p10le', 'yuv444p10le', 'nv16', 'p210', 'yuyv422', "
                         "'uyvy422' or 'y210'")
    return LAYOUTS[name]


def yuv_code(name: str) -> int:
    if name in YUV:
        return YUV[name]
    if name in YUV_P010:
        return YUV_P010[name]
    raise ValueError(f"unknown YUV colour {name!r}: use 'bt709', 'bt601', 'bt709_full', 'bt601_full' or, for P010 frames, "
                     "'bt2020', 'bt2020_full'")


# the layout bits 8..11 of a code are an enumeration: compare whole values (0x500 = BGRA shares a bit with NV12's 0x400)
def _is_nv12(code: int) -> bool:
    return code & 0xF00 == _lib.TU_LAYOUT_NV12


def _is_p010(code: int) -> bool:
    return code & 0xF00 == _lib.TU_LAYOUT_P010


def _is_yuv420p(code: int) -> bool:
    return code & 0xF00 == _lib.TU_LAYOUT_YUV420P


def _is_yuv444p(code: int) -> bool:
    """yuv444p (TU_U8) or yuv444p16 (TU_U16): (B, 3, H, W)"""
    return code & 0xF00 == _lib.TU_LAYOUT_YUV444P


def _is_yuv422p(code: int) -> bool:
    """yuv422p (TU_U8) or yuv422p10le (TU_U16 | TU_YUV_LSB10): (B, 2H, W)"""
    return code & 0xF00 == _lib.TU_LAYOUT_YUV422P


def _is_nv16(code: int) -> bool:
    """nv16 (TU_U8) or p210 (TU_U16): (B, 2H, W), frame surfaces are (y, uv) pairs"""
    return code & 0xF00 == _lib.TU_LAYOUT_NV16


def _is_packed422(code: int) -> bool:
    """yuyv422 / y210 (YUYV) or uyvy422 (UYVY): one plane (B, H, W, 2), frame surfaces are single (H, W, 2) tensors"""
    return code & 0xF00 in (_lib.TU_LAYOUT_YUYV, _lib.TU_LAYOUT_UYVY)


def _is_yuvp(code: int) -> bool:
    """planar YUV: frame surfaces are (y, u, v) triples"""
    return _is_yuv420p(code) or _is_yuv444p(code) or _is_yuv422p(code)


def _yuv_name(code: int, dtype: torch.dtype) -> str:
    """layout name of a planar or 4:2:2 YUV code whose frames have dtype `dtype`"""
    lsb = code & _lib.TU_YUV_LSB10
    if _is_yuv420p(code):
        return "yuv420p10le" if lsb else "yuv420p"
    if _is_yuv422p(code):
        return "yuv422p10le" if lsb else "yuv422p"
    if _is_nv16(code):
        return "p210" if dtype == torch.uint16 else "nv16"
    if _is_packed422(code):
        return "y210" if dtype == torch.uint16 else "uyvy422" if code & 0xF00 == _lib.TU_LAYOUT_UYVY else "yuyv422"
    return "yuv444p10le" if lsb else "yuv444p16" if dtype == torch.uint16 else "yuv444p"


def _is_px4(code: int) -> bool:
    """RGBA / BGRA: 4-byte pixels (B, H, W, 4)"""
    return code & 0xF00 in (_lib.TU_LAYOUT_RGBA, _lib.TU_LAYOUT_BGRA)


def _image_shape(B: int, C_: int, h: int, w: int, code: int) -> Tuple[int, ...]:
    """shape of a (B, C_, h, w) image stored with dtype (| layout) code `code`: planar, interleaved (B,h,w,3), 4-byte pixels
    (B,h,w,4), NV12 / P010 / yuv420p[10le] (B,3h/2,w), 4:2:2 (B,2h,w), packed 4:2:2 (B,h,w,2) or 4:4:4 (B,3,h,w)"""
    if _is_nv12(code) or _is_p010(code) or _is_yuv420p(code):
        return (B, 3 * h // 2, w)
    if _is_yuv444p(code):
        return (B, 3, h, w)
    if _is_yuv422p(code) or _is_nv16(code):
        return (B, 2 * h, w)
    if _is_px4(code):
        return (B, h, w, 4)
    if _is_packed422(code):
        return (B, h, w, 2)
    return (B, h, w, 3) if code & 0xF00 in (_lib.TU_LAYOUT_HWC, _lib.TU_LAYOUT_HWC_BGR) else (B, C_, h, w)


def _yuv420_hw(x: torch.Tensor, fmt: str, dtype: torch.dtype) -> Tuple[int, int]:
    """(H, W) of 4:2:0 frames (B, 3H/2, W); raises ValueError for a shape or dtype that is not one"""
    if x.dim() != 3 or x.dtype != dtype:
        raise ValueError(f"{fmt} frames must be {str(dtype)[6:]} of shape (B, 3H/2, W), got {x.dtype} {tuple(x.shape)}")
    if x.shape[1] % 3:
        raise ValueError(f"{fmt} frames (B, 3H/2, W) need a row count divisible by 3, got {tuple(x.shape)}")
    H, W = int(x.shape[1]) * 2 // 3, int(x.shape[2])
    if H % 2 or W % 2:
        raise ValueError(f"{fmt} frames need an even height and width, got H={H} W={W}")
    return H, W


def _nv12_hw(x: torch.Tensor) -> Tuple[int, int]:
    """(H, W) of NV12 frames (B, 3H/2, W) uint8"""
    return _yuv420_hw(x, "NV12", torch.uint8)


def _p010_hw(x: torch.Tensor) -> Tuple[int, int]:
    """(H, W) of P010 frames (B, 3H/2, W) uint16"""
    return _yuv420_hw(x, "P010", torch.uint16)


def plane_pairs(frames, fmt: str, what: str) -> Tuple[int, int, int]:
    """(B, H, W) of semi-planar frames given as a list / tuple of B (y, uv) plane pairs -- strided views of a decoder's or encoder's
    pitched surfaces: y (H, W) and uv (H/2, W) for 4:2:0 or (H, W) for 4:2:2, uint8 for NV12 / NV16 and uint16 for P010 / P210, unit
    stride along W, any row stride, all CUDA tensors on one device.  Raises ValueError for anything else."""
    dtype = torch.uint8 if fmt in ("NV12", "NV16") else torch.uint16
    sub = fmt in ("NV12", "P010")
    if not isinstance(frames, (list, tuple)) or not frames:
        raise ValueError(f"{what}: {fmt} frame planes are a non-empty list of (y, uv) tensor pairs")
    dev, hw = None, None
    for b, pair in enumerate(frames):
        if not isinstance(pair, (list, tuple)) or len(pair) != 2 or not all(isinstance(t, torch.Tensor) for t in pair):
            raise ValueError(f"{what}[{b}] must be a (y, uv) pair of tensors")
        for name, t in zip(("y", "uv"), pair):
            if t.dim() != 2 or t.dtype != dtype:
                raise ValueError(f"{what}[{b}].{name}: {fmt} planes are 2-D {str(dtype)[6:]} tensors, got {t.dtype} {tuple(t.shape)}")
            if t.stride(1) != 1 and t.shape[1] > 1:
                raise ValueError(f"{what}[{b}].{name}: a plane needs unit stride along its rows, got strides {t.stride()}")
            if not t.is_cuda or (dev is not None and t.device != dev):
                raise ValueError(f"{what}[{b}].{name}: every plane must be a CUDA tensor on one device, got {t.device}")
            dev = t.device
        y, uv = pair
        H, W = int(y.shape[0]), int(y.shape[1])
        if sub and (H % 2 or W % 2 or tuple(uv.shape) != (H // 2, W)):
            raise ValueError(f"{what}[{b}]: {fmt} planes are y (H, W) and uv (H/2, W) with H and W even, got {tuple(y.shape)} and "
                             f"{tuple(uv.shape)}")
        if not sub and (W % 2 or tuple(uv.shape) != (H, W)):
            raise ValueError(f"{what}[{b}]: {fmt} planes are y and uv of one size (H, W) with W even, got {tuple(y.shape)} and "
                             f"{tuple(uv.shape)}")
        if hw is not None and hw != (H, W):
            raise ValueError(f"{what}[{b}]: every frame of a batch has the same size, got {(H, W)} after {hw}")
        hw = (H, W)
    return len(frames), hw[0], hw[1]


def _yuv444_hw(x: torch.Tensor, fmt: str, dtype: torch.dtype) -> Tuple[int, int]:
    """(H, W) of 4:4:4 planar frames (B, 3, H, W); raises ValueError for a shape or dtype that is not one"""
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != dtype:
        raise ValueError(f"{fmt} frames must be {str(dtype)[6:]} of shape (B, 3, H, W), got {x.dtype} {tuple(x.shape)}")
    return int(x.shape[2]), int(x.shape[3])


def _yuv422_hw(x: torch.Tensor, fmt: str, dtype: torch.dtype) -> Tuple[int, int]:
    """(H, W) of 4:2:2 frames (B, 2H, W); raises ValueError for a shape or dtype that is not one"""
    if x.dim() != 3 or x.dtype != dtype:
        raise ValueError(f"{fmt} frames must be {str(dtype)[6:]} of shape (B, 2H, W), got {x.dtype} {tuple(x.shape)}")
    if x.shape[1] % 2 or x.shape[2] % 2:
        raise ValueError(f"{fmt} frames (B, 2H, W) need an even row count and an even width, got {tuple(x.shape)}")
    return int(x.shape[1]) // 2, int(x.shape[2])


def _packed422_hw(x: torch.Tensor, fmt: str) -> Tuple[int, int]:
    """(H, W) of packed 4:2:2 frames (B, H, W, 2); raises ValueError for a shape or dtype that is not one"""
    dtype = PACKED422[fmt]
    if x.dim() != 4 or x.shape[3] != 2 or x.dtype != dtype:
        raise ValueError(f"{fmt} frames must be {str(dtype)[6:]} of shape (B, H, W, 2), got {x.dtype} {tuple(x.shape)}")
    if x.shape[2] % 2:
        raise ValueError(f"{fmt} frames (B, H, W, 2) need an even width, got {tuple(x.shape)}")
    return int(x.shape[1]), int(x.shape[2])


def _yuvp_hw(x: torch.Tensor, fmt: str) -> Tuple[int, int]:
    """(H, W) of dense planar, semi-planar or packed 4:2:2 YUV frames of layout name `fmt`"""
    if fmt in PACKED422:
        return _packed422_hw(x, fmt)
    if fmt in SEMI422 or fmt.startswith("yuv422p"):
        return _yuv422_hw(x, fmt, SEMI422.get(fmt) or PLANAR[fmt])
    return _yuv420_hw(x, fmt, PLANAR[fmt]) if fmt.startswith("yuv420p") else _yuv444_hw(x, fmt, PLANAR[fmt])


def plane_triples(frames, fmt: str, what: str) -> Tuple[int, int, int]:
    """(B, H, W) of planar YUV frames (fmt: a key of PLANAR) given as a list / tuple of B (y, u, v) plane triples -- strided views of a
    decoder's surfaces or an FFmpeg frame's data[0..2]: y (H, W), u and v (H/2, W/2) for 4:2:0, (H, W/2) for 4:2:2 or (H, W) for 4:4:4,
    of the layout's dtype, unit stride along W, any row stride, all CUDA tensors on one device.  Raises ValueError for anything else."""
    dtype = PLANAR[fmt]
    if not isinstance(frames, (list, tuple)) or not frames:
        raise ValueError(f"{what}: {fmt} frame planes are a non-empty list of (y, u, v) tensor triples")
    dev, hw = None, None
    for b, tri in enumerate(frames):
        if not isinstance(tri, (list, tuple)) or len(tri) != 3 or not all(isinstance(t, torch.Tensor) for t in tri):
            raise ValueError(f"{what}[{b}] must be a (y, u, v) triple of tensors")
        for name, t in zip(("y", "u", "v"), tri):
            if t.dim() != 2 or t.dtype != dtype:
                raise ValueError(f"{what}[{b}].{name}: {fmt} planes are 2-D {str(dtype)[6:]} tensors, got {t.dtype} {tuple(t.shape)}")
            if t.stride(1) != 1 and t.shape[1] > 1:
                raise ValueError(f"{what}[{b}].{name}: a plane needs unit stride along its rows, got strides {t.stride()}")
            if not t.is_cuda or (dev is not None and t.device != dev):
                raise ValueError(f"{what}[{b}].{name}: every plane must be a CUDA tensor on one device, got {t.device}")
            dev = t.device
        y, u, v = tri
        H, W = int(y.shape[0]), int(y.shape[1])
        if fmt.startswith("yuv420p"):
            if H % 2 or W % 2 or tuple(u.shape) != (H // 2, W // 2) or tuple(v.shape) != (H // 2, W // 2):
                raise ValueError(f"{what}[{b}]: {fmt} planes are y (H, W), u and v (H/2, W/2) with H and W even, got {tuple(y.shape)}, "
                                 f"{tuple(u.shape)} and {tuple(v.shape)}")
        elif fmt.startswith("yuv422p"):
            if W % 2 or tuple(u.shape) != (H, W // 2) or tuple(v.shape) != (H, W // 2):
                raise ValueError(f"{what}[{b}]: {fmt} planes are y (H, W), u and v (H, W/2) with W even, got {tuple(y.shape)}, "
                                 f"{tuple(u.shape)} and {tuple(v.shape)}")
        elif tuple(u.shape) != (H, W) or tuple(v.shape) != (H, W):
            raise ValueError(f"{what}[{b}]: {fmt} planes are y, u and v of one size (H, W), got {tuple(y.shape)}, {tuple(u.shape)} and "
                             f"{tuple(v.shape)}")
        if hw is not None and hw != (H, W):
            raise ValueError(f"{what}[{b}]: every frame of a batch has the same size, got {(H, W)} after {hw}")
        hw = (H, W)
    return len(frames), hw[0], hw[1]


def packed_surfaces(frames, fmt: str, what: str) -> Tuple[int, int, int]:
    """(B, H, W) of packed 4:2:2 frames (fmt: a key of PACKED422) given as a list / tuple of B surfaces -- strided views of a capture
    buffer or a decoder's pitched surface: (H, W, 2) tensors of the layout's dtype with strides (row pitch in samples, 2, 1), W even,
    all CUDA tensors on one device.  Raises ValueError for anything else."""
    dtype = PACKED422[fmt]
    if not isinstance(frames, (list, tuple)) or not frames:
        raise ValueError(f"{what}: {fmt} frame surfaces are a non-empty list of (H, W, 2) tensors")
    dev, hw = None, None
    for b, t in enumerate(frames):
        if not isinstance(t, torch.Tensor) or t.dim() != 3 or t.shape[2] != 2 or t.dtype != dtype:
            got = f"{t.dtype} {tuple(t.shape)}" if isinstance(t, torch.Tensor) else type(t).__name__
            raise ValueError(f"{what}[{b}]: {fmt} surfaces are {str(dtype)[6:]} tensors (H, W, 2), got {got}")
        if t.stride(2) != 1 or (t.stride(1) != 2 and t.shape[1] > 1):
            raise ValueError(f"{what}[{b}]: a {fmt} surface needs strides (row pitch, 2, 1), got {t.stride()}")
        if not t.is_cuda or (dev is not None and t.device != dev):
            raise ValueError(f"{what}[{b}]: every surface must be a CUDA tensor on one device, got {t.device}")
        dev = t.device
        H, W = int(t.shape[0]), int(t.shape[1])
        if W % 2:
            raise ValueError(f"{what}[{b}]: {fmt} frames need an even width, got {tuple(t.shape)}")
        if hw is not None and hw != (H, W):
            raise ValueError(f"{what}[{b}]: every frame of a batch has the same size, got {(H, W)} after {hw}")
        hw = (H, W)
    return len(frames), hw[0], hw[1]


def frame_planes(frames, layout: str, what: str) -> Tuple[int, int, int]:
    """(B, H, W) of a list of frame planes of layout `layout`: (y, uv) pairs for 'nv12' / 'p010', (y, u, v) triples for planar YUV,
    single (H, W, 2) surfaces for packed 4:2:2"""
    if layout in PACKED422:
        return packed_surfaces(frames, layout, what)
    if layout in PLANAR:
        return plane_triples(frames, layout, what)
    return plane_pairs(frames, layout.upper(), what)


def _flat(frames) -> List[torch.Tensor]:
    """the planes of a list of frames, in order (a packed 4:2:2 frame is its one surface)"""
    return [t for planes in frames for t in ((planes,) if isinstance(planes, torch.Tensor) else planes)]


def _planes_per_frame(code: int) -> int:
    return 3 if _is_yuvp(code) else 1 if _is_packed422(code) else 2


def _descriptors(flat: Sequence[torch.Tensor], code: int = _lib.TU_U8 | _lib.TU_LAYOUT_NV12):
    """descriptor array of the flattened planes of a side of code `code`: TuFramePlanes of [y0, uv0, y1, uv1, ...] (NV12 / P010 / NV16 / P210),
    TuFramePlanes3 of [y0, u0, v0, y1, ...] (planar YUV) or TuFramePacked of [s0, s1, ...] (packed 4:2:2); a plane of one row has no
    meaningful row stride"""
    def pitch(t):
        return (t.stride(0) if t.shape[0] > 1 else t.shape[1] * (t.shape[2] if t.dim() == 3 else 1)) * t.element_size()
    k = _planes_per_frame(code)
    S = {1: _lib.TuFramePacked, 2: _lib.TuFramePlanes, 3: _lib.TuFramePlanes3}[k]
    n = len(flat) // k
    return (S * n)(*[S(*[flat[k * b + i].data_ptr() for i in range(k)], *[pitch(flat[k * b + i]) for i in range(k)])
                     for b in range(n)])


def _forward_impl(x: torch.Tensor, handle: int, out_h: int, out_w: int, scale: int, compute_bf16: bool,
                  out_code: int, clamp: bool, in_layout: int = 0) -> torch.Tensor:
    lib = _lib.load()
    pw = _REGISTRY.get(handle)
    if pw is None:
        raise RuntimeError(f"tu::forward: packed-weights handle {handle} is not alive (its TransformerModel was deleted or repacked)")
    _require_cuda(x)
    if _is_nv12(in_layout) or _is_p010(in_layout):
        H, W = _nv12_hw(x) if _is_nv12(in_layout) else _p010_hw(x)
        x = x.contiguous()
        B = x.shape[0]
    elif _is_yuvp(in_layout) or _is_nv16(in_layout) or _is_packed422(in_layout):
        H, W = _yuvp_hw(x, _yuv_name(in_layout, x.dtype))
        x = x.contiguous()
        B = x.shape[0]
    elif in_layout:
        px = 4 if _is_px4(in_layout) else 3
        if x.dim() != 4 or x.shape[3] != px or x.dtype != torch.uint8:
            raise RuntimeError(f"interleaved frames must be uint8 of shape (B,H,W,{px}), got {x.dtype} {tuple(x.shape)}")
        x = x.contiguous()
        B, H, W, _ = x.shape
    else:
        if x.dim() != 4 or x.shape[1] != 3:
            raise RuntimeError(f"expected input of shape (B,3,H,W), got {tuple(x.shape)}")
        x = x.contiguous()
        B, _, H, W = x.shape
    cdt = _lib.TU_BF16 if compute_bf16 else _lib.TU_F32
    out_shape = _image_shape(B, 3, out_h, out_w, out_code)
    u16_out = (out_code & 0xFF) == _lib.TU_U16
    u16_layout = _is_yuv444p(out_code) or _is_nv16(out_code) or _is_packed422(out_code) or out_code & _lib.TU_YUV_LSB10
    if (u16_out and not (u16_layout or _is_p010(out_code))) or (_is_p010(out_code) and not u16_out):
        raise RuntimeError("the P010 output layout is for uint16 frames, and uint16 output is P010 only")
    if out_code >> 8 and not _is_p010(out_code) and not u16_out and (out_code & 0xFF) != _lib.TU_U8:
        raise RuntimeError("interleaved and NV12 output layouts are for uint8 frames")
    out = torch.empty(out_shape, dtype=_TORCH_DT[out_code & 0xFF], device=x.device)
    in_code = _code(x.dtype) | in_layout
    nbytes = lib.tu_forward_workspace_bytes_io(C.byref(pw.struct), B, H, W, out_h, out_w, scale, cdt, in_code, out_code)
    if nbytes == 0:
        _lib.check(_lib.TU_ERR_SCALE if "was not built" in _lib.last_error() else _lib.TU_ERR_ARG)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        rc = lib.tu_forward(C.byref(pw.struct), x.data_ptr(), in_code, out.data_ptr(), out_code,
                            B, H, W, out_h, out_w, scale, cdt, int(clamp), ws.data_ptr(), nbytes, _stream())
    _lib.check(rc)
    return out


@torch.library.custom_op("tu::forward", mutates_args=(), device_types="cuda")
def tu_forward(x: torch.Tensor, handle: int, out_h: int, out_w: int, scale: int, compute_bf16: bool,
               out_code: int, clamp: bool, in_layout: int = 0) -> torch.Tensor:
    return _forward_impl(x, handle, out_h, out_w, scale, compute_bf16, out_code, clamp, in_layout)


@tu_forward.register_fake
def _(x, handle, out_h, out_w, scale, compute_bf16, out_code, clamp, in_layout=0):
    return x.new_empty(_image_shape(x.shape[0], 3, out_h, out_w, out_code), dtype=_TORCH_DT[out_code & 0xFF])


@torch.library.custom_op("tu::forward_planes", mutates_args=("out_planes",), device_types="cuda")
def tu_forward_planes(x: Optional[torch.Tensor], x_planes: List[torch.Tensor], out_planes: List[torch.Tensor], handle: int, out_h: int,
                      out_w: int, scale: int, compute_bf16: bool, out_code: int, clamp: bool, in_layout: int) -> torch.Tensor:
    """tu::forward with frame surfaces on a YUV side: the input is x (dense) or x_planes ([y0, uv0, y1, uv1, ...] for NV12 / P010,
    [y0, u0, v0, y1, ...] for planar YUV, [s0, s1, ...] for packed 4:2:2); the output is written into out_planes (flattened the same way by out_code; an empty tensor is
    returned), or returned as a new dense tensor when out_planes is empty"""
    lib = _lib.load()
    pw = _REGISTRY.get(handle)
    if pw is None:
        raise RuntimeError(f"tu::forward_planes: packed-weights handle {handle} is not alive (its TransformerModel was deleted or repacked)")
    ref = x if x is not None else x_planes[0]
    _require_cuda(ref)
    if x is not None:
        if _is_nv12(in_layout) or _is_p010(in_layout):
            H, W = _nv12_hw(x) if _is_nv12(in_layout) else _p010_hw(x)
            B = x.shape[0]
        elif _is_yuvp(in_layout) or _is_nv16(in_layout) or _is_packed422(in_layout):
            H, W = _yuvp_hw(x, _yuv_name(in_layout, x.dtype))
            B = x.shape[0]
        elif in_layout:
            B, H, W = x.shape[0], x.shape[1], x.shape[2]
        else:
            B, H, W = x.shape[0], x.shape[2], x.shape[3]
        x = x.contiguous()
        in_code = _code(x.dtype) | in_layout
    else:
        B, (H, W) = len(x_planes) // _planes_per_frame(in_layout), x_planes[0].shape[:2]
        in_code = _code(x_planes[0].dtype) | in_layout
    cdt = _lib.TU_BF16 if compute_bf16 else _lib.TU_F32
    odt = _TORCH_DT[out_code & 0xFF]
    out = ref.new_empty((0,) if out_planes else _image_shape(B, 3, out_h, out_w, out_code), dtype=odt)
    nbytes = lib.tu_forward_workspace_bytes_io(C.byref(pw.struct), B, H, W, out_h, out_w, scale, cdt, in_code, out_code)
    if nbytes == 0:
        _lib.check(_lib.TU_ERR_SCALE if "was not built" in _lib.last_error() else _lib.TU_ERR_ARG)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=ref.device)
    xd = _descriptors(x_planes, in_code) if x is None else None
    od = _descriptors(out_planes, out_code) if out_planes else None
    with torch.cuda.device(ref.device):
        rc = lib.tu_forward_frames(C.byref(pw.struct), x.data_ptr() if x is not None else None, xd, in_code,
                                   None if out_planes else out.data_ptr(), od, out_code, B, H, W, out_h, out_w, scale, cdt, int(clamp),
                                   ws.data_ptr(), nbytes, _stream())
    _lib.check(rc)
    return out


@tu_forward_planes.register_fake
def _(x, x_planes, out_planes, handle, out_h, out_w, scale, compute_bf16, out_code, clamp, in_layout):
    ref = x if x is not None else x_planes[0]
    B = x.shape[0] if x is not None else len(x_planes) // _planes_per_frame(in_layout)
    return ref.new_empty((0,) if out_planes else _image_shape(B, 3, out_h, out_w, out_code), dtype=_TORCH_DT[out_code & 0xFF])


@torch.library.custom_op("tu::resize_aa", mutates_args=(), device_types="cuda")
def tu_resize_aa(x: torch.Tensor, out_h: int, out_w: int, clamp: bool, out_code: int = -1,
                 alpha: Optional[torch.Tensor] = None) -> torch.Tensor:
    """antialiased bilinear Resize of a (B,3,H,W) float image; out_code < 0: same dtype as x, else a dtype (| layout) code.
    alpha: the (B, out_h, out_w) uint8 alpha plane of an RGBA / BGRA output (tu::resample_alpha); None writes alpha 255"""
    lib = _lib.load()
    _require_cuda(x, alpha)
    x = x.contiguous()
    B, Cc, H, W = x.shape
    if out_code < 0:
        out_code = _code(x.dtype)
    if Cc != 3 and out_code >> 8:
        raise RuntimeError("interleaved output needs a 3-channel image")
    if alpha is not None and (not _is_px4(out_code) or alpha.dtype != torch.uint8 or tuple(alpha.shape) != (B, out_h, out_w)):
        raise RuntimeError(f"an alpha plane is (B, out_h, out_w) uint8 for an RGBA / BGRA output, got {alpha.dtype} {tuple(alpha.shape)}")
    out = torch.empty(_image_shape(B, Cc, out_h, out_w, out_code), dtype=_TORCH_DT[out_code & 0xFF], device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_resize_bilinear_aa_to_alpha(x.data_ptr(), _code(x.dtype), None if alpha is None else alpha.contiguous().data_ptr(),
                                                      out.data_ptr(), out_code, B * Cc // 3, H, W, out_h, out_w, int(clamp), _stream()))
    return out


@tu_resize_aa.register_fake
def _(x, out_h, out_w, clamp, out_code=-1, alpha=None):
    if out_code < 0:
        return x.new_empty((x.shape[0], x.shape[1], out_h, out_w))
    return x.new_empty(_image_shape(x.shape[0], x.shape[1], out_h, out_w, out_code), dtype=_TORCH_DT[out_code & 0xFF])


@torch.library.custom_op("tu::resample_alpha", mutates_args=(), device_types="cuda")
def tu_resample_alpha(x: torch.Tensor, code: int, out_h: int, out_w: int) -> torch.Tensor:
    """the alpha bytes of RGBA / BGRA frames (B,H,W,4) uint8 resampled (bicubic, tu_resample_alpha) to a (B,out_h,out_w) uint8 plane"""
    lib = _lib.load()
    _require_cuda(x)
    if x.dim() != 4 or x.shape[3] != 4 or x.dtype != torch.uint8:
        raise RuntimeError(f"resample_alpha takes (B,H,W,4) uint8 frames, got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, H, W, _ = x.shape
    out = torch.empty((B, out_h, out_w), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_resample_alpha(x.data_ptr(), code, out.data_ptr(), B, H, W, out_h, out_w, _stream()))
    return out


@tu_resample_alpha.register_fake
def _(x, code, out_h, out_w):
    return x.new_empty((x.shape[0], out_h, out_w), dtype=torch.uint8)


@torch.library.custom_op("tu::rgb_to_nv12", mutates_args=(), device_types="cuda")
def tu_rgb_to_nv12(x: torch.Tensor, code: int) -> torch.Tensor:
    """planar fp16 RGB (B,3,H,W) -> NV12 frames (B,3H/2,W) uint8; code = TU_U8 | TU_LAYOUT_NV12 | colour bits"""
    lib = _lib.load()
    _require_cuda(x)
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != torch.float16:
        raise RuntimeError(f"rgb_to_nv12 takes planar fp16 RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    out = torch.empty((B, 3 * H // 2, W), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_nv12(x.data_ptr(), out.data_ptr(), code, B, H, W, _stream()))
    return out


@tu_rgb_to_nv12.register_fake
def _(x, code):
    return x.new_empty((x.shape[0], 3 * x.shape[2] // 2, x.shape[3]), dtype=torch.uint8)


@torch.library.custom_op("tu::rgb_to_p010", mutates_args=(), device_types="cuda")
def tu_rgb_to_p010(x: torch.Tensor, code: int) -> torch.Tensor:
    """planar fp32 RGB (B,3,H,W) -> P010 frames (B,3H/2,W) uint16; code = TU_U16 | TU_LAYOUT_P010 | colour bits"""
    lib = _lib.load()
    _require_cuda(x)
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != torch.float32:
        raise RuntimeError(f"rgb_to_p010 takes planar fp32 RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    out = torch.empty((B, 3 * H // 2, W), dtype=torch.uint16, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_p010(x.data_ptr(), out.data_ptr(), code, B, H, W, _stream()))
    return out


@tu_rgb_to_p010.register_fake
def _(x, code):
    return x.new_empty((x.shape[0], 3 * x.shape[2] // 2, x.shape[3]), dtype=torch.uint16)


@torch.library.custom_op("tu::rgb_to_yuv420_planes", mutates_args=("planes",), device_types="cuda")
def tu_rgb_to_yuv420_planes(x: torch.Tensor, planes: List[torch.Tensor], code: int) -> None:
    """planar RGB (B,3,H,W) -> NV12 (fp16 RGB) or P010 (fp32 RGB) frames written into the surfaces [y0, uv0, y1, uv1, ...]"""
    lib = _lib.load()
    _require_cuda(x)
    want = torch.float32 if _is_p010(code) else torch.float16
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != want:
        raise RuntimeError(f"rgb_to_yuv420_planes takes planar {str(want)[6:]} RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_yuv420_planes(x.data_ptr(), _descriptors(planes), code, B, H, W, _stream()))


@tu_rgb_to_yuv420_planes.register_fake
def _(x, planes, code):
    return None


@torch.library.custom_op("tu::rgb_to_yuvp", mutates_args=(), device_types="cuda")
def tu_rgb_to_yuvp(x: torch.Tensor, code: int) -> torch.Tensor:
    """planar RGB (B,3,H,W) -> planar YUV frames: fp16 RGB -> yuv420p (B,3H/2,W) / yuv422p (B,2H,W) / yuv444p (B,3,H,W) uint8, fp32 RGB
    -> yuv444p16 or the *p10le frames of those shapes, uint16; code = the frames' TU_U8 / TU_U16 | planar layout [| TU_YUV_LSB10] |
    colour bits"""
    lib = _lib.load()
    _require_cuda(x)
    w16 = (code & 0xFF) == _lib.TU_U16
    want = torch.float32 if w16 else torch.float16
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != want:
        raise RuntimeError(f"rgb_to_yuvp takes planar {str(want)[6:]} RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    out = torch.empty(_image_shape(B, 3, H, W, code), dtype=torch.uint16 if w16 else torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_yuvp(x.data_ptr(), out.data_ptr(), None, code, B, H, W, _stream()))
    return out


@tu_rgb_to_yuvp.register_fake
def _(x, code):
    w16 = (code & 0xFF) == _lib.TU_U16
    return x.new_empty(_image_shape(x.shape[0], 3, x.shape[2], x.shape[3], code), dtype=torch.uint16 if w16 else torch.uint8)


@torch.library.custom_op("tu::rgb_to_yuvp_planes", mutates_args=("planes",), device_types="cuda")
def tu_rgb_to_yuvp_planes(x: torch.Tensor, planes: List[torch.Tensor], code: int) -> None:
    """planar RGB (B,3,H,W) -> planar YUV frames (fp16 RGB for 8-bit codes, fp32 for 16-bit ones) written into the surfaces
    [y0, u0, v0, y1, ...]"""
    lib = _lib.load()
    _require_cuda(x)
    want = torch.float32 if (code & 0xFF) == _lib.TU_U16 else torch.float16
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != want:
        raise RuntimeError(f"rgb_to_yuvp_planes takes planar {str(want)[6:]} RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_yuvp(x.data_ptr(), None, _descriptors(planes, code), code, B, H, W, _stream()))


@tu_rgb_to_yuvp_planes.register_fake
def _(x, planes, code):
    return None


@torch.library.custom_op("tu::rgb_to_yuv422sp", mutates_args=(), device_types="cuda")
def tu_rgb_to_yuv422sp(x: torch.Tensor, code: int) -> torch.Tensor:
    """planar RGB (B,3,H,W) -> semi-planar 4:2:2 frames (B,2H,W): fp16 RGB -> nv16 uint8, fp32 RGB -> p210 uint16; code = the frames'
    TU_U8 / TU_U16 | TU_LAYOUT_NV16 | colour bits"""
    lib = _lib.load()
    _require_cuda(x)
    w16 = (code & 0xFF) == _lib.TU_U16
    want = torch.float32 if w16 else torch.float16
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != want:
        raise RuntimeError(f"rgb_to_yuv422sp takes planar {str(want)[6:]} RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    out = torch.empty(_image_shape(B, 3, H, W, code), dtype=torch.uint16 if w16 else torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_yuv422sp(x.data_ptr(), out.data_ptr(), None, code, B, H, W, _stream()))
    return out


@tu_rgb_to_yuv422sp.register_fake
def _(x, code):
    w16 = (code & 0xFF) == _lib.TU_U16
    return x.new_empty(_image_shape(x.shape[0], 3, x.shape[2], x.shape[3], code), dtype=torch.uint16 if w16 else torch.uint8)


@torch.library.custom_op("tu::rgb_to_yuv422sp_planes", mutates_args=("planes",), device_types="cuda")
def tu_rgb_to_yuv422sp_planes(x: torch.Tensor, planes: List[torch.Tensor], code: int) -> None:
    """planar RGB (B,3,H,W) -> semi-planar 4:2:2 frames (fp16 RGB for nv16, fp32 for p210) written into the surfaces [y0, uv0, y1, ...]"""
    lib = _lib.load()
    _require_cuda(x)
    want = torch.float32 if (code & 0xFF) == _lib.TU_U16 else torch.float16
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != want:
        raise RuntimeError(f"rgb_to_yuv422sp_planes takes planar {str(want)[6:]} RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_yuv422sp(x.data_ptr(), None, _descriptors(planes, code), code, B, H, W, _stream()))


@tu_rgb_to_yuv422sp_planes.register_fake
def _(x, planes, code):
    return None


@torch.library.custom_op("tu::rgb_to_packed422", mutates_args=(), device_types="cuda")
def tu_rgb_to_packed422(x: torch.Tensor, code: int) -> torch.Tensor:
    """planar RGB (B,3,H,W) -> packed 4:2:2 frames (B,H,W,2): fp16 RGB -> yuyv422 / uyvy422 uint8, fp32 RGB -> y210 uint16; code = the
    frames' TU_U8 | TU_LAYOUT_YUYV / TU_LAYOUT_UYVY or TU_U16 | TU_LAYOUT_YUYV | colour bits"""
    lib = _lib.load()
    _require_cuda(x)
    w16 = (code & 0xFF) == _lib.TU_U16
    want = torch.float32 if w16 else torch.float16
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != want:
        raise RuntimeError(f"rgb_to_packed422 takes planar {str(want)[6:]} RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    out = torch.empty(_image_shape(B, 3, H, W, code), dtype=torch.uint16 if w16 else torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_packed422(x.data_ptr(), out.data_ptr(), None, code, B, H, W, _stream()))
    return out


@tu_rgb_to_packed422.register_fake
def _(x, code):
    w16 = (code & 0xFF) == _lib.TU_U16
    return x.new_empty(_image_shape(x.shape[0], 3, x.shape[2], x.shape[3], code), dtype=torch.uint16 if w16 else torch.uint8)


@torch.library.custom_op("tu::rgb_to_packed422_planes", mutates_args=("planes",), device_types="cuda")
def tu_rgb_to_packed422_planes(x: torch.Tensor, planes: List[torch.Tensor], code: int) -> None:
    """planar RGB (B,3,H,W) -> packed 4:2:2 frames (fp16 RGB for yuyv422 / uyvy422, fp32 for y210) written into the surfaces
    [s0, s1, ...], each (H, W, 2) with strides (row pitch, 2, 1)"""
    lib = _lib.load()
    _require_cuda(x)
    want = torch.float32 if (code & 0xFF) == _lib.TU_U16 else torch.float16
    if x.dim() != 4 or x.shape[1] != 3 or x.dtype != want:
        raise RuntimeError(f"rgb_to_packed422_planes takes planar {str(want)[6:]} RGB (B,3,H,W), got {x.dtype} {tuple(x.shape)}")
    x = x.contiguous()
    B, _, H, W = x.shape
    with torch.cuda.device(x.device):
        _lib.check(lib.tu_rgb_to_packed422(x.data_ptr(), None, _descriptors(planes, code), code, B, H, W, _stream()))


@tu_rgb_to_packed422_planes.register_fake
def _(x, planes, code):
    return None


def run_forward(pw_handle: int, model: str, x, res_out: Tuple[int, int], upscale_factor: Optional[int],
                require_ratio: bool, compute_bf16: bool, out_dtype: torch.dtype, clamp: bool = True,
                in_layout: str = "chw", out_layout: str = "chw", yuv: str = "bt709", out=None):
    """Shape logic of the three reference forwards (W:237-238, F:245-248,323-327, R:121-122) around tu::forward.
    in_layout / out_layout ('chw' | 'hwc' | 'hwc_bgr' | 'rgba' | 'bgra' | 'nv12' | 'p010' | 'yuv420p' | 'yuv444p' | 'yuv444p16' |
    'yuv420p10le' | 'yuv422p' | 'yuv422p10le' | 'yuv444p10le' | 'nv16' | 'p210' | 'yuyv422' | 'uyvy422' | 'y210'): uint8 frames may be
    interleaved (B,H,W,3), 4-byte pixels with alpha (B,H,W,4), NV12 or yuv420p (B,3H/2,W), yuv422p or nv16 (B,2H,W), yuv444p (B,3,H,W) or
    packed yuyv422 / uyvy422 (B,H,W,2) on either side, and either side may be P010 or yuv420p10le (B,3H/2,W), yuv422p10le or p210
    (B,2H,W), yuv444p16 or yuv444p10le (B,3,H,W), or y210 (B,H,W,2) uint16 frames (the *p10le words hold the code in their low 10 bits,
    the others in their high 10 bits); yuv ('bt709' | 'bt601' | 'bt709_full' |
    'bt601_full', and 'bt2020' | 'bt2020_full' with a 16-bit YUV side and no 8-bit one) is the colour of the YUV side(s).  An RGBA / BGRA
    output carries the input alpha resampled to the output size (tu_resample_alpha) when the input is RGBA / BGRA too, else alpha 255; an
    RGBA / BGRA input going to an output without alpha loses its alpha.
    Frame surfaces: with in_layout 'nv12' / 'p010' / 'nv16' / 'p210', x may be a list of B (y, uv) plane pairs (see plane_pairs), with a planar YUV
    in_layout a list of B (y, u, v) triples (see plane_triples), with a packed 4:2:2 in_layout a list of B (H, W, 2) surfaces (see
    packed_surfaces); with a YUV out_layout, out= a list of B such pairs / triples / surfaces receives the result and is returned."""
    il, ol = layout_code(in_layout), layout_code(out_layout)
    nv12_in, nv12_out = in_layout == "nv12", out_layout == "nv12"
    p010_in, p010_out = in_layout == "p010", out_layout == "p010"
    yuv_in, yuv_out = in_layout in YUV_LAYOUTS, out_layout in YUV_LAYOUTS
    yuvp_in, yuvp_out = in_layout in PLANAR, out_layout in PLANAR
    sp422_in, sp422_out = in_layout in SEMI422, out_layout in SEMI422
    pk422_in, pk422_out = in_layout in PACKED422, out_layout in PACKED422
    if yuv != "bt709" and not (yuv_in or yuv_out):
        raise ValueError(f"yuv={yuv!r} applies to NV12 / P010 frames only: pass in_layout / out_layout 'nv12' or 'p010'")
    yc = yuv_code(yuv)
    if yuv in YUV_P010:
        side16 = in_layout in YUV16_LAYOUTS or out_layout in YUV16_LAYOUTS
        side8 = (yuv_in and in_layout not in YUV16_LAYOUTS) or (yuv_out and out_layout not in YUV16_LAYOUTS)
        if (yuvp_in or yuvp_out or sp422_in or sp422_out or pk422_in or pk422_out) and (side8 or not side16):
            raise ValueError(f"yuv={yuv!r} (BT.2020) is defined for 10-bit frames: it needs a 16-bit YUV side ({', '.join(YUV16_LAYOUTS)}) "
                             "and no 8-bit YUV side (nv12, nv16, yuv420p, yuv422p, yuv444p, yuyv422, uyvy422)")
        if nv12_in or nv12_out or not (p010_in or p010_out or yuvp_in or yuvp_out or sp422_in or sp422_out or pk422_in or pk422_out):
            raise ValueError(f"yuv={yuv!r} (BT.2020) is defined for 10-bit frames: it needs a P010 side and no NV12 side")
    if nv12_out and out_dtype != torch.uint8:
        raise ValueError("out_layout='nv12' writes uint8 frames")
    if p010_out and out_dtype != torch.uint16:
        raise ValueError("out_layout='p010' writes uint16 frames")
    if yuvp_out and out_dtype != PLANAR[out_layout]:
        raise ValueError(f"out_layout={out_layout!r} writes {str(PLANAR[out_layout])[6:]} frames")
    if sp422_out and out_dtype != SEMI422[out_layout]:
        raise ValueError(f"out_layout={out_layout!r} writes {str(SEMI422[out_layout])[6:]} frames")
    if pk422_out and out_dtype != PACKED422[out_layout]:
        raise ValueError(f"out_layout={out_layout!r} writes {str(PACKED422[out_layout])[6:]} frames")
    px4_in, px4_out = in_layout in ("rgba", "bgra"), out_layout in ("rgba", "bgra")
    if px4_out and out_dtype != torch.uint8:
        raise ValueError(f"out_layout={out_layout!r} writes uint8 frames")
    if px4_in and not (isinstance(x, torch.Tensor) and x.dim() == 4 and x.shape[3] == 4 and x.dtype == torch.uint8):
        got = f"{x.dtype} {tuple(x.shape)}" if isinstance(x, torch.Tensor) else type(x).__name__
        raise ValueError(f"in_layout={in_layout!r} takes uint8 frames of shape (B, H, W, 4), got {got}")
    il |= yc if yuv_in else 0
    planes_in = isinstance(x, (list, tuple))
    if planes_in and not yuv_in:
        raise ValueError("a list of (y, uv) frame planes is NV12 / P010 input: pass in_layout='nv12' or 'p010'")
    if out is not None and not yuv_out:
        raise ValueError("out= takes NV12 / P010 frame planes: pass out_layout='nv12' or 'p010'")
    if planes_in:
        B, H, W = frame_planes(x, in_layout, "frames")
    elif nv12_in:
        H, W = _nv12_hw(x)
    elif p010_in:
        H, W = _p010_hw(x)
    elif yuvp_in or sp422_in or pk422_in:
        H, W = _yuvp_hw(x, in_layout)
    else:
        H, W = (int(x.shape[1]), int(x.shape[2])) if il else (int(x.shape[2]), int(x.shape[3]))
    if upscale_factor is not None:
        res_out = (H * upscale_factor, W * upscale_factor)
    res_out = (int(res_out[0]), int(res_out[1]))
    out_code = _code(out_dtype) | ol | (yc if yuv_out else 0)

    def even_out(oh, ow):
        if (nv12_out or p010_out) and (oh % 2 or ow % 2):
            raise ValueError(f"{'NV12' if nv12_out else 'P010'} output frames need an even height and width, got {oh}x{ow}")
        if out_layout in ("yuv420p", "yuv420p10le") and (oh % 2 or ow % 2):
            raise ValueError(f"{out_layout} output frames need an even height and width, got {oh}x{ow}")
        if out_layout in ("yuv422p", "yuv422p10le", *SEMI422, *PACKED422) and ow % 2:
            raise ValueError(f"{out_layout} output frames need an even width, got {oh}x{ow}")
        if out is not None:
            fmt = out_layout if yuvp_out or sp422_out or pk422_out else "NV12" if nv12_out else "P010"
            if not isinstance(out, (list, tuple)) or len(out) != (len(x) if planes_in else x.shape[0]):
                one = "(y, u, v) plane triple" if yuvp_out else "(H, W, 2) surface" if pk422_out else "(y, uv) plane pair"
                raise ValueError(f"out= must be a list of one {one} per input frame")
            n, h, w = frame_planes(out, out_layout, "out")
            dev = (x[0][0] if planes_in else x).device
            if (h, w) != (oh, ow) or out[0][0].device != dev:
                raise ValueError(f"out= planes must be {fmt} frames of {oh}x{ow} on {dev}, got {h}x{w} on {out[0][0].device}")

    def forward(oh, ow, scale_, code, clamp_):
        if not planes_in and out is None:
            return tu_forward(x, pw_handle, oh, ow, scale_, compute_bf16, code, clamp_, il)
        oplanes = _flat(out) if out is not None and code == out_code else []
        y = tu_forward_planes(None if planes_in else x, _flat(x) if planes_in else [], oplanes, pw_handle, oh, ow, scale_, compute_bf16,
                              code, clamp_, il)
        return out if oplanes else y

    if model != "FastTransformer":
        even_out(*res_out)
        return forward(res_out[0], res_out[1], 0, out_code, clamp)
    scale = upscale_factor if upscale_factor is not None else math.ceil(max(res_out[0] / H, res_out[1] / W))
    if scale not in (2, 3, 4, 6):
        raise ValueError(f"Requested scale={scale} was not built.")
    oh, ow = H * scale, W * scale
    # the reference tests res_out against (H_out, H_out) (sic): Resize is requested for every non-square
    # output and is the identity when the size already matches
    need_resize = require_ratio and res_out != (oh, oh) and res_out != (oh, ow)
    if not need_resize:
        even_out(oh, ow)
        return forward(oh, ow, scale, out_code, clamp)
    even_out(*res_out)
    # Resize is the last op: the un-clamped full-size image stays in the compute dtype and the Resize kernel writes the requested
    # output dtype / layout (uint8 frames: (out*255).clamp(0,255).to(uint8) fused into its store).  fp16 output keeps an fp32
    # intermediate, so that it is the fp32 result rounded once, at the Resize's store.  An 8-bit YUV output (NV12, NV16, yuv420p, yuv422p,
    # yuv444p, yuyv422, uyvy422) is the fp16 output converted, a 16-bit one (P010, P210, yuv444p16, *p10le, y210) the fp32 output converted
    yuv8_out = yuv_out and out_dtype == torch.uint8
    mid_code = _code(torch.bfloat16 if compute_bf16 and out_dtype in (torch.bfloat16, torch.uint8) and not yuv8_out else torch.float32)
    full = forward(oh, ow, scale, mid_code, False)
    if yuv_out:
        rgb = tu_resize_aa(full, res_out[0], res_out[1], clamp, _lib.TU_F16 if yuv8_out else _lib.TU_F32)
        if out is not None:
            (tu_rgb_to_yuvp_planes if yuvp_out else tu_rgb_to_yuv422sp_planes if sp422_out else tu_rgb_to_packed422_planes if pk422_out
             else tu_rgb_to_yuv420_planes)(rgb, _flat(out), out_code)
            return out
        if yuvp_out:
            return tu_rgb_to_yuvp(rgb, out_code)
        if sp422_out:
            return tu_rgb_to_yuv422sp(rgb, out_code)
        if pk422_out:
            return tu_rgb_to_packed422(rgb, out_code)
        return tu_rgb_to_nv12(rgb, out_code) if nv12_out else tu_rgb_to_p010(rgb, out_code)
    if px4_in and px4_out:
        # alpha is resampled straight from the input to the requested size, by the rule of every other output path
        return tu_resize_aa(full, res_out[0], res_out[1], clamp, out_code, tu_resample_alpha(x, _lib.TU_U8 | il, res_out[0], res_out[1]))
    return tu_resize_aa(full, res_out[0], res_out[1], clamp, out_code)
