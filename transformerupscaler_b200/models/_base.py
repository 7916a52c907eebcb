"""Shared scaffolding of the drop-in model classes.

The classes below only *hold parameters* under the reference's names and shapes so that
``load_state_dict(strict=True)`` of reference checkpoints works (SURVEY.md §8b); none of their
``forward`` methods does arithmetic.  ``EngineModel.forward`` routes the whole forward pass into
libtu_b200 through the ``tu::forward`` custom op.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.nn as nn

from .. import engine
from ..packing import PackedWeights


def _relative_position_index(ws: int) -> torch.Tensor:
    ys, xs = torch.meshgrid(torch.arange(ws), torch.arange(ws), indexing="ij")
    ys, xs = ys.reshape(-1), xs.reshape(-1)
    return (ys[:, None] - ys[None, :] + ws - 1) * (2 * ws - 1) + (xs[:, None] - xs[None, :] + ws - 1)


class _ParamsOnly(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover - never used
        raise RuntimeError("this sub-module only stores parameters; call TransformerModel.forward")


class WindowAttention(_ParamsOnly):
    """Parameter holder for reference WindowAttention (WindowTransformer/model.py:63-100)."""

    def __init__(self, dim: int, window_size: int, num_heads: int, dropout: float = 0.0):
        super().__init__()
        assert (dim // num_heads) * num_heads == dim, "dim must be divisible by num_heads"
        self.dim, self.window_size, self.num_heads = dim, window_size, num_heads
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.attn_drop = nn.Dropout(dropout)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(dropout)
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * window_size - 1) ** 2, num_heads))
        self.register_buffer("relative_position_index", _relative_position_index(window_size))
        nn.init.trunc_normal_(self.relative_position_bias_table, std=0.02)


def _mlp(dim: int, hidden: int, dropout: float) -> nn.Sequential:
    return nn.Sequential(nn.Linear(dim, hidden), nn.GELU(), nn.Linear(hidden, dim), nn.Dropout(dropout))


class WindowTransformerBlock(_ParamsOnly):
    """Parameter holder for reference WindowTransformerBlock (WindowTransformer/model.py:133-149)."""

    def __init__(self, dim: int, window_size: int, num_heads: int, mlp_ratio: float = 4.0, dropout: float = 0.1):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn = WindowAttention(dim, window_size, num_heads, dropout)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = _mlp(dim, int(dim * mlp_ratio), dropout)


class GlobalTransformerBlock(_ParamsOnly):
    """Parameter holder for ResidualTransformer's TransformerBlock (ResidualTransformer/model.py:22-38)."""

    def __init__(self, embed_dim: int, num_heads: int, mlp_ratio: float = 4.0, dropout: float = 0.1):
        super().__init__()
        self.norm1 = nn.LayerNorm(embed_dim)
        self.attn = nn.MultiheadAttention(embed_dim, num_heads, dropout=dropout, batch_first=True)
        self.norm2 = nn.LayerNorm(embed_dim)
        self.mlp = _mlp(embed_dim, int(embed_dim * mlp_ratio), dropout)


def _invalidate_after_load(module, incompatible_keys) -> None:
    module.invalidate_engine_cache()


class EngineModel(nn.Module):
    """Base of the three TransformerModel classes: precision selection, weight packing cache, dispatch."""

    ENGINE_MODEL = ""          # "WindowTransformer" | "FastTransformer" | "ResidualTransformer"
    AUTOCAST_OUT_FP32 = True   # reference output dtype under autocast: fp32 (Window/Residual), low precision (Fast)

    def __init__(self):
        super().__init__()
        # (compute_bf16, device) -> (key, PackedWeights, registry handle).  The PackedWeights objects are owned HERE; the engine's
        # registry only holds weak references, so deleting the module (or dropping the entry) frees the packed GPU tensors.
        self._tu_cache = {}
        self._tu_tensors = None      # cached [parameters..., buffers...] (walking the module tree costs ~0.5 ms per forward)
        # None = follow the reference's dtype semantics; "fp32" / "bf16" force the compute path
        self.engine_precision: Optional[str] = None
        self.register_load_state_dict_post_hook(_invalidate_after_load)

    # -- packing ------------------------------------------------------------------------------
    def invalidate_engine_cache(self) -> None:
        """Forget the packed weights (they are rebuilt by the next forward).  Called automatically by load_state_dict and by
        .to() / .cuda() / .float() / .bfloat16(); in-place edits of a parameter are detected through its version counter.  Only
        code that assigns NEW Parameter objects to sub-modules has to call this itself."""
        self._tu_cache = {}
        self._tu_tensors = None

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self.invalidate_engine_cache()
        return out

    # a copy.deepcopy / pickle of the module must not share the original's packed weights (both go through __getstate__)
    def __getstate__(self):
        st = dict(self.__dict__)
        st["_tu_cache"], st["_tu_tensors"] = {}, None
        return st

    def _packed(self, compute_bf16: bool, device: torch.device) -> int:
        if self._tu_tensors is None:
            self._tu_tensors = list(self.parameters()) + list(self.buffers())
        key = tuple([(t.data_ptr(), t._version) for t in self._tu_tensors])
        slot = (bool(compute_bf16), str(device))
        hit = self._tu_cache.get(slot)
        if hit is None or hit[0] != key:
            sd = {k: v for k, v in self.state_dict(keep_vars=True).items()}
            pw = PackedWeights(self.ENGINE_MODEL, sd, torch.bfloat16 if compute_bf16 else torch.float32, device)
            # The repacking kernels run on the caller's current stream.  Forwards may follow on OTHER streams (FramePipeline alternates
            # compute streams), so the packed tensors are complete before anyone can use them: one host wait per state_dict version.
            if torch.device(device).type == "cuda":
                torch.cuda.current_stream(device).synchronize()
            hit = (key, pw, engine.register_weights(pw))
            self._tu_cache[slot] = hit
        return hit[2]

    def _select_precision(self, x: torch.Tensor) -> Tuple[bool, torch.dtype]:
        """(compute in bf16?, output dtype) mirroring what the reference returns for this input/autocast state.  An fp16 module
        runs on the bf16 tensor-core path (or the fp32 one under engine_precision="fp32") and returns fp16: fp16 is an I/O dtype
        here, and the fp16 result is the fp32 result of that path rounded once."""
        pdt = self.conv1.weight.dtype
        if pdt not in (torch.float32, torch.bfloat16, torch.float16):
            raise TypeError(f"unsupported parameter dtype {pdt}: the engine runs fp32, bf16 or fp16 modules")
        autocast = x.is_cuda and torch.is_autocast_enabled("cuda")
        if self.engine_precision == "fp32":
            bf16 = False
        elif self.engine_precision == "bf16":
            bf16 = True
        else:
            bf16 = autocast or pdt != torch.float32
        if pdt != torch.float32:
            out_dt = pdt
        elif autocast and not self.AUTOCAST_OUT_FP32:
            out_dt = torch.bfloat16
        else:
            out_dt = torch.float32
        return bf16, out_dt

    def forward(self, x: torch.Tensor, res_out: Tuple[int, int] = (1080, 1920), upscale_factor: int = None,
                require_ratio: bool = True, in_layout: str = "chw", out_layout: str = "chw", yuv: str = "bt709", out=None):
        """The reference's signature (W:224, F:231, R:114) plus keyword-only-in-spirit extensions for uint8 video frames:
        in_layout / out_layout in {'chw', 'hwc', 'hwc_bgr', 'nv12'} — uint8 frames may arrive / leave interleaved (B,H,W,3), the form PIL
        and OpenCV hold them in (inference.py:65-70, app_overlay.py:382-386), with the channel swap done in the last kernel, or as
        NV12 video frames (B,3H/2,W), the form video decoders hand out and encoders take, converted on the GPU at both ends.
        'rgba' / 'bgra' on either side: 4-byte uint8 pixels (B,H,W,4) with a straight alpha byte (screen capture, swap chains, PNG),
        read and written like 'hwc' / 'hwc_bgr'.  The alpha never reaches the network: with RGBA / BGRA on both sides the output
        alpha is the input alpha resampled bicubically to the output size (rounded to the nearest code), else it is 255; an
        RGBA / BGRA input going to an output without alpha loses it.
        'p010' on either side: 10-bit P010 video frames (B,3H/2,W) uint16 (HEVC Main10, AV1, VP9 profile 2, HDR), code in the high
        10 bits of each word.  in_layout='p010' takes uint16 frames; out_layout='p010' returns uint16 frames for any frame input
        (uint8 in any layout, or P010), and a P010 input with any other out_layout returns uint8 frames.
        yuv in {'bt709', 'bt601', 'bt709_full', 'bt601_full'} is the colour matrix and range of the NV12 / P010 side(s); 'bt2020' and
        'bt2020_full' (BT.2020 / BT.2100) need a P010 side and no NV12 side.
        Decoder / encoder surfaces: with in_layout 'nv12' / 'p010', x may be a list of B (y, uv) plane pairs -- y (H, W), uv (H/2, W),
        uint8 (NV12) or uint16 (P010), unit stride along W and any row stride (strided views of a pitched surface pool) -- and with
        out_layout 'nv12' / 'p010', out= a list of B such pairs of the output size receives the result and is returned.  Each side is
        independent of the other; pitch padding and the bytes around the planes are never written.
        Planar YUV (FFmpeg's pix_fmt names) on either side: 'yuv420p' (I420) uint8 (B,3H/2,W) -- Y, then U and V of (H/2, W/2) --
        converted exactly as NV12; 'yuv444p' uint8 and 'yuv444p16' uint16 (B,3,H,W) planes Y, U, V at full resolution, the 16-bit
        words holding the code in the high 10 bits as P010 (in_layout='yuv444p16' takes uint16 frames; out_layout='yuv444p16' returns
        uint16 frames for any frame input).  Their surfaces are lists of B (y, u, v) plane triples, in x and in out=.
        4:2:2 and LSB-aligned 10-bit frames: 'yuv422p' uint8 (B,2H,W) -- Y, then U and V of (H, W/2) -- and 'nv16' uint8 / 'p210' uint16
        (B,2H,W) -- Y, then H rows of (U, V) pairs, p210 words holding the code in the high 10 bits; 'yuv420p10le' (B,3H/2,W),
        'yuv422p10le' (B,2H,W) and 'yuv444p10le' (B,3,H,W) uint16 with the code in the LOW 10 bits of each word (FFmpeg's software
        10-bit formats).  Surfaces: (y, uv) pairs for nv16 / p210, (y, u, v) triples for the planar ones.
        Packed 4:2:2 (FFmpeg's names), luma and chroma interleaved in one plane, (B,H,W,2) with W even: 'yuyv422' (YUY2: webcams, V4L2,
        Media Foundation) and 'uyvy422' (UYVY: capture cards, DeckLink, NDI) uint8, 'y210' uint16 words Y0 U Y1 V with the code in the
        high 10 bits (D3D11 / QSV / VAAPI 4:2:2 10-bit decoders).  Converted bitwise as the nv16 / p210 frame of the same samples.
        Surfaces: lists of B (H, W, 2) tensors with strides (row pitch, 2, 1), in x and in out=."""
        if isinstance(x, (list, tuple)):
            if in_layout not in engine.YUV_LAYOUTS:
                raise ValueError("a list of (y, uv) frame planes is NV12 / P010 input: pass in_layout='nv12' or 'p010'")
            engine.frame_planes(x, in_layout, "frames")
            x0 = x[0] if isinstance(x[0], torch.Tensor) else x[0][0]        # a packed 4:2:2 frame is one surface
            return self._forward(x, x0, res_out, upscale_factor, require_ratio, in_layout, out_layout, yuv, out)
        return self._forward(x, x, res_out, upscale_factor, require_ratio, in_layout, out_layout, yuv, out)

    def _forward(self, x, x0: torch.Tensor, res_out, upscale_factor, require_ratio, in_layout, out_layout, yuv, out):
        """x0: x, or the first plane of a list of frame planes (device, dtype and autocast state of the call)"""
        if self.training:
            raise RuntimeError("transformerupscaler_b200 is a forward-only inference engine: call .eval() first "
                               "(dropout is treated as identity; there is no backward)")
        if not x0.is_cuda:
            raise RuntimeError("transformerupscaler_b200 has no CPU path: move the model and the input to a CUDA device")
        if x0.requires_grad and torch.is_grad_enabled():
            raise RuntimeError("transformerupscaler_b200 is forward-only (no autograd): the input requires grad; call under torch.no_grad()")
        # uint8 frames in -> uint8 frames out (ToTensor scaling on read, (out*255).clamp(0,255).to(uint8) on write, fused into
        # the first and last kernels): the video-pipeline entry, an extension of the reference's float-only signature
        # 16-bit YUV frames are uint16; any other uint16 tensor is an image like any other and is read as float32
        if in_layout == "p010" and x0.dtype != torch.uint16:
            raise ValueError(f"in_layout='p010' takes uint16 frames (B, 3H/2, W), got {x0.dtype}")
        if in_layout == "yuv444p16" and x0.dtype != torch.uint16:
            raise ValueError(f"in_layout='yuv444p16' takes uint16 frames (B, 3, H, W), got {x0.dtype}")
        if in_layout in engine.YUV16_LAYOUTS and x0.dtype != torch.uint16:
            raise ValueError(f"in_layout={in_layout!r} takes uint16 frames, got {x0.dtype}")
        frames_u8 = x0.dtype == torch.uint8
        frames = frames_u8 or in_layout in engine.YUV16_LAYOUTS
        if x0.dtype not in (torch.float32, torch.bfloat16, torch.float16, torch.uint8) and not frames:
            x = x0 = x.float()
        bf16, out_dt = self._select_precision(x0)
        if frames:
            out_dt = torch.uint16 if out_layout in engine.YUV16_LAYOUTS else torch.uint8
        handle = self._packed(bf16, x0.device)
        if (in_layout != "chw" or out_layout != "chw") and not frames:
            raise ValueError("in_layout / out_layout other than 'chw' apply to uint8 / P010 frames only")
        if out is not None and out_layout not in engine.YUV_LAYOUTS:
            raise ValueError("out= takes NV12 / P010 frame planes: pass out_layout='nv12' or 'p010'")
        y = engine.run_forward(handle, self.ENGINE_MODEL, x, res_out, upscale_factor, require_ratio, bf16, out_dt,
                               in_layout=in_layout, out_layout=out_layout, yuv=yuv, out=out)
        if out is not None:
            return y
        out = y
        if not frames and x0.is_cuda and torch.is_autocast_enabled("cuda") and not self.AUTOCAST_OUT_FP32:
            want = torch.get_autocast_dtype("cuda")
            if out.dtype != want:
                out = out.to(want)
        return out
