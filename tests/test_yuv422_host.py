"""CPU: 4:2:2 frames (yuv422p, nv16, p210, yuv422p10le) and LSB-aligned 10-bit planar frames (yuv420p10le, yuv422p10le, yuv444p10le) --
the conversion oracle, its agreement with a float64 evaluation of the defining equations and with the NV12 / P010 / yuv444p16 oracles,
the two 4:2:2 identities, the C-ABI constants and symbols, every host-side rejection of the single ops, the forward and the workspace
queries (all made before anything is enqueued, so they run without a GPU), the workspace sizes of every code pair, and the Python-side
errors and fake shapes.

The oracle functions below are the definition the kernels of csrc/resample.cu follow operation for operation: plain fp32 torch ops on
the CPU, each one correctly rounded, no fused multiply-add.  tests/test_gpu_yuv422.py compares the kernels with them bit for bit."""
import ctypes as C
import os
import re

import pytest
import torch

from tests.test_nv12_host import _geometry, _packed, _upsample, coefficients, oracle_nv12_to_rgb, oracle_rgb_to_nv12
from tests.test_p010_host import COLOURS10, MATRIX, coefficients10, oracle_p010_to_rgb, oracle_rgb_to_p010
from tests.test_yuvp_host import (COLOURS8, FAKE, _to_rgb, both_ops, expect, frames3, oracle_rgb_to_yuv444, oracle_yuv444_to_rgb,
                                  split420)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U8, U16 = torch.uint8, torch.uint16
# the new layouts: FFmpeg's pix_fmt name -> (chroma subsampling, frame dtype, semi-planar)
NEW = {"yuv420p10le": ("420", U16, False), "yuv422p": ("422", U8, False), "yuv422p10le": ("422", U16, False),
       "yuv444p10le": ("444", U16, False), "nv16": ("422", U8, True), "p210": ("422", U16, True)}


def code(fmt, yuv="bt709"):
    from transformerupscaler_b200 import _lib as L, engine
    return (L.TU_U16 if NEW[fmt][1] == U16 else L.TU_U8) | engine.LAYOUTS[fmt] | engine.yuv_code(yuv)


def is16(fmt):
    return NEW[fmt][1] == U16


def colours(fmt):
    return COLOURS10 if is16(fmt) else COLOURS8


def dense_shape(fmt, B, H, W):
    return {"420": (B, 3 * H // 2, W), "422": (B, 2 * H, W), "444": (B, 3, H, W)}[NEW[fmt][0]]


def read_codes(words, fmt):
    """stored samples -> int32 codes: bytes as they are, p210 words >> 6, LSB words min(word, 1023)"""
    c = words.cpu().to(torch.int32) & 0xFFFF
    if fmt == "p210":
        return c >> 6
    return c.clamp(max=1023) if fmt.endswith("10le") else c


def write_codes(c, fmt):
    c = c.to(torch.int32)
    if fmt == "p210":
        return (c << 6).to(U16)
    return c.to(U16 if is16(fmt) else U8)


def to_planes(f, fmt):
    """dense frames -> the stored Y, U, V planes (B, h, w)"""
    sub, _, semi = NEW[fmt]
    if sub == "444":
        return f[:, 0], f[:, 1], f[:, 2]
    if sub == "420":
        return split420(f)
    B, R, W = f.shape
    H = R // 2
    if semi:
        ch = f[:, H:].reshape(B, H, W // 2, 2)
        return f[:, :H], ch[..., 0], ch[..., 1]
    flat = f.reshape(B, -1)
    n = H * W
    return flat[:, :n].reshape(B, H, W), flat[:, n:n + n // 2].reshape(B, H, W // 2), flat[:, n + n // 2:].reshape(B, H, W // 2)


def from_planes(y, u, v, fmt):
    sub, _, semi = NEW[fmt]
    if sub == "444":
        return torch.stack([y, u, v], 1)
    B, H, W = y.shape
    if semi:
        return torch.cat([y, torch.stack([u, v], -1).reshape(B, H, W)], 1)
    return torch.cat([y.reshape(B, -1), u.reshape(B, -1), v.reshape(B, -1)], 1).reshape(dense_shape(fmt, B, H, W))


def upsample422(c):
    """(B, H, W/2) chroma codes -> (B, H, W): column 2j takes C[j], column 2j+1 (C[j] + C[j+1]) / 2 (j+1 clamped); exact in fp32"""
    right = torch.cat([c[..., 1:], c[..., -1:]], -1)
    return torch.stack([c, (c + right) * 0.5], -1).reshape(c.shape[0], c.shape[1], 2 * c.shape[2])


def oracle_to_rgb(f, fmt, yuv="bt709"):
    """frames of a new layout -> planar RGB (B, 3, H, W) fp32 clamped to [0, 1] (the 8-bit kernels store it rounded to fp16)"""
    y, u, v = (read_codes(p, fmt).float() for p in to_planes(f.cpu(), fmt))
    H, W = y.shape[1:]
    up = {"420": lambda c: _upsample(c, H, W), "422": upsample422, "444": lambda c: c}[NEW[fmt][0]]
    k, mid = (coefficients10(yuv), 512.0) if is16(fmt) else (coefficients(yuv), 128.0)
    return _to_rgb(y, up(u), up(v), k, mid)


def _code(v, cmax):
    return torch.floor(v + 0.5).clamp(0, cmax).to(torch.int32)


def oracle_from_rgb(rgb, fmt, yuv="bt709"):
    """planar RGB (B, 3, H, W) (fp16 values for 8-bit layouts, fp32 for 16-bit) -> frames of a new layout"""
    sub = NEW[fmt][0]
    if fmt == "yuv420p10le":                       # P010's codes in the low bits of separate U and V planes
        c = oracle_rgb_to_p010(rgb, yuv).to(torch.int32) >> 6
        B, R, W = c.shape
        H = R * 2 // 3
        ch = c[:, H:].reshape(B, H // 2, W // 2, 2)
        return from_planes(c[:, :H], ch[..., 0], ch[..., 1], fmt).to(U16)
    if sub == "444":                               # yuv444p16's codes in the low bits
        return (oracle_rgb_to_yuv444(rgb, yuv, True).to(torch.int32) >> 6).to(U16)
    p = rgb.cpu().float()
    k, mid, cmax = (coefficients10(yuv), 512.0, 1023) if is16(fmt) else (coefficients(yuv), 128.0, 255)
    yl = (k["kr"] * p[:, 0] + k["kg"] * p[:, 1]) + k["kb"] * p[:, 2]
    c1, c2 = p[..., 0::2], p[..., 1::2]                        # columns 2j, 2j+1 of each row
    c0 = torch.cat([c1[..., :1], c2[..., :-1]], -1)            # column 2j-1, clamped at 0
    bar = ((c0 + 2 * c1) + c2) * 0.25
    cb = (k["cb_r"] * bar[:, 0] + k["cb_g"] * bar[:, 1]) + 0.5 * bar[:, 2]
    cr = (0.5 * bar[:, 0] + k["cr_g"] * bar[:, 1]) + k["cr_b"] * bar[:, 2]
    return from_planes(write_codes(_code(k["ys"] * yl + k["yo"], cmax), fmt), write_codes(_code(k["cs"] * cb + mid, cmax), fmt),
                       write_codes(_code(k["cs"] * cr + mid, cmax), fmt), fmt)


def random_frames(fmt, B, H, W, seed, hi=None):
    """random stored samples; 16-bit layouts draw whole words (LSB words above 1023 included)"""
    g = torch.Generator().manual_seed(seed)
    hi = hi or (65536 if is16(fmt) else 256)
    return torch.randint(0, hi, dense_shape(fmt, B, H, W), generator=g, dtype=torch.int32).to(NEW[fmt][1])


# ---------------------------------------------------------------------------------------------------------------------------------
# the oracle
def _f64_to_rgb(Y, U, V, yuv, w16):
    kr, kb = MATRIX[yuv.split("_")[0]]
    full = yuv.endswith("_full")
    yo, ys, cs, mid = ((0.0, 1023.0, 1023.0, 512.0) if full else (64.0, 876.0, 896.0, 512.0)) if w16 else \
        ((0.0, 255.0, 255.0, 128.0) if full else (16.0, 219.0, 224.0, 128.0))
    kg = 1.0 - kr - kb
    y, u, v = (Y - yo) / ys, (U - mid) / cs, (V - mid) / cs
    return torch.stack([y + 2 * (1 - kr) * v, y - 2 * (1 - kb) * kb / kg * u - 2 * (1 - kr) * kr / kg * v, y + 2 * (1 - kb) * u],
                       1).clamp(0, 1)


@pytest.mark.parametrize("fmt", ["yuv422p", "yuv422p10le"])
def test_422_oracle_matches_float64_equations(fmt):
    """random frames, every colour: within one code of the float64 equations on the float64-upsampled chroma (in fact far closer);
    the from-RGB codes within one of the float64 rounding of the equations on the float64 filter"""
    w16, cmax = is16(fmt), 1023 if is16(fmt) else 255
    f = random_frames(fmt, 4, 6, 34, seed=1, hi=cmax + 1)
    y, u, v = (read_codes(p, fmt).double() for p in to_planes(f, fmt))
    g = torch.Generator().manual_seed(2)
    rgb = torch.rand(4, 3, 6, 34, generator=g)
    rgb = rgb if w16 else rgb.half()
    p = rgb.double()
    for yuv in colours(fmt):
        err = (oracle_to_rgb(f, fmt, yuv).double() - _f64_to_rgb(y, upsample422(u), upsample422(v), yuv, w16)).abs().max().item()
        assert err * cmax <= 1 and err < 1e-6, (yuv, err)
        kr, kb = MATRIX[yuv.split("_")[0]]
        kg, full = 1.0 - kr - kb, yuv.endswith("_full")
        yo, ys, cs, mid = ((0.0, cmax, cmax) if full else ((64.0, 876.0, 896.0) if w16 else (16.0, 219.0, 224.0))) + \
            ((512.0,) if w16 else (128.0,))
        got = [read_codes(t, fmt).double() for t in to_planes(oracle_from_rgb(rgb, fmt, yuv), fmt)]
        yl = kr * p[:, 0] + kg * p[:, 1] + kb * p[:, 2]
        c0 = torch.cat([p[..., :1], p[..., 1::2][..., :-1]], -1)
        bar = (c0 + 2 * p[..., 0::2] + p[..., 1::2]) / 4
        ybar = kr * bar[:, 0] + kg * bar[:, 1] + kb * bar[:, 2]
        want = [torch.floor(ys * yl + yo + 0.5).clamp(0, cmax), torch.floor(cs * (bar[:, 2] - ybar) / (2 * (1 - kb)) + mid + 0.5).clamp(0, cmax),
                torch.floor(cs * (bar[:, 0] - ybar) / (2 * (1 - kr)) + mid + 0.5).clamp(0, cmax)]
        for a, b in zip(got, want):
            assert (a - b).abs().max().item() <= 1, yuv


@pytest.mark.parametrize("fmt", ["yuv422p", "yuv422p10le", "nv16", "p210"])
def test_422_exact_endpoints(fmt):
    w16 = is16(fmt)
    for yuv in colours(fmt):
        full = yuv.endswith("_full")
        lo, hi = (0, 1023 if w16 else 255) if full else ((64, 940) if w16 else (16, 235))
        mid = 512 if w16 else 128
        y = torch.tensor([lo, hi], dtype=torch.int32)[:, None, None].expand(2, 3, 4)
        c = torch.full((2, 3, 2), mid, dtype=torch.int32)
        f = from_planes(write_codes(y, fmt), write_codes(c, fmt), write_codes(c, fmt), fmt)
        rgb = oracle_to_rgb(f, fmt, yuv)
        assert torch.equal(rgb[0], torch.zeros(3, 3, 4)) and torch.equal(rgb[1], torch.ones(3, 3, 4)), yuv
        assert torch.equal(oracle_from_rgb(rgb if w16 else rgb.half(), fmt, yuv), f), yuv


def test_lsb_oracles_are_the_msb_oracles_on_shifted_words():
    """yuv420p10le is P010 with the words >> 6 and the chroma de-interleaved, yuv444p10le is yuv444p16 with the words >> 6, p210 /
    yuv422p10le likewise; an LSB word above 1023 reads as 1023"""
    g = torch.Generator().manual_seed(5)
    B, H, W = 2, 6, 10
    lsb = random_frames("yuv420p10le", B, H, W, seed=3)                  # stray high bits included
    sat = read_codes(lsb, "yuv420p10le")
    assert int(sat.max()) == 1023 and bool((lsb.to(torch.int32) & 0xFFFF > 1023).any())
    y, u, v = to_planes(sat, "yuv420p10le")
    p010 = (torch.cat([y, torch.stack([u, v], -1).reshape(B, H // 2, W)], 1) << 6).to(U16)
    f444 = random_frames("yuv444p10le", B, H, W, seed=4)
    rgb = torch.rand(B, 3, H, W, generator=g) * 1.4 - 0.2
    for yuv in COLOURS10:
        assert torch.equal(oracle_to_rgb(lsb, "yuv420p10le", yuv), oracle_p010_to_rgb(p010, yuv)), yuv
        assert torch.equal(oracle_to_rgb(f444, "yuv444p10le", yuv),
                           oracle_yuv444_to_rgb((read_codes(f444, "yuv444p10le") << 6).to(U16), yuv)), yuv
        out = oracle_from_rgb(rgb, "yuv420p10le", yuv).to(torch.int32)
        assert int(out.max()) <= 1023
        y2, u2, v2 = to_planes(out, "yuv420p10le")
        assert torch.equal(torch.cat([y2, torch.stack([u2, v2], -1).reshape(B, H // 2, W)], 1) << 6,
                           oracle_rgb_to_p010(rgb, yuv).to(torch.int32)), yuv
        assert torch.equal(oracle_from_rgb(rgb, "yuv444p10le", yuv).to(torch.int32) << 6,
                           oracle_rgb_to_yuv444(rgb, yuv, True).to(torch.int32)), yuv
        f = random_frames("yuv422p10le", B, H, W, seed=6)
        pl = [read_codes(t, "yuv422p10le") for t in to_planes(f, "yuv422p10le")]
        assert torch.equal(oracle_to_rgb(f, "yuv422p10le", yuv), oracle_to_rgb(from_planes(*[write_codes(t, "p210") for t in pl], "p210"),
                                                                               "p210", yuv)), yuv
        a = [read_codes(t, "yuv422p10le") for t in to_planes(oracle_from_rgb(rgb, "yuv422p10le", yuv), "yuv422p10le")]
        b = [read_codes(t, "p210") for t in to_planes(oracle_from_rgb(rgb, "p210", yuv), "p210")]
        assert all(torch.equal(x, z) for x, z in zip(a, b)), yuv


def test_yuv422p_oracle_is_the_nv16_oracle_interleaved():
    g = torch.Generator().manual_seed(8)
    for B, H, W in ((2, 5, 10), (1, 1, 2), (3, 4, 6)):
        f = random_frames("yuv422p", B, H, W, seed=H + W)
        nv16 = from_planes(*to_planes(f, "yuv422p"), "nv16")
        assert torch.equal(from_planes(*to_planes(nv16, "nv16"), "yuv422p"), f)
        rgb = torch.rand(B, 3, H, W, generator=g).half()
        for yuv in COLOURS8:
            assert torch.equal(oracle_to_rgb(f, "yuv422p", yuv), oracle_to_rgb(nv16, "nv16", yuv))
            assert torch.equal(from_planes(*to_planes(oracle_from_rgb(rgb, "yuv422p", yuv), "yuv422p"), "nv16"),
                               oracle_from_rgb(rgb, "nv16", yuv))


def identity_pairs_image(B, H, W, seed, w16):
    """an RGB image whose rows come in equal pairs (values outside [0, 1] too)"""
    half = torch.rand(B, 3, H // 2, W, generator=torch.Generator().manual_seed(seed)) * 1.4 - 0.2
    rgb = half.repeat_interleave(2, 2)
    return rgb if w16 else rgb.half()


@pytest.mark.parametrize("fmt", ["nv16", "p210", "yuv422p", "yuv422p10le"])
def test_identity_equal_row_pairs_give_the_420_chroma(fmt):
    """identity 1: the 4:2:2 chroma rows 2i and 2i+1 of an image whose rows come in equal pairs are the NV12 / P010 chroma row i, and
    its luma is NV12's / P010's"""
    B, H, W = 2, 8, 14
    w16 = is16(fmt)
    rgb = identity_pairs_image(B, H, W, seed=9, w16=w16)
    for yuv in colours(fmt):
        y, u, v = (read_codes(t, fmt) for t in to_planes(oracle_from_rgb(rgb, fmt, yuv), fmt))
        f420 = (oracle_rgb_to_p010(rgb, yuv).to(torch.int32) >> 6) if w16 else oracle_rgb_to_nv12(rgb, yuv).to(torch.int32)
        ch = f420[:, H:].reshape(B, H // 2, W // 2, 2)
        assert torch.equal(y, f420[:, :H]), yuv
        assert torch.equal(u, ch[..., 0].repeat_interleave(2, 1)) and torch.equal(v, ch[..., 1].repeat_interleave(2, 1)), yuv


@pytest.mark.parametrize("fmt", ["nv16", "p210", "yuv422p", "yuv422p10le"])
def test_identity_row_constant_chroma_is_444(fmt):
    """identity 2: a 4:2:2 frame whose chroma is constant along each row converts to the RGB of the yuv444p (8-bit) / yuv444p16 frame
    holding that chroma at every pixel"""
    B, H, W = 2, 5, 12
    w16, cmax = is16(fmt), 1023 if is16(fmt) else 255
    g = torch.Generator().manual_seed(10)
    y = torch.randint(0, cmax + 1, (B, H, W), generator=g, dtype=torch.int32)
    u, v = (torch.randint(0, cmax + 1, (B, H, 1), generator=g, dtype=torch.int32) for _ in range(2))
    f = from_planes(write_codes(y, fmt), write_codes(u.expand(B, H, W // 2), fmt), write_codes(v.expand(B, H, W // 2), fmt), fmt)
    f444 = torch.stack([y, u.expand(B, H, W), v.expand(B, H, W)], 1)
    f444 = (f444 << 6).to(U16) if w16 else f444.to(U8)
    for yuv in colours(fmt):
        assert torch.equal(oracle_to_rgb(f, fmt, yuv), oracle_yuv444_to_rgb(f444, yuv)), yuv


# ---------------------------------------------------------------------------------------------------------------------------------
# the C ABI
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from transformerupscaler_b200 import _lib
    return _lib.load()


def L():
    from transformerupscaler_b200 import _lib
    return _lib


def test_abi_constants_and_symbols(lib):
    from transformerupscaler_b200 import _lib, engine
    src = open(os.path.join(ROOT, "include", "tu_b200.h")).read()
    for name, val in (("TU_LAYOUT_YUV422P", 0x900), ("TU_LAYOUT_NV16", 0xA00), ("TU_YUV_LSB10", 0x10000)):
        assert re.search(r"#define\s+%s\s+0x%x\b" % (name, val), src, re.I), name
        assert getattr(_lib, name) == val
    for name, expr in (("TU_U8_YUV422P", r"\(TU_U8 \| TU_LAYOUT_YUV422P\)"), ("TU_U8_NV16", r"\(TU_U8 \| TU_LAYOUT_NV16\)"),
                       ("TU_U16_P210", r"\(TU_U16 \| TU_LAYOUT_NV16\)"),
                       ("TU_U16_YUV420P10", r"\(TU_U16 \| TU_LAYOUT_YUV420P \| TU_YUV_LSB10\)"),
                       ("TU_U16_YUV422P10", r"\(TU_U16 \| TU_LAYOUT_YUV422P \| TU_YUV_LSB10\)"),
                       ("TU_U16_YUV444P10", r"\(TU_U16 \| TU_LAYOUT_YUV444P \| TU_YUV_LSB10\)")):
        assert re.search(r"#define\s+%s\s+%s" % (name, expr), src), name
    for n in ("tu_yuv422sp_to_rgb", "tu_rgb_to_yuv422sp"):
        assert hasattr(lib, n) and n in _lib.SIGNATURES and re.search(r"\b%s\(" % n, src), n
    for n in ("yuv422p_to_rgb", "rgb_to_p210", "nv16_to_rgb", "rgb_to_yuv420p10le", "yuv444p10le_to_rgb", "rgb_to_yuv422p10le"):
        assert '"%s"' % n in src, n
    assert engine.LAYOUTS["yuv422p"] == 0x900 and engine.LAYOUTS["nv16"] == engine.LAYOUTS["p210"] == 0xA00
    assert engine.LAYOUTS["yuv420p10le"] == 0x10600 and engine.LAYOUTS["yuv444p10le"] == 0x10700
    for fmt in NEW:
        assert engine._image_shape(2, 3, 6, 10, code(fmt)) == dense_shape(fmt, 2, 6, 10), fmt
    assert not engine._is_nv12(0xA00) and not engine._is_px4(0x900) and not engine._is_p010(0xA00)


def bad_codes():
    """every invalid combination the new codes border on"""
    _l = L()
    U8_, U16_, LSB = _l.TU_U8, _l.TU_U16, _l.TU_YUV_LSB10
    p422, nv16 = U8_ | _l.TU_LAYOUT_YUV422P, U8_ | _l.TU_LAYOUT_NV16
    return (U16_ | _l.TU_LAYOUT_YUV420P, U16_ | _l.TU_LAYOUT_YUV422P,                                 # MSB planar 4:2:0 / 4:2:2
            p422 | LSB, nv16 | LSB, U8_ | _l.TU_LAYOUT_YUV420P | LSB, U8_ | _l.TU_LAYOUT_YUV444P | LSB,  # LSB with TU_U8
            U16_ | _l.TU_LAYOUT_NV16 | LSB, U16_ | _l.TU_LAYOUT_P010 | LSB, U8_ | _l.TU_LAYOUT_NV12 | LSB,  # LSB with a semi-planar layout
            _l.TU_F32 | LSB, _l.TU_F16 | LSB, U8_ | LSB, U8_ | _l.TU_LAYOUT_HWC | LSB, U8_ | _l.TU_LAYOUT_RGBA | LSB,  # non-YUV layouts
            p422 | _l.TU_YUV_BT2020, nv16 | _l.TU_YUV_BT2020,                                          # BT.2020 on 8-bit codes
            code("p210") | _l.TU_YUV_BT601 | _l.TU_YUV_BT2020, code("yuv422p10le") | _l.TU_YUV_BT601 | _l.TU_YUV_BT2020,
            code("yuv420p10le") | _l.TU_YUV_BT601 | _l.TU_YUV_BT2020, code("yuv444p10le") | _l.TU_YUV_BT601 | _l.TU_YUV_BT2020,
            _l.TU_F32 | _l.TU_LAYOUT_YUV422P, _l.TU_F16 | _l.TU_LAYOUT_NV16, _l.TU_BF16 | _l.TU_LAYOUT_NV16)


def chroma_w(fmt, W):
    return W if NEW[fmt][0] == "444" else W // 2


def planes_of_new(fmt, B, H, W, pitch_extra=256):
    """B valid descriptors (fake, aligned addresses) of a new layout: TuFramePlanes3 for the planar ones, TuFramePlanes for nv16 / p210"""
    s = 2 if is16(fmt) else 1
    base = [FAKE + b * (1 << 20) for b in range(B)]
    if NEW[fmt][2]:
        P = L().TuFramePlanes
        return (P * B)(*[P(a, a + (1 << 19), W * s + pitch_extra, W * s + pitch_extra) for a in base])
    P, cw = L().TuFramePlanes3, chroma_w(fmt, W)
    return (P * B)(*[P(a, a + (1 << 18), a + (1 << 19), W * s + pitch_extra, cw * s + pitch_extra, cw * s + pitch_extra) for a in base])


def ops(lib, fmt_or_semi, dense, fr, c, B, H, W, rgb=FAKE):
    """both single ops of a side kind: the planar ones, or the semi-planar 4:2:2 ones"""
    if fmt_or_semi is True or (fmt_or_semi in NEW and NEW[fmt_or_semi][2]):
        return [(lib.tu_yuv422sp_to_rgb(dense, fr, c, rgb, B, H, W, None), L().last_error()),
                (lib.tu_rgb_to_yuv422sp(rgb, dense, fr, c, B, H, W, None), L().last_error())]
    return both_ops(lib, dense, fr, c, B, H, W, rgb)


def test_single_ops_reject_codes_and_arguments(lib):
    _l = L()
    P2 = _l.TuFramePlanes
    pairs = (P2 * 1)(P2(FAKE, FAKE + 8192, 256, 256))
    planar_others = (code("yuv420p10le"), code("yuv422p"), code("yuv422p10le"), code("yuv444p10le"))
    for c in bad_codes():
        expect(ops(lib, False, FAKE, None, c, 1, 4, 4), "code must be")
        expect(ops(lib, True, FAKE, None, c, 1, 4, 4), "code must be")
    # the semi-planar ops take NV16 / P210 only, the planar ops never take them
    for c in planar_others + (_l.TU_U8 | _l.TU_LAYOUT_NV12, _l.TU_U16 | _l.TU_LAYOUT_P010, _l.TU_U16 | _l.TU_LAYOUT_YUV444P):
        expect(ops(lib, True, FAKE, None, c, 1, 4, 4), "code must be")
        expect(ops(lib, True, None, pairs, c, 1, 4, 4), "code must be")
    for fmt in ("nv16", "p210"):
        expect(ops(lib, False, FAKE, None, code(fmt), 1, 4, 4), "code must be")
    # the 4:2:0 surface ops never take NV16 / P210
    for fmt in ("nv16", "p210"):
        rc = lib.tu_yuv420_planes_to_rgb(pairs, code(fmt), FAKE, 1, 4, 4, None)
        assert rc == _l.TU_ERR_ARG and "NV12" in _l.last_error()
    for fmt in NEW:
        c, semi, w16 = code(fmt), NEW[fmt][2], is16(fmt)
        expect(ops(lib, fmt, FAKE, planes_of_new(fmt, 1, 4, 4), c, 1, 4, 4), "exactly one")
        expect(ops(lib, fmt, None, None, c, 1, 4, 4), "exactly one")
        for B, H, W in ((0, 4, 4), (65536, 4, 4), (1, 0, 4), (1, 4, 0)):
            expect(ops(lib, fmt, FAKE, None, c, B, H, W), "bad argument")
        expect(ops(lib, fmt, FAKE, None, c, 1, 4, 4, rgb=None), "bad argument")
        # pairs of RGB values are one access for 4:2:0 / 4:2:2 (4 bytes fp16, 8 bytes fp32), single elements for 4:4:4
        ra = (2 if NEW[fmt][0] != "444" else 1) * (4 if w16 else 2)
        expect(ops(lib, fmt, FAKE, None, c, 1, 4, 4, rgb=FAKE + ra // 2), "RGB buffer", "fp32" if w16 else "fp16", "%d-byte" % ra)
        fa = (2 if NEW[fmt][0] != "444" else 1) * (2 if w16 else 1)
        expect(ops(lib, fmt, FAKE + fa // 2, None, c, 1, 4, 4), "dense", "%d-byte aligned" % fa)
        expect(ops(lib, fmt, FAKE, None, c, 1, 30000, 30000), "too large")
        if NEW[fmt][0] != "444":
            expect(ops(lib, fmt, FAKE, None, c, 1, 4, 5), "even")
            expect(ops(lib, fmt, None, planes_of_new(fmt, 1, 4, 6), c, 1, 4, 5), "even")
    for fmt in ("yuv422p", "yuv422p10le", "nv16", "p210", "yuv444p10le"):       # any height
        for rc, msg in ops(lib, fmt, FAKE, None, code(fmt), 1, 3, 4, rgb=None):
            assert "bad argument" in msg
    expect(ops(lib, "yuv420p10le", FAKE, None, code("yuv420p10le"), 1, 3, 4), "yuv420p10le", "even height and width")


@pytest.mark.parametrize("fmt", list(NEW))
def test_descriptor_rejections(lib, fmt):
    c, semi, w16 = code(fmt), NEW[fmt][2], is16(fmt)
    B, H, W = 3, 6, 10
    s = 2 if w16 else 1
    fields = ("y", "uv") if semi else ("y", "u", "v")
    rows = {"y": W, "uv": W, "u": chroma_w(fmt, W), "v": chroma_w(fmt, W)}
    for f in fields:
        fr = planes_of_new(fmt, B, H, W)
        setattr(fr[1], f, None)
        expect(ops(lib, fmt, None, fr, c, B, H, W), "frame 1", f"{f} is NULL")
        fr = planes_of_new(fmt, B, H, W)
        setattr(fr[2], f + "_pitch", (rows[f] - 1) * s)
        expect(ops(lib, fmt, None, fr, c, B, H, W), "frame 2", f + "_pitch")
    # alignment: the luma pair is one access on 4:2:0 / 4:2:2 (2 bytes 8-bit, 4 bytes 16-bit), nv16 / p210 chroma pairs too; every 16-bit
    # plane is one word per sample; 8-bit planar chroma may sit anywhere
    pair = NEW[fmt][0] != "444"
    need = {"y": (2 * s if pair else s), "uv": 2 * s, "u": s, "v": s}
    for f in fields:
        for field in (f, f + "_pitch"):
            for off in (1, 2):
                if off >= need[f]:
                    continue
                fr = planes_of_new(fmt, B, H, W)
                setattr(fr[0], field, getattr(fr[0], field) + off)
                expect(ops(lib, fmt, None, fr, c, B, H, W), "frame 0", f, "multiple")
        if need[f] == 1:
            fr = planes_of_new(fmt, B, H, W)
            setattr(fr[0], f, getattr(fr[0], f) + 1)
            assert all("bad argument" in m for _, m in ops(lib, fmt, None, fr, c, B, H, W, rgb=None))
    if not pair:
        expect(ops(lib, fmt, None, planes_of_new(fmt, 1, 70000, 8), c, 1, 70000, 8), "65535 rows")


def test_forward_rejections_before_any_launch(lib):
    _l = L()
    pw = _packed("WindowTransformer", torch.bfloat16)
    w = C.byref(pw.struct)
    B, H, W, oh, ow = 2, 72, 104, 108, 156

    def fwd(x, xfr, i, o, ofr, oc, Hn=H, Wn=W, ohn=oh, own=ow):
        rc = lib.tu_forward_frames(w, x, xfr, i, o, ofr, oc, B, Hn, Wn, ohn, own, 0, _l.TU_BF16, 1, FAKE, 1 << 40, None)
        return rc, _l.last_error()

    for c in bad_codes():
        expect([fwd(FAKE, None, c, FAKE, None, _l.TU_F32)], "TU_LAYOUT_")
        expect([fwd(FAKE, None, _l.TU_F32, FAKE, None, c)], "TU_LAYOUT_")
        assert lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, c, _l.TU_F32) == 0, hex(c)
        assert lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, _l.TU_F32, c) == 0, hex(c)
    for fmt in ("yuv422p", "yuv422p10le", "nv16", "p210"):
        expect([fwd(FAKE, None, code(fmt), FAKE, None, _l.TU_F32, Wn=W + 1)], "4:2:2 input", "even width")
        expect([fwd(FAKE, None, _l.TU_F32, FAKE, None, code(fmt), own=ow + 1)], "4:2:2 output", "even width")
        assert lib.tu_forward_workspace_bytes_io(w, B, H, W + 1, oh, ow, 0, _l.TU_BF16, code(fmt), _l.TU_F32) == 0
        assert lib.tu_forward_workspace_bytes_io(w, B, H + 1, W, oh + 1, ow, 0, _l.TU_BF16, code(fmt), code(fmt)) > 0   # any height
    expect([fwd(FAKE, None, code("yuv420p10le"), FAKE, None, _l.TU_F32, Hn=H + 1)], "yuv420p10le input", "even")
    expect([fwd(FAKE, None, _l.TU_F32, FAKE, None, code("yuv420p10le"), ohn=oh + 1)], "yuv420p10le output", "even")
    # descriptors are read as the side's type, and a bad one names the side, the frame and the field
    bad = planes_of_new("p210", B, H, W)
    bad[1].uv_pitch = 2 * W - 2
    expect([fwd(None, bad, code("p210"), FAKE, None, _l.TU_F32)], "x_frames", "frame 1", "uv_pitch")
    bad = planes_of_new("yuv422p10le", B, oh, ow)
    bad[0].y += 2
    expect([fwd(FAKE, None, _l.TU_F32, None, bad, code("yuv422p10le"))], "out_frames", "frame 0", "multiples of 4 bytes")
    bad = planes_of_new("yuv420p10le", B, H, W)
    bad[1].v = None
    expect([fwd(None, bad, code("yuv420p10le"), None, planes_of_new("nv16", B, oh, ow), code("nv16"))], "x_frames", "frame 1", "v is NULL")
    # tu_forward_planes takes TuFramePlanes: NV16 / P210 sides, never a planar one
    pl = planes_of_new("nv16", B, H, W)
    for c in (code("yuv422p"), code("yuv420p10le"), code("yuv444p10le")):
        rc = lib.tu_forward_planes(w, None, pl, c, FAKE, None, _l.TU_F32, B, H, W, oh, ow, 0, _l.TU_BF16, 1, FAKE, 1 << 40, None)
        expect([(rc, _l.last_error())], "TuFramePlanes3")
    need = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, code("nv16"), code("p210"))
    rc = lib.tu_forward_planes(w, None, pl, code("nv16"), None, planes_of_new("p210", B, oh, ow), code("p210"), B, H, W, oh, ow, 0,
                               _l.TU_BF16, 1, FAKE, need - 1, None)
    assert rc == _l.TU_ERR_WORKSPACE and ("need %d bytes" % need) in _l.last_error()
    for fmt in NEW:                                                         # never a compute dtype
        assert lib.tu_forward_workspace_bytes(0, 1, 72, 104, 108, 156, 0, code(fmt)) == 0


def _align(n):
    return (n + 1023) // 1024 * 1024


def test_workspace_sizes(lib):
    """every pre-existing code pair sizes as the parent commit did: the base, plus the planar fp16 (8-bit YUV) / fp32 (16-bit YUV) frame
    of each YUV side, plus the alpha plane of a 4-byte pair; each new side adds its planar fp16 / fp32 frame; surfaces need exactly the
    dense call's workspace"""
    from tests.golden.cases import CASES
    _l = L()
    u8 = _l.TU_U8
    # every pre-existing code (kind: 0 plain, 1 / 2 an 8-bit / 16-bit YUV frame, 3 a 4-byte frame; 4:2:0 needs even sizes)
    old = [(_l.TU_F32, 0, False), (_l.TU_BF16, 0, False), (_l.TU_F16, 0, False), (u8, 0, False), (u8 | _l.TU_LAYOUT_HWC, 0, False),
           (u8 | _l.TU_LAYOUT_HWC_BGR, 0, False), (u8 | _l.TU_LAYOUT_RGBA, 3, False), (u8 | _l.TU_LAYOUT_BGRA, 3, False),
           (u8 | _l.TU_LAYOUT_NV12, 1, True), (u8 | _l.TU_LAYOUT_NV12 | _l.TU_YUV_BT601 | _l.TU_YUV_FULL_RANGE, 1, True),
           (_l.TU_U16 | _l.TU_LAYOUT_P010, 2, True), (_l.TU_U16 | _l.TU_LAYOUT_P010 | _l.TU_YUV_BT2020, 2, True),
           (u8 | _l.TU_LAYOUT_YUV420P, 1, True), (u8 | _l.TU_LAYOUT_YUV444P | _l.TU_YUV_BT601, 1, False),
           (_l.TU_U16 | _l.TU_LAYOUT_YUV444P | _l.TU_YUV_BT2020 | _l.TU_YUV_FULL_RANGE, 2, False)]
    new = [(code(f, y), 2 if is16(f) else 1, NEW[f][0]) for f in NEW for y in ("bt709", "bt601_full")] + \
          [(code(f, "bt2020"), 2, NEW[f][0]) for f in NEW if is16(f)]
    packs = {}
    for name, c in CASES.items():
        H, W, oh, ow, s = _geometry(c)
        B = c["shape"][0]
        fin, fout = B * 3 * H * W, B * 3 * oh * ow
        for cdt, tdt in ((_l.TU_BF16, torch.bfloat16), (_l.TU_F32, torch.float32)):
            key = (c["model"], cdt)
            if key not in packs:
                packs[key] = _packed(c["model"], tdt)
            w = C.byref(packs[key].struct)
            base = lib.tu_forward_workspace_bytes_for(w, B, H, W, oh, ow, s, cdt)
            assert base > 0, name

            def q(i, o):
                return lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, i, o)

            def extra(kind, n):
                return _align(n * (2 if kind == 1 else 4)) if kind in (1, 2) else 0

            def valid(sub, h, w_):
                return sub is True and h % 2 == 0 and w_ % 2 == 0 or sub == "420" and h % 2 == 0 and w_ % 2 == 0 or \
                    sub == "422" and w_ % 2 == 0 or sub in (False, "444")
            for i, ki, si in old:
                for o, ko, so in old:
                    want = base + extra(ki, fin) + extra(ko, fout) + (_align(B * oh * ow) if ki == ko == 3 else 0)
                    want = want if valid(si, H, W) and valid(so, oh, ow) else 0
                    assert q(i, o) == want, (name, hex(i), hex(o))
            for c_, k, sub in new:
                ok_in, ok_out = valid(sub, H, W), valid(sub, oh, ow)
                assert q(c_, _l.TU_F32) == (base + extra(k, fin) if ok_in else 0), (name, hex(c_))
                assert q(_l.TU_F32, c_) == (base + extra(k, fout) if ok_out else 0), (name, hex(c_))
                assert q(c_, u8 | _l.TU_LAYOUT_BGRA) == q(c_, _l.TU_F32), name
                assert q(c_, c_) == (base + extra(k, fin) + extra(k, fout) if ok_in and ok_out else 0), (name, hex(c_))
    # surfaces: one byte less than the dense query is TU_ERR_WORKSPACE from the sizing pass, before any launch
    pw = _packed("WindowTransformer", torch.bfloat16)
    w = C.byref(pw.struct)
    B, H, W, oh, ow = 2, 72, 104, 108, 156
    for fi, fo in (("yuv422p", "p210"), ("nv16", "yuv420p10le"), ("yuv444p10le", "yuv422p10le"), ("p210", "nv16")):
        need = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, code(fi), code(fo))
        rc = lib.tu_forward_frames(w, None, planes_of_new(fi, B, H, W), code(fi), None, planes_of_new(fo, B, oh, ow), code(fo), B, H, W,
                                   oh, ow, 0, _l.TU_BF16, 1, FAKE, need - 1, None)
        assert rc == _l.TU_ERR_WORKSPACE and ("need %d bytes" % need) in _l.last_error(), (fi, fo)


def test_yuvp_ops_still_take_the_old_planar_codes_with_the_old_checks(lib):
    """the planar op's dense / RGB alignment rules of yuv420p, yuv444p, yuv444p16 are unchanged"""
    _l = L()
    for fmt, c, ra, fa in (("yuv420p", _l.TU_U8 | _l.TU_LAYOUT_YUV420P, 4, 2), ("yuv444p", _l.TU_U8 | _l.TU_LAYOUT_YUV444P, 2, 1),
                           ("yuv444p16", _l.TU_U16 | _l.TU_LAYOUT_YUV444P, 4, 2)):
        expect(both_ops(lib, FAKE, None, c, 1, 4, 4, rgb=FAKE + ra // 2), "%d-byte aligned" % ra)
        if fa > 1:
            expect(both_ops(lib, FAKE + 1, None, c, 1, 4, 4), "dense", "%d-byte aligned" % fa)
        fr = frames3(1, 4, 4, fmt)
        fr[0].y = None
        expect(both_ops(lib, None, fr, c, 1, 4, 4), "frame 0", "y is NULL")


# ---------------------------------------------------------------------------------------------------------------------------------
# Python
def test_plane_lists_rejections():
    from transformerupscaler_b200 import engine
    y, h = torch.zeros(5, 16, dtype=U8), torch.zeros(5, 8, dtype=U8)
    for fr in ([(y, h, h[:4])], [(y, y, y)], [(y, h.to(U16), h)], [(torch.zeros(5, 15, dtype=U8), h, h)], [(y, h, h)]):
        with pytest.raises(ValueError):
            engine.plane_triples(fr, "yuv422p", "frames")
    with pytest.raises(ValueError):
        engine.plane_triples([(y.to(U16), h.to(U16), h.to(U16))], "yuv422p10le", "frames")          # host tensors
    with pytest.raises(ValueError):
        engine.plane_triples([(y, h, h)], "yuv420p10le", "frames")                                  # 8-bit planes, odd H
    for fr in ([(y, y[:4])], [(y, h)], [(torch.zeros(5, 15, dtype=U8), torch.zeros(5, 15, dtype=U8))], [(y, y)]):
        with pytest.raises(ValueError):
            engine.plane_pairs(fr, "NV16", "frames")
    with pytest.raises(ValueError):
        engine.plane_pairs([(y, y)], "P210", "frames")                                               # uint8 planes for p210


def test_run_forward_value_errors():
    from transformerupscaler_b200 import engine
    x16 = torch.zeros(1, 16, 16, dtype=U16)
    x8 = torch.zeros(1, 16, 16, dtype=U8)

    def rf(x, out_dtype=U8, res=(12, 24), **kw):
        return engine.run_forward(0, "WindowTransformer", x, res, None, True, True, out_dtype, **kw)
    with pytest.raises(ValueError, match="BT.2020"):
        rf(x8, in_layout="nv16", yuv="bt2020")
    with pytest.raises(ValueError, match="BT.2020"):
        rf(x16, U8, in_layout="p210", out_layout="yuv422p", yuv="bt2020")
    with pytest.raises(ValueError, match="BT.2020"):
        rf(x8, U16, in_layout="yuv422p", out_layout="yuv422p10le", yuv="bt2020_full")
    with pytest.raises(ValueError, match="uint16 frames"):
        rf(x8, U8, in_layout="nv16", out_layout="p210")
    with pytest.raises(ValueError, match="uint8 frames"):
        rf(x16, U16, in_layout="p210", out_layout="nv16")
    with pytest.raises(ValueError, match=r"\(B, 2H, W\)"):
        rf(x8, U16, in_layout="yuv422p10le", out_layout="p210")
    with pytest.raises(ValueError, match=r"\(B, 3H/2, W\)"):
        rf(x8, U16, in_layout="yuv420p10le", out_layout="p210")
    with pytest.raises(ValueError, match="even width"):
        rf(x8, U8, res=(12, 25), in_layout="yuv422p", out_layout="nv16")
    with pytest.raises(ValueError, match="yuv420p10le output frames need an even"):
        rf(x16, U16, res=(13, 24), in_layout="p210", out_layout="yuv420p10le")
    y, u = torch.zeros(8, 16, dtype=U8), torch.zeros(8, 8, dtype=U8)
    with pytest.raises(ValueError, match="pair"):                       # out= of an nv16 side takes pairs
        rf(x8, in_layout="nv16", out_layout="nv16", out=[(y, u, u)])
    with pytest.raises(ValueError, match="unknown frame layout"):
        engine.layout_code("yuv422p12le")


def test_model_and_wrappers():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.models.WindowTransformer.model import TransformerModel
    m = TransformerModel().eval()
    y = torch.zeros(8, 16, dtype=U8)
    with pytest.raises(ValueError, match="in_layout"):
        m([(y, y)], in_layout="hwc", res_out=(12, 24))
    with pytest.raises((ValueError, RuntimeError)):                     # no CUDA here: the CPU check may come first
        m(torch.zeros(1, 16, 16, dtype=U8), in_layout="p210", res_out=(12, 12))
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(m)([(y, y)], in_layout="nv16")


def test_resize_plumbing(monkeypatch):
    """FastTransformer's Resize path ends in tu::rgb_to_yuvp / tu::rgb_to_yuv422sp, from fp16 (8-bit) or fp32 (16-bit) RGB"""
    from transformerupscaler_b200 import _lib as L_, engine
    calls = []

    def fake_forward(x, handle, oh, ow, scale, cbf, code_, clamp, in_layout=0):
        calls.append(("fwd", hex(code_), hex(in_layout)))
        return torch.zeros(*engine._image_shape(x.shape[0], 3, oh, ow, code_), dtype=engine._TORCH_DT[code_ & 0xFF])

    def fake_resize(x, oh, ow, clamp, out_code=-1, alpha=None):
        calls.append(("resize", hex(out_code)))
        return torch.zeros(x.shape[0], 3, oh, ow, dtype=engine._TORCH_DT[out_code & 0xFF])

    def fake_to(name):
        def f(x, code_):
            calls.append((name, x.dtype, hex(code_)))
            return torch.zeros(*engine._image_shape(x.shape[0], 3, x.shape[2], x.shape[3], code_))
        return f

    monkeypatch.setattr(engine, "tu_forward", fake_forward)
    monkeypatch.setattr(engine, "tu_resize_aa", fake_resize)
    monkeypatch.setattr(engine, "tu_rgb_to_yuvp", fake_to("to_yuvp"))
    monkeypatch.setattr(engine, "tu_rgb_to_yuv422sp", fake_to("to_422sp"))
    x = torch.zeros(2, 80, 56, dtype=U8)
    out = engine.run_forward(1, "FastTransformer", x, (60, 84), None, True, True, U8, in_layout="yuv422p", out_layout="nv16", yuv="bt601")
    assert tuple(out.shape) == (2, 120, 84)
    assert calls == [("fwd", hex(L_.TU_F32), hex(L_.TU_LAYOUT_YUV422P | L_.TU_YUV_BT601)), ("resize", hex(L_.TU_F16)),
                     ("to_422sp", torch.float16, hex(code("nv16", "bt601")))]
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", torch.zeros(2, 60, 56, dtype=U16), (60, 84), None, True, True, U16,
                             in_layout="yuv420p10le", out_layout="yuv422p10le", yuv="bt2020")
    assert tuple(out.shape) == (2, 120, 84)
    assert calls == [("fwd", hex(L_.TU_F32), hex(code("yuv420p10le", "bt2020") & ~0xFF)), ("resize", hex(L_.TU_F32)),
                     ("to_yuvp", torch.float32, hex(code("yuv422p10le", "bt2020")))]


def test_fake_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from transformerupscaler_b200 import _lib as L_, engine  # noqa: F401  (registers the tu:: ops)
    with FakeTensorMode():
        x = torch.empty(2, 12, 16, dtype=U16)
        for fmt in NEW:
            y = torch.ops.tu.forward(x, 1, 12, 18, 0, True, code(fmt), True, engine.LAYOUTS["yuv420p10le"])
            assert tuple(y.shape) == dense_shape(fmt, 2, 12, 18) and y.dtype == NEW[fmt][1], fmt
        planes = [torch.empty(6, 16, dtype=U8), torch.empty(6, 16, dtype=U8)] * 2
        y = torch.ops.tu.forward_planes(None, planes, [], 1, 12, 18, 0, True, code("p210"), True, L_.TU_LAYOUT_NV16)
        assert tuple(y.shape) == (2, 24, 18) and y.dtype == U16
        f = torch.empty(2, 3, 6, 10, dtype=torch.float16)
        assert tuple(torch.ops.tu.rgb_to_yuvp(f, code("yuv422p")).shape) == (2, 12, 10)
        r = torch.ops.tu.rgb_to_yuvp(f.float(), code("yuv420p10le"))
        assert tuple(r.shape) == (2, 9, 10) and r.dtype == U16
        r = torch.ops.tu.rgb_to_yuv422sp(f.float(), code("p210"))
        assert tuple(r.shape) == (2, 12, 10) and r.dtype == U16
        r = torch.ops.tu.rgb_to_yuv422sp(f, code("nv16"))
        assert tuple(r.shape) == (2, 12, 10) and r.dtype == U8
        assert torch.ops.tu.rgb_to_yuv422sp_planes(f, planes, code("nv16")) is None
