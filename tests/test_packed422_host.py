"""CPU: packed 4:2:2 frames (yuyv422, uyvy422, y210) -- the conversion oracle (the samples de-interleaved to the nv16 / p210 frame they
hold, then the 4:2:2 oracle of tests/test_yuv422_host.py), its agreement with a float64 evaluation of the defining equations, the C-ABI
constants, struct and symbols, every host-side rejection of the single ops, the forward and the workspace queries (all made before
anything is enqueued, so they run without a GPU), the workspace sizes of every code pair, and the Python-side errors and fake shapes.
tests/test_gpu_packed422.py compares the kernels with this oracle bit for bit."""
import ctypes as C
import os
import re
import subprocess

import pytest
import torch

from tests.test_nv12_host import _geometry, _packed
from tests.test_yuv422_host import (MATRIX, NEW, _align, _f64_to_rgb, code as code_422, from_planes, is16,
                                    oracle_from_rgb, oracle_to_rgb, planes_of_new, to_planes, upsample422)
from tests.test_yuvp_host import COLOURS8, FAKE, HEADER, expect
from tests.test_p010_host import COLOURS10

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U8, U16 = torch.uint8, torch.uint16
# FFmpeg's pix_fmt name -> (frame dtype, the semi-planar layout of the same samples, positions of Y0, U, Y1, V in a macropixel)
PACKED = {"yuyv422": (U8, "nv16", (0, 1, 2, 3)), "uyvy422": (U8, "nv16", (1, 0, 3, 2)), "y210": (U16, "p210", (0, 1, 2, 3))}


def L():
    from transformerupscaler_b200 import _lib
    return _lib


def code(fmt, yuv="bt709"):
    from transformerupscaler_b200 import engine
    return (L().TU_U16 if PACKED[fmt][0] == U16 else L().TU_U8) | engine.LAYOUTS[fmt] | engine.yuv_code(yuv)


def colours(fmt):
    return COLOURS10 if PACKED[fmt][0] == U16 else COLOURS8


def to_semi(f, fmt):
    """packed frames (B, H, W, 2) -> the nv16 / p210 frames (B, 2H, W) of the same stored samples"""
    B, H, W, _ = f.shape
    iy0, iu, iy1, iv = PACKED[fmt][2]
    m = f.reshape(B, H, W // 2, 4)
    y = torch.stack([m[..., iy0], m[..., iy1]], -1).reshape(B, H, W)
    return from_planes(y, m[..., iu], m[..., iv], PACKED[fmt][1])


def from_semi(f, fmt):
    """nv16 / p210 frames (B, 2H, W) -> packed frames (B, H, W, 2) of the same stored samples"""
    y, u, v = to_planes(f, PACKED[fmt][1])
    B, H, W = y.shape
    m = torch.empty(B, H, W // 2, 4, dtype=f.dtype, device=f.device)
    iy0, iu, iy1, iv = PACKED[fmt][2]
    m[..., iy0], m[..., iy1], m[..., iu], m[..., iv] = y[..., 0::2], y[..., 1::2], u, v
    return m.reshape(B, H, W, 2)


def oracle_packed_to_rgb(f, fmt, yuv="bt709"):
    """packed frames -> planar RGB (B, 3, H, W) fp32 in [0, 1]: the nv16 / p210 oracle on the de-interleaved samples"""
    return oracle_to_rgb(to_semi(f.cpu(), fmt), PACKED[fmt][1], yuv)


def oracle_rgb_to_packed(rgb, fmt, yuv="bt709"):
    """planar RGB (fp16 values for the 8-bit layouts, fp32 for y210) -> packed frames: the nv16 / p210 samples interleaved"""
    return from_semi(oracle_from_rgb(rgb, PACKED[fmt][1], yuv), fmt)


def random_packed(fmt, B, H, W, seed, hi=None):
    g = torch.Generator().manual_seed(seed)
    hi = hi or (65536 if PACKED[fmt][0] == U16 else 256)
    return torch.randint(0, hi, (B, H, W, 2), generator=g, dtype=torch.int32).to(PACKED[fmt][0])


def codes_of(f, fmt):
    """stored samples -> int codes (y210 words >> 6)"""
    c = f.to(torch.int32) & 0xFFFF
    return c >> 6 if fmt == "y210" else c


# ---------------------------------------------------------------------------------------------------------------------------------
# the oracle
def test_interleave_positions():
    """macropixel j of row i: Y0 U Y1 V (yuyv422, y210) or U Y0 V Y1 (uyvy422), read back through the nv16 / p210 planes"""
    for fmt in PACKED:
        B, H, W = 2, 3, 6
        f = random_packed(fmt, B, H, W, seed=1)
        y, u, v = to_planes(to_semi(f, fmt), PACKED[fmt][1])
        m = f.reshape(B, H, W // 2, 4)
        order = "yuyv" if fmt != "uyvy422" else "uyvy"
        for i in range(H):
            for j in range(W // 2):
                got = {"y0": y[0, i, 2 * j], "y1": y[0, i, 2 * j + 1], "u": u[0, i, j], "v": v[0, i, j]}
                want = dict(zip(("y0", "u", "y1", "v") if order == "yuyv" else ("u", "y0", "v", "y1"), m[0, i, j]))
                assert all(int(got[k]) == int(want[k]) for k in got), (fmt, i, j)
        assert torch.equal(from_semi(to_semi(f, fmt), fmt), f)


@pytest.mark.parametrize("fmt", list(PACKED))
def test_oracle_matches_float64_equations(fmt):
    """to RGB within one code of the float64 equations on the float64-upsampled chroma; from RGB within one code of the float64
    rounding of the equations on the float64 chroma filter, for every colour code"""
    w16 = PACKED[fmt][0] == U16
    cmax = 1023 if w16 else 255
    B, H, W = 3, 5, 18
    f = random_packed(fmt, B, H, W, seed=2, hi=65536 if w16 else 256)
    y, u, v = (codes_of(p, fmt).double() for p in to_planes(to_semi(f, fmt), PACKED[fmt][1]))
    rgb = torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(3))
    rgb = rgb if w16 else rgb.half()
    p = rgb.double()
    for yuv in colours(fmt):
        err = (oracle_packed_to_rgb(f, fmt, yuv).double() - _f64_to_rgb(y, upsample422(u), upsample422(v), yuv, w16)).abs().max().item()
        assert err * cmax <= 1 and err < 1e-6, (yuv, err)
        kr, kb = MATRIX[yuv.split("_")[0]]
        kg, full = 1.0 - kr - kb, yuv.endswith("_full")
        yo, ys, cs = (0.0, cmax, cmax) if full else ((64.0, 876.0, 896.0) if w16 else (16.0, 219.0, 224.0))
        mid = 512.0 if w16 else 128.0
        out = oracle_rgb_to_packed(rgb, fmt, yuv)
        if w16:
            assert int((out.to(torch.int32) & 0x3F).max()) == 0, yuv           # the low 6 bits of a written word are zero
        gy, gu, gv = (codes_of(t, fmt).double() for t in to_planes(to_semi(out, fmt), PACKED[fmt][1]))
        yl = kr * p[:, 0] + kg * p[:, 1] + kb * p[:, 2]
        c0 = torch.cat([p[..., :1], p[..., 1::2][..., :-1]], -1)
        bar = (c0 + 2 * p[..., 0::2] + p[..., 1::2]) / 4
        ybar = kr * bar[:, 0] + kg * bar[:, 1] + kb * bar[:, 2]
        want = [torch.floor(ys * yl + yo + 0.5).clamp(0, cmax),
                torch.floor(cs * (bar[:, 2] - ybar) / (2 * (1 - kb)) + mid + 0.5).clamp(0, cmax),
                torch.floor(cs * (bar[:, 0] - ybar) / (2 * (1 - kr)) + mid + 0.5).clamp(0, cmax)]
        for a, b in zip((gy, gu, gv), want):
            assert (a - b).abs().max().item() <= 1, yuv


@pytest.mark.parametrize("fmt", list(PACKED))
def test_exact_endpoints(fmt):
    w16 = PACKED[fmt][0] == U16
    sh = 6 if w16 else 0
    for yuv in colours(fmt):
        full = yuv.endswith("_full")
        lo, hi = (0, 1023 if w16 else 255) if full else ((64, 940) if w16 else (16, 235))
        mid = 512 if w16 else 128
        f = torch.empty(2, 3, 4, 2, dtype=torch.int32)
        m = f.view(2, 3, 2, 4)
        iy0, iu, iy1, iv = PACKED[fmt][2]
        for b, yv in enumerate((lo, hi)):
            m[b, ..., iy0] = m[b, ..., iy1] = yv << sh
            m[b, ..., iu] = m[b, ..., iv] = mid << sh
        f = f.to(PACKED[fmt][0])
        rgb = oracle_packed_to_rgb(f, fmt, yuv)
        assert torch.equal(rgb[0], torch.zeros(3, 3, 4)) and torch.equal(rgb[1], torch.ones(3, 3, 4)), yuv
        assert torch.equal(oracle_rgb_to_packed(rgb if w16 else rgb.half(), fmt, yuv), f), yuv


def test_y210_low_bits_are_ignored():
    g = torch.Generator().manual_seed(4)
    f = random_packed("y210", 2, 4, 8, seed=5)
    clean = ((f.to(torch.int32) >> 6) << 6).to(U16)
    assert not torch.equal(f, clean)
    noise = torch.randint(0, 64, f.shape, generator=g, dtype=torch.int32)
    for yuv in COLOURS10:
        assert torch.equal(oracle_packed_to_rgb(f, "y210", yuv), oracle_packed_to_rgb(clean, "y210", yuv))
        assert torch.equal(oracle_packed_to_rgb((clean.to(torch.int32) | noise).to(U16), "y210", yuv),
                           oracle_packed_to_rgb(clean, "y210", yuv))


# ---------------------------------------------------------------------------------------------------------------------------------
# the C ABI
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    return L().load()


def test_abi_constants_and_symbols(lib):
    from transformerupscaler_b200 import engine
    _l = L()
    src = open(os.path.join(ROOT, "include", "tu_b200.h")).read()
    for name, val in (("TU_LAYOUT_YUYV", 0xB00), ("TU_LAYOUT_UYVY", 0xC00)):
        assert re.search(r"#define\s+%s\s+0x%x\b" % (name, val), src, re.I), name
        assert getattr(_l, name) == val
    for name, expr in (("TU_U8_YUYV422", r"\(TU_U8 \| TU_LAYOUT_YUYV\)"), ("TU_U8_UYVY422", r"\(TU_U8 \| TU_LAYOUT_UYVY\)"),
                       ("TU_U16_Y210", r"\(TU_U16 \| TU_LAYOUT_YUYV\)")):
        assert re.search(r"#define\s+%s\s+%s" % (name, expr), src), name
    assert re.search(r"10 NV16, 11 YUYV, 12 UYVY\.", src)
    for n in ("tu_packed422_to_rgb", "tu_rgb_to_packed422"):
        assert hasattr(lib, n) and n in _l.SIGNATURES and re.search(r"\b%s\(" % n, src), n
    for n in ("yuyv422_to_rgb", "rgb_to_yuyv422", "uyvy422_to_rgb", "rgb_to_uyvy422", "y210_to_rgb", "rgb_to_y210"):
        assert '"%s"' % n in src, n
    assert engine.LAYOUTS["yuyv422"] == engine.LAYOUTS["y210"] == 0xB00 and engine.LAYOUTS["uyvy422"] == 0xC00
    for fmt in PACKED:
        assert engine._image_shape(2, 3, 6, 10, code(fmt)) == (2, 6, 10, 2), fmt
        assert fmt in engine.YUV_LAYOUTS and (fmt in engine.YUV16_LAYOUTS) == (fmt == "y210")
    # whole-value comparisons: 0xB00 / 0xC00 share bits with HWC_BGR, RGBA, NV12, P010, BGRA
    for c in (0xB00, 0xC00):
        assert not any(f(c) for f in (engine._is_nv12, engine._is_p010, engine._is_px4, engine._is_yuvp, engine._is_nv16))
    assert engine._is_packed422(0xB00) and engine._is_packed422(0xC00) and not engine._is_packed422(0xA00)


def test_frame_packed_layout_matches_c(lib, tmp_path):
    src = tmp_path / "fpk.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu\\n",sizeof(TuFramePacked),'
                   'offsetof(TuFramePacked,data),offsetof(TuFramePacked,pitch));return 0;}\n' % HEADER)
    exe = tmp_path / "fpk"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(t) for t in subprocess.check_output([str(exe)]).split()]
    P = L().TuFramePacked
    assert got == [C.sizeof(P), P.data.offset, P.pitch.offset] == [16, 0, 8]


def bad_codes():
    """every invalid combination the packed codes border on, and the nibbles that stay unused"""
    _l = L()
    U8_, U16_, YUYV, UYVY = _l.TU_U8, _l.TU_U16, _l.TU_LAYOUT_YUYV, _l.TU_LAYOUT_UYVY
    out = [U16_ | UYVY,                                                                          # no producer writes 16-bit UYVY
           _l.TU_F32 | YUYV, _l.TU_F16 | YUYV, _l.TU_BF16 | YUYV, _l.TU_F32 | UYVY, _l.TU_F16 | UYVY, _l.TU_BF16 | UYVY,   # float dtypes
           U8_ | YUYV | _l.TU_YUV_LSB10, U8_ | UYVY | _l.TU_YUV_LSB10, U16_ | YUYV | _l.TU_YUV_LSB10, U16_ | UYVY | _l.TU_YUV_LSB10,
           U8_ | YUYV | _l.TU_YUV_BT2020, U8_ | UYVY | _l.TU_YUV_BT2020,                           # BT.2020 on the 8-bit codes
           U16_ | YUYV | _l.TU_YUV_BT601 | _l.TU_YUV_BT2020]
    out += [c | 0x8000 for c in (code("yuyv422"), code("uyvy422"), code("y210"))]             # bit 15
    out += [b | (n << 8) for n in (0xD, 0xE, 0xF) for b in (U8_, U16_)]                         # unused nibbles
    return tuple(out)


def ops(lib, dense, fr, c, B, H, W, rgb=FAKE):
    return [(lib.tu_packed422_to_rgb(dense, fr, c, rgb, B, H, W, None), L().last_error()),
            (lib.tu_rgb_to_packed422(rgb, dense, fr, c, B, H, W, None), L().last_error())]


def surfaces(fmt, B, H, W, pitch_extra=256):
    """B valid descriptors (fake, aligned addresses) of a packed layout"""
    P = L().TuFramePacked
    row = 2 * W * (2 if PACKED[fmt][0] == U16 else 1)
    return (P * B)(*[P(FAKE + b * (1 << 20), row + pitch_extra) for b in range(B)])


def test_single_ops_reject_codes_and_arguments(lib):
    _l = L()
    for c in bad_codes() + tuple(code_422(f) for f in NEW) + (_l.TU_U8 | _l.TU_LAYOUT_NV12, _l.TU_U16 | _l.TU_LAYOUT_P010, _l.TU_U8):
        expect(ops(lib, FAKE, None, c, 1, 4, 4), "code must be")
        expect(ops(lib, None, surfaces("y210", 1, 4, 4), c, 1, 4, 4), "code must be")
    # the other YUV ops never take the packed codes
    for fmt in PACKED:
        c = code(fmt)
        assert lib.tu_yuv422sp_to_rgb(FAKE, None, c, FAKE, 1, 4, 4, None) == _l.TU_ERR_ARG
        assert lib.tu_rgb_to_yuvp(FAKE, FAKE, None, c, 1, 4, 4, None) == _l.TU_ERR_ARG
        assert lib.tu_nv12_to_rgb(FAKE, c, FAKE, 1, 4, 4, None) == _l.TU_ERR_ARG
    for fmt in PACKED:
        c, w16 = code(fmt), PACKED[fmt][0] == U16
        expect(ops(lib, FAKE, surfaces(fmt, 1, 4, 4), c, 1, 4, 4), "exactly one")
        expect(ops(lib, None, None, c, 1, 4, 4), "exactly one")
        for B, H, W in ((0, 4, 4), (65536, 4, 4), (1, 0, 4), (1, 4, 0)):
            expect(ops(lib, FAKE, None, c, B, H, W), "bad argument")
        expect(ops(lib, FAKE, None, c, 1, 4, 4, rgb=None), "bad argument")
        ra = 8 if w16 else 4
        expect(ops(lib, FAKE, None, c, 1, 4, 4, rgb=FAKE + ra // 2), "RGB buffer", "fp32" if w16 else "fp16", "%d-byte" % ra)
        for off in ((2, 4) if w16 else (1, 2)):
            expect(ops(lib, FAKE + off, None, c, 1, 4, 4), "dense", fmt, "%d-byte aligned" % (8 if w16 else 4))
        expect(ops(lib, FAKE, None, c, 1, 30000, 30000), "too large")
        expect(ops(lib, FAKE, None, c, 1, 4, 5), fmt, "even width")
        expect(ops(lib, None, surfaces(fmt, 1, 4, 6), c, 1, 4, 5), fmt, "even width")
        for rc, msg in ops(lib, FAKE, None, c, 1, 3, 4, rgb=None):        # any height: only the NULL RGB buffer is wrong
            assert rc == _l.TU_ERR_ARG and "bad argument" in msg


@pytest.mark.parametrize("fmt", list(PACKED))
def test_descriptor_rejections(lib, fmt):
    c, s = code(fmt), 2 if PACKED[fmt][0] == U16 else 1
    B, H, W = 3, 6, 10
    fr = surfaces(fmt, B, H, W)
    fr[1].data = None
    expect(ops(lib, None, fr, c, B, H, W), "frame 1", "data is NULL")
    fr = surfaces(fmt, B, H, W)
    fr[2].pitch = 2 * W * s - 4 * s
    expect(ops(lib, None, fr, c, B, H, W), "frame 2", "pitch", "smaller")
    for field in ("data", "pitch"):
        for off in (1, 2, 4):
            if off >= 4 * s:
                continue
            fr = surfaces(fmt, B, H, W)
            setattr(fr[0], field, getattr(fr[0], field) + off)
            expect(ops(lib, None, fr, c, B, H, W), "frame 0", field, "multiple of %d bytes" % (4 * s))
    fr = surfaces(fmt, B, H, W, pitch_extra=0)                               # pitch == 2W samples is valid
    assert all("bad argument" in m for _, m in ops(lib, None, fr, c, B, H, W, rgb=None))


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
    for fmt in PACKED:
        c = code(fmt)
        expect([fwd(FAKE, None, c, FAKE, None, _l.TU_F32, Wn=W + 1)], "4:2:2 input", "even width")
        expect([fwd(FAKE, None, _l.TU_F32, FAKE, None, c, own=ow + 1)], "4:2:2 output", "even width")
        assert lib.tu_forward_workspace_bytes_io(w, B, H, W + 1, oh, ow, 0, _l.TU_BF16, c, _l.TU_F32) == 0
        assert lib.tu_forward_workspace_bytes_io(w, B, H + 1, W, oh + 1, ow, 0, _l.TU_BF16, c, c) > 0          # any height
        assert lib.tu_forward_workspace_bytes(0, 1, 72, 104, 108, 156, 0, c) == 0                            # never a compute dtype
        al = 8 if fmt == "y210" else 4
        expect([fwd(FAKE + al // 2, None, c, FAKE, None, _l.TU_F32)], "dense packed 4:2:2 input", "%d-byte aligned" % al)
        expect([fwd(FAKE, None, _l.TU_F32, FAKE + al // 2, None, c)], "dense packed 4:2:2 output", "%d-byte aligned" % al)
    # descriptors are read as TuFramePacked, and a bad one names the side, the frame and the field
    bad = surfaces("yuyv422", B, H, W)
    bad[1].pitch = 2 * W - 2
    expect([fwd(None, bad, code("yuyv422"), FAKE, None, _l.TU_F32)], "x_frames", "frame 1", "pitch")
    bad = surfaces("y210", B, oh, ow)
    bad[0].data += 4
    expect([fwd(FAKE, None, _l.TU_F32, None, bad, code("y210"))], "out_frames", "frame 0", "data", "multiple of 8 bytes")
    bad = surfaces("uyvy422", B, oh, ow)
    bad[1].data = None
    expect([fwd(None, planes_of_new("nv16", B, H, W), code_422("nv16"), None, bad, code("uyvy422"))], "out_frames", "frame 1",
           "data is NULL")
    # tu_forward_planes takes TuFramePlanes, which cannot describe a packed frame; dense packed sides pass through it
    pl = planes_of_new("nv16", B, H, W)
    for fmt in PACKED:
        rc = lib.tu_forward_planes(w, None, pl, code(fmt), FAKE, None, _l.TU_F32, B, H, W, oh, ow, 0, _l.TU_BF16, 1, FAKE, 1 << 40, None)
        expect([(rc, _l.last_error())], "x_frames", "TuFramePacked")
        rc = lib.tu_forward_planes(w, FAKE, None, _l.TU_F32, None, planes_of_new("nv16", B, oh, ow), code(fmt), B, H, W, oh, ow, 0,
                                   _l.TU_BF16, 1, FAKE, 1 << 40, None)
        expect([(rc, _l.last_error())], "out_frames", "TuFramePacked")
        need = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, code(fmt), code(fmt))
        rc = lib.tu_forward_planes(w, FAKE, None, code(fmt), FAKE, None, code(fmt), B, H, W, oh, ow, 0, _l.TU_BF16, 1, FAKE, need - 1, None)
        assert rc == _l.TU_ERR_WORKSPACE and ("need %d bytes" % need) in _l.last_error(), fmt


def test_workspace_sizes(lib):
    """every pre-existing code pair sizes as the parent commit did; each packed side adds exactly its planar fp16 (8-bit) / fp32 (y210)
    frame; surfaces need exactly the dense call's workspace"""
    from tests.golden.cases import CASES
    _l = L()
    u8 = _l.TU_U8
    # every pre-existing code (kind: 0 plain, 1 / 2 an 8-bit / 16-bit YUV frame, 3 a 4-byte frame; sub: the size rule)
    old = [(_l.TU_F32, 0, None), (_l.TU_BF16, 0, None), (_l.TU_F16, 0, None), (u8, 0, None), (u8 | _l.TU_LAYOUT_HWC, 0, None),
           (u8 | _l.TU_LAYOUT_HWC_BGR, 0, None), (u8 | _l.TU_LAYOUT_RGBA, 3, None), (u8 | _l.TU_LAYOUT_BGRA, 3, None),
           (u8 | _l.TU_LAYOUT_NV12 | _l.TU_YUV_BT601, 1, "420"), (_l.TU_U16 | _l.TU_LAYOUT_P010 | _l.TU_YUV_BT2020, 2, "420"),
           (u8 | _l.TU_LAYOUT_YUV420P, 1, "420"), (u8 | _l.TU_LAYOUT_YUV444P, 1, None),
           (_l.TU_U16 | _l.TU_LAYOUT_YUV444P | _l.TU_YUV_FULL_RANGE, 2, None)] + \
          [(code_422(f), 2 if is16(f) else 1, NEW[f][0] if NEW[f][0] != "444" else None) for f in NEW]
    new = [(code(f, y), 2 if PACKED[f][0] == U16 else 1, "422") for f in PACKED for y in ("bt709", "bt601_full")] + \
          [(code("y210", "bt2020"), 2, "422")]

    def valid(sub, h, w_):
        return sub is None or sub == "420" and h % 2 == 0 and w_ % 2 == 0 or sub == "422" and w_ % 2 == 0

    def extra(kind, n):
        return _align(n * (2 if kind == 1 else 4)) if kind in (1, 2) else 0

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
            for i, ki, si in old:
                for o, ko, so in old:
                    want = base + extra(ki, fin) + extra(ko, fout) + (_align(B * oh * ow) if ki == ko == 3 else 0)
                    assert q(i, o) == (want if valid(si, H, W) and valid(so, oh, ow) else 0), (name, hex(i), hex(o))
            for c_, k, sub in new:
                ok_in, ok_out = valid(sub, H, W), valid(sub, oh, ow)
                assert q(c_, _l.TU_F32) == (base + extra(k, fin) if ok_in else 0), (name, hex(c_))
                assert q(_l.TU_F32, c_) == (base + extra(k, fout) if ok_out else 0), (name, hex(c_))
                assert q(c_, c_) == (base + extra(k, fin) + extra(k, fout) if ok_in and ok_out else 0), (name, hex(c_))
                for o, ko, so in old:
                    assert q(c_, o) == (base + extra(k, fin) + extra(ko, fout) if ok_in and valid(so, oh, ow) else 0), (name, hex(c_), hex(o))
                    assert q(o, c_) == (base + extra(ko, fin) + extra(k, fout) if ok_out and valid(so, H, W) else 0), (name, hex(o), hex(c_))
    # surfaces: one byte less than the dense query is TU_ERR_WORKSPACE from the sizing pass, before any launch
    pw = _packed("WindowTransformer", torch.bfloat16)
    w = C.byref(pw.struct)
    B, H, W, oh, ow = 2, 72, 104, 108, 156
    for fi, fo in (("yuyv422", "uyvy422"), ("y210", "y210"), ("uyvy422", "yuyv422")):
        need = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, code(fi), code(fo))
        rc = lib.tu_forward_frames(w, None, surfaces(fi, B, H, W), code(fi), None, surfaces(fo, B, oh, ow), code(fo), B, H, W, oh, ow, 0,
                                   _l.TU_BF16, 1, FAKE, need - 1, None)
        assert rc == _l.TU_ERR_WORKSPACE and ("need %d bytes" % need) in _l.last_error(), (fi, fo)


# ---------------------------------------------------------------------------------------------------------------------------------
# Python
def test_surface_list_rejections():
    from transformerupscaler_b200 import engine
    s8 = torch.zeros(5, 16, 2, dtype=U8)
    pool = torch.zeros(5, 40, 2, dtype=U8)
    for fr, msg in (([], "non-empty"), ([s8.to(U16)], "uint8 tensors"), ([torch.zeros(5, 16, 3, dtype=U8)], r"\(H, W, 2\)"),
                    ([(s8, s8)], "tensors"), ([torch.zeros(5, 2, 16, dtype=U8).transpose(1, 2)], "strides"),
                    ([pool[:, ::2][:, :16]], "strides"), ([s8], "CUDA")):                     # the last: a host tensor
        with pytest.raises(ValueError, match=msg):
            engine.packed_surfaces(fr, "yuyv422", "frames")
    with pytest.raises(ValueError):
        engine.packed_surfaces([s8], "y210", "frames")                              # uint8 surfaces for y210
    for x in (torch.zeros(1, 4, 6, 3, dtype=U8), torch.zeros(1, 4, 5, 2, dtype=U8), torch.zeros(1, 4, 6, 2, dtype=U16),
              torch.zeros(4, 6, 2, dtype=U8)):
        with pytest.raises(ValueError):
            engine._yuvp_hw(x, "uyvy422")
    assert engine._yuvp_hw(torch.zeros(1, 3, 6, 2, dtype=U16), "y210") == (3, 6)


def test_descriptors_of_surfaces():
    """a surface's pitch is its row stride in bytes; a one-row surface has 2W samples"""
    from transformerupscaler_b200 import engine
    pool = torch.zeros(2, 4, 40, 2, dtype=U16)
    fr = [pool[1, :, 4:16], pool[0, :1, :12]]
    d = engine._descriptors(engine._flat(fr), code("y210"))
    assert len(d) == 2 and d[0].data == fr[0].data_ptr() and d[0].pitch == 40 * 2 * 2 and d[1].pitch == 12 * 2 * 2
    assert engine._flat(fr) == fr and engine._planes_per_frame(code("uyvy422")) == 1


def test_run_forward_value_errors():
    from transformerupscaler_b200 import engine
    x8 = torch.zeros(1, 16, 16, 2, dtype=U8)
    x16 = torch.zeros(1, 16, 16, 2, dtype=U16)

    def rf(x, out_dtype=U8, res=(12, 24), **kw):
        return engine.run_forward(0, "WindowTransformer", x, res, None, True, True, out_dtype, **kw)
    with pytest.raises(ValueError, match="BT.2020"):
        rf(x8, in_layout="yuyv422", yuv="bt2020")
    with pytest.raises(ValueError, match="BT.2020"):
        rf(x16, U8, in_layout="y210", out_layout="uyvy422", yuv="bt2020")
    with pytest.raises(ValueError, match="BT.2020"):
        rf(x8, U16, in_layout="nv12", out_layout="y210", yuv="bt2020_full")
    with pytest.raises(ValueError, match="uint16 frames"):
        rf(x8, U8, in_layout="yuyv422", out_layout="y210")
    with pytest.raises(ValueError, match="uint8 frames"):
        rf(x16, U16, in_layout="y210", out_layout="uyvy422")
    with pytest.raises(ValueError, match=r"\(B, H, W, 2\)"):
        rf(x8, U16, in_layout="y210", out_layout="p010")
    with pytest.raises(ValueError, match=r"\(B, H, W, 2\)"):
        rf(torch.zeros(1, 16, 16, dtype=U8), U8, in_layout="uyvy422")
    with pytest.raises(ValueError, match="even width"):
        rf(x8, U8, res=(12, 25), in_layout="yuyv422", out_layout="uyvy422")
    with pytest.raises(ValueError, match="even width"):
        rf(torch.zeros(1, 16, 15, 2, dtype=U8), U8, in_layout="yuyv422")
    with pytest.raises(ValueError, match="surface"):                    # out= of a packed side takes one surface per frame
        rf(x8, in_layout="yuyv422", out_layout="yuyv422", out=[])
    for name in ("argb", "yuv422p12le", "yuyv", "y210le", "v210"):
        with pytest.raises(ValueError, match="unknown frame layout"):
            engine.layout_code(name)


def test_model_and_wrappers():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.models.WindowTransformer.model import TransformerModel
    m = TransformerModel().eval()
    s = torch.zeros(8, 16, 2, dtype=U8)
    with pytest.raises(ValueError, match="in_layout"):
        m([s], in_layout="hwc", res_out=(12, 24))
    with pytest.raises((ValueError, RuntimeError)):                     # no CUDA here: the CPU check may come first
        m(torch.zeros(1, 16, 16, 2, dtype=U8), in_layout="y210", res_out=(12, 12))
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(m)([s], in_layout="yuyv422")


def test_resize_plumbing(monkeypatch):
    """FastTransformer's Resize path ends in tu::rgb_to_packed422, from fp16 (8-bit) or fp32 (y210) RGB"""
    from transformerupscaler_b200 import engine
    _l = L()
    calls = []

    def fake_forward(x, handle, oh, ow, scale, cbf, code_, clamp, in_layout=0):
        calls.append(("fwd", hex(code_), hex(in_layout)))
        return torch.zeros(*engine._image_shape(x.shape[0], 3, oh, ow, code_), dtype=engine._TORCH_DT[code_ & 0xFF])

    def fake_resize(x, oh, ow, clamp, out_code=-1, alpha=None):
        calls.append(("resize", hex(out_code)))
        return torch.zeros(x.shape[0], 3, oh, ow, dtype=engine._TORCH_DT[out_code & 0xFF])

    def fake_to(x, code_):
        calls.append(("to_packed", x.dtype, hex(code_)))
        return torch.zeros(*engine._image_shape(x.shape[0], 3, x.shape[2], x.shape[3], code_))

    monkeypatch.setattr(engine, "tu_forward", fake_forward)
    monkeypatch.setattr(engine, "tu_resize_aa", fake_resize)
    monkeypatch.setattr(engine, "tu_rgb_to_packed422", fake_to)
    out = engine.run_forward(1, "FastTransformer", torch.zeros(2, 40, 56, 2, dtype=U8), (60, 84), None, True, True, U8,
                             in_layout="yuyv422", out_layout="uyvy422", yuv="bt601")
    assert tuple(out.shape) == (2, 60, 84, 2)
    assert calls == [("fwd", hex(_l.TU_F32), hex(_l.TU_LAYOUT_YUYV | _l.TU_YUV_BT601)), ("resize", hex(_l.TU_F16)),
                     ("to_packed", torch.float16, hex(code("uyvy422", "bt601")))]
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", torch.zeros(2, 40, 56, 2, dtype=U16), (60, 84), None, True, True, U16,
                             in_layout="y210", out_layout="y210", yuv="bt2020")
    assert tuple(out.shape) == (2, 60, 84, 2)
    assert calls == [("fwd", hex(_l.TU_F32), hex(code("y210", "bt2020") & ~0xFF)), ("resize", hex(_l.TU_F32)),
                     ("to_packed", torch.float32, hex(code("y210", "bt2020")))]


def test_fake_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from transformerupscaler_b200 import engine
    with FakeTensorMode():
        x = torch.empty(2, 12, 16, 2, dtype=U8)
        for fmt in PACKED:
            y = torch.ops.tu.forward(x, 1, 12, 18, 0, True, code(fmt), True, engine.LAYOUTS["yuyv422"])
            assert tuple(y.shape) == (2, 12, 18, 2) and y.dtype == PACKED[fmt][0], fmt
        surf = [torch.empty(12, 16, 2, dtype=U16)] * 3
        y = torch.ops.tu.forward_planes(None, surf, [], 1, 12, 18, 0, True, code("uyvy422"), True, L().TU_LAYOUT_YUYV)
        assert tuple(y.shape) == (3, 12, 18, 2) and y.dtype == U8
        f = torch.empty(2, 3, 6, 10, dtype=torch.float16)
        r = torch.ops.tu.rgb_to_packed422(f, code("yuyv422"))
        assert tuple(r.shape) == (2, 6, 10, 2) and r.dtype == U8
        r = torch.ops.tu.rgb_to_packed422(f.float(), code("y210"))
        assert tuple(r.shape) == (2, 6, 10, 2) and r.dtype == U16
        assert torch.ops.tu.rgb_to_packed422_planes(f, [torch.empty(6, 10, 2, dtype=U8)] * 2, code("uyvy422")) is None
