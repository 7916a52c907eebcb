"""CPU: planar YUV frames (yuv420p, yuv444p, yuv444p16) -- the conversion oracle, its agreement with a float64 evaluation of the
defining equations and with the NV12 oracle, the C-ABI constants, symbols and TuFramePlanes3 layout, every host-side rejection of the
single ops, the forward and the workspace queries (all made before anything is enqueued, so they run without a GPU), the workspace
sizes, and the Python-side errors and fake shapes.

The oracle functions below are the definition the kernels of csrc/resample.cu follow operation for operation: plain fp32 torch ops on
the CPU, each one correctly rounded, no fused multiply-add.  tests/test_gpu_yuvp.py compares the kernels with them bit for bit."""
import ctypes as C
import os
import re
import subprocess

import pytest
import torch

from tests.test_abi import HEADER
from tests.test_nv12_host import _div, _geometry, _packed, _upsample, coefficients, oracle_nv12_to_rgb, oracle_rgb_to_nv12
from tests.test_p010_host import COLOURS10, MATRIX, coefficients10, f64_ycc_to_rgb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLOURS8 = ("bt709", "bt601", "bt709_full", "bt601_full")
FAKE = 1 << 20                       # never dereferenced: every call below fails its checks before any launch


# ---------------------------------------------------------------------------------------------------------------------------------
# the oracle
def split420(f):
    """yuv420p frames (B, 3H/2, W) -> the Y (B, H, W), U and V (B, H/2, W/2) planes"""
    B, R, W = f.shape
    H = R * 2 // 3
    flat = f.reshape(B, -1)
    n, q = H * W, H * W // 4
    return (flat[:, :n].reshape(B, H, W), flat[:, n:n + q].reshape(B, H // 2, W // 2),
            flat[:, n + q:].reshape(B, H // 2, W // 2))


def join420(y, u, v):
    B, H, W = y.shape
    return torch.cat([y.reshape(B, -1), u.reshape(B, -1), v.reshape(B, -1)], 1).reshape(B, 3 * H // 2, W)


def yuv420p_to_nv12(f):
    y, u, v = split420(f)
    B, H, W = y.shape
    return torch.cat([y, torch.stack([u, v], -1).reshape(B, H // 2, W)], 1)


def nv12_to_yuv420p(f):
    B, R, W = f.shape
    H = R * 2 // 3
    ch = f[:, H:].reshape(B, H // 2, W // 2, 2)
    return join420(f[:, :H], ch[..., 0], ch[..., 1])


def _coef(yuv, w16):
    return coefficients10(yuv) if w16 else coefficients(yuv)


def _to_rgb(Y, U, V, k, mid):
    """codes (fp32) -> planar RGB (B, 3, H, W) fp32 clamped to [0, 1]: the formulas of include/tu_b200.h"""
    yn = _div(Y - k["yo"], k["ys"])
    un = _div(U - mid, k["cs"])
    vn = _div(V - mid, k["cs"])
    r = yn + k["a_rv"] * vn
    g = (yn + k["a_gu"] * un) + k["a_gv"] * vn
    b = yn + k["a_bu"] * un
    return torch.stack([r, g, b], 1).clamp(0, 1)


def oracle_yuv420p_to_rgb(f, yuv="bt709"):
    """yuv420p (B, 3H/2, W) uint8 -> planar RGB fp32 (the kernel stores it rounded to fp16): NV12's chroma upsampling on the U and V
    planes"""
    y, u, v = (t.float() for t in split420(f.cpu()))
    H, W = y.shape[1:]
    return _to_rgb(y, _upsample(u, H, W), _upsample(v, H, W), coefficients(yuv), 128.0)


def oracle_rgb_to_yuv420p(rgb, yuv="bt709"):
    return nv12_to_yuv420p(oracle_rgb_to_nv12(rgb, yuv))


def oracle_yuv444_to_rgb(f, yuv="bt709"):
    """yuv444p (uint8) / yuv444p16 (uint16, code = word >> 6) frames (B, 3, H, W) -> planar RGB fp32 (fp16-rounded by the 8-bit kernel)"""
    w16 = f.dtype == torch.uint16
    c = (f.cpu().to(torch.int32) >> (6 if w16 else 0)).float()
    return _to_rgb(c[:, 0], c[:, 1], c[:, 2], _coef(yuv, w16), 512.0 if w16 else 128.0)


def oracle_rgb_to_yuv444(rgb, yuv="bt709", w16=False):
    """planar RGB (B, 3, H, W) -> yuv444p (uint8) or yuv444p16 (uint16 words, code << 6): each pixel from its own R, G, B"""
    p = rgb.cpu().float()
    k = _coef(yuv, w16)
    mid, cmax = (512.0, 1023) if w16 else (128.0, 255)
    R, G, B_ = p[:, 0], p[:, 1], p[:, 2]
    yl = (k["kr"] * R + k["kg"] * G) + k["kb"] * B_
    cb = (k["cb_r"] * R + k["cb_g"] * G) + 0.5 * B_
    cr = (0.5 * R + k["cr_g"] * G) + k["cr_b"] * B_

    def code(v):
        return torch.floor(v + 0.5).clamp(0, cmax).to(torch.int32)
    c = torch.stack([code(k["ys"] * yl + k["yo"]), code(k["cs"] * cb + mid), code(k["cs"] * cr + mid)], 1)
    return (c << 6).to(torch.uint16) if w16 else c.to(torch.uint8)


def _params(yuv, w16):
    kr, kb = MATRIX[yuv.split("_")[0]]
    full = yuv.endswith("_full")
    if w16:
        return kr, kb, (0.0 if full else 64.0), (1023.0 if full else 876.0), (1023.0 if full else 896.0), 512.0, 1023
    return kr, kb, (0.0 if full else 16.0), (255.0 if full else 219.0), (255.0 if full else 224.0), 128.0, 255


def _colours(w16):
    return COLOURS10 if w16 else COLOURS8


@pytest.mark.parametrize("w16", [False, True])
def test_444_oracle_to_rgb_matches_float64_equations(w16):
    """every Y code against a lattice of (U, V) codes (special codes included), every colour: within one code of the float64
    equations (in fact far closer)"""
    cmax = 1023 if w16 else 255
    special = (0, 16, 64, 128, 235, 240, 255) if not w16 else (0, 64, 512, 940, 960, 1023)
    us = sorted(set(range(0, cmax + 1, 33 if w16 else 9)) | set(special))
    vs = sorted(set(range(0, cmax + 1, 31 if w16 else 7)) | set(special))
    pairs = torch.tensor([(u, v) for u in us for v in vs], dtype=torch.int32)
    n = pairs.shape[0]
    Y = torch.arange(cmax + 1, dtype=torch.int32)[None].expand(n, cmax + 1)
    f = torch.stack([Y, pairs[:, :1].expand_as(Y), pairs[:, 1:].expand_as(Y)], 1)[:, :, None, :]     # (n, 3, 1, cmax + 1)
    f = (f << 6).to(torch.uint16) if w16 else f.to(torch.uint8)
    for yuv in _colours(w16):
        got = oracle_yuv444_to_rgb(f, yuv)[:, :, 0].double()
        kr, kb, yo, ys, cs, mid, _ = _params(yuv, w16)
        Yd, Ud, Vd = Y.double(), pairs[:, :1].double().expand(n, cmax + 1), pairs[:, 1:].double().expand(n, cmax + 1)
        if w16:
            want = f64_ycc_to_rgb(Yd, Ud, Vd, yuv)
        else:
            kg = 1.0 - kr - kb
            y, u, v = (Yd - yo) / ys, (Ud - mid) / cs, (Vd - mid) / cs
            want = torch.stack([y + 2 * (1 - kr) * v, y - 2 * (1 - kb) * kb / kg * u - 2 * (1 - kr) * kr / kg * v,
                                y + 2 * (1 - kb) * u], 1).clamp(0, 1)
        err = (got - want).abs().max().item()
        assert err * cmax <= 1 and err < 1e-6, (yuv, err)


@pytest.mark.parametrize("w16", [False, True])
def test_444_oracle_from_rgb_matches_float64_equations(w16):
    """random colours: every code within one of the float64 rounding of the equations"""
    g = torch.Generator().manual_seed(7)
    n = 8192
    col = torch.rand(n, 3, generator=g, dtype=torch.float64)
    img = col.float()[:, :, None, None]
    if not w16:
        img = img.half().float()                     # the 8-bit side reads fp16 RGB
    for yuv in _colours(w16):
        kr, kb, yo, ys, cs, mid, cmax = _params(yuv, w16)
        kg = 1.0 - kr - kb
        got = oracle_rgb_to_yuv444(img, yuv, w16).to(torch.int32)[:, :, 0, 0] >> (6 if w16 else 0)
        c = img[:, :, 0, 0].double()
        yl = kr * c[:, 0] + kg * c[:, 1] + kb * c[:, 2]
        want = torch.stack([torch.floor(ys * yl + yo + 0.5), torch.floor(cs * (c[:, 2] - yl) / (2 * (1 - kb)) + mid + 0.5),
                            torch.floor(cs * (c[:, 0] - yl) / (2 * (1 - kr)) + mid + 0.5)], 1).clamp(0, cmax)
        assert (got.double() - want).abs().max().item() <= 1, yuv


@pytest.mark.parametrize("w16", [False, True])
def test_444_exact_endpoints(w16):
    for yuv in _colours(w16):
        full = yuv.endswith("_full")
        lo, hi = (0, 1023 if w16 else 255) if full else ((64, 940) if w16 else (16, 235))
        mid = 512 if w16 else 128
        f = torch.full((2, 3, 2, 3), mid, dtype=torch.int32)
        f[0, 0], f[1, 0] = lo, hi
        f = (f << 6).to(torch.uint16) if w16 else f.to(torch.uint8)
        rgb = oracle_yuv444_to_rgb(f, yuv)
        assert torch.equal(rgb[0], torch.zeros(3, 2, 3)) and torch.equal(rgb[1], torch.ones(3, 2, 3)), yuv
        assert torch.equal(oracle_rgb_to_yuv444(rgb, yuv, w16), f), yuv


def test_yuv420p_oracle_is_the_nv12_oracle_interleaved():
    g = torch.Generator().manual_seed(3)
    for B, H, W in ((3, 12, 18), (2, 2, 2), (1, 6, 10)):             # W/2 odd in the last two
        f = torch.randint(0, 256, (B, 3 * H // 2, W), generator=g, dtype=torch.uint8)
        assert torch.equal(nv12_to_yuv420p(yuv420p_to_nv12(f)), f)
        rgb = torch.rand(B, 3, H, W, generator=g).half()
        for yuv in COLOURS8:
            assert torch.equal(oracle_yuv420p_to_rgb(f, yuv), oracle_nv12_to_rgb(yuv420p_to_nv12(f), yuv))
            assert torch.equal(yuv420p_to_nv12(oracle_rgb_to_yuv420p(rgb, yuv)), oracle_rgb_to_nv12(rgb, yuv))


def test_444_constant_chroma_matches_420():
    """a frame of constant chroma converts to the same RGB as 4:4:4 and as NV12 / P010 (the chroma filter of a flat plane is exact),
    and the luma codes of an RGB frame are the same either way"""
    from tests.test_p010_host import oracle_p010_to_rgb, oracle_rgb_to_p010
    g = torch.Generator().manual_seed(11)
    H, W = 8, 12
    for w16 in (False, True):
        cmax = 1023 if w16 else 255
        y = torch.randint(0, cmax + 1, (2, H, W), generator=g, dtype=torch.int32)
        u, v = torch.tensor([[37], [901 if w16 else 201]]), torch.tensor([[650 if w16 else 90], [12]])
        f444 = torch.stack([y, u[:, :, None].expand(2, H, W), v[:, :, None].expand(2, H, W)], 1)
        uv = torch.stack([u[:, :, None].expand(2, H // 2, W // 2), v[:, :, None].expand(2, H // 2, W // 2)], -1).reshape(2, H // 2, W)
        f420 = torch.cat([y, uv], 1)
        if w16:
            f444, f420 = (f444 << 6).to(torch.uint16), (f420 << 6).to(torch.uint16)
        else:
            f444, f420 = f444.to(torch.uint8), f420.to(torch.uint8)
        for yuv in _colours(w16):
            want = oracle_p010_to_rgb(f420, yuv) if w16 else oracle_nv12_to_rgb(f420, yuv)
            assert torch.equal(oracle_yuv444_to_rgb(f444, yuv), want), yuv
            rgb = torch.rand(2, 3, H, W, generator=g)
            rgb = rgb if w16 else rgb.half()
            luma420 = (oracle_rgb_to_p010(rgb, yuv) if w16 else oracle_rgb_to_nv12(rgb, yuv))[:, :H]
            assert torch.equal(oracle_rgb_to_yuv444(rgb, yuv, w16)[:, 0], luma420), yuv


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
    for name, val in (("TU_LAYOUT_YUV420P", 0x600), ("TU_LAYOUT_YUV444P", 0x700)):
        assert re.search(r"#define\s+%s\s+0x%x\b" % (name, val), src, re.I), name
        assert getattr(_lib, name) == val
    assert re.search(r"#define\s+TU_U8_YUV420P\s+\(TU_U8 \| TU_LAYOUT_YUV420P\)", src)
    assert re.search(r"#define\s+TU_U8_YUV444P\s+\(TU_U8 \| TU_LAYOUT_YUV444P\)", src)
    assert re.search(r"#define\s+TU_U16_YUV444P16\s+\(TU_U16 \| TU_LAYOUT_YUV444P\)", src)
    for n in ("tu_forward_frames", "tu_yuvp_to_rgb", "tu_rgb_to_yuvp"):
        assert hasattr(lib, n) and n in _lib.SIGNATURES and re.search(r"\b%s\(" % n, src), n
    assert engine.LAYOUTS["yuv420p"] == 0x600 and engine.LAYOUTS["yuv444p"] == engine.LAYOUTS["yuv444p16"] == 0x700
    assert engine._image_shape(2, 3, 8, 10, _lib.TU_U8 | 0x600) == (2, 12, 10)
    assert engine._image_shape(2, 3, 7, 9, _lib.TU_U8 | 0x700) == engine._image_shape(2, 3, 7, 9, _lib.TU_U16 | 0x700) == (2, 3, 7, 9)
    assert not engine._is_nv12(0x600) and not engine._is_px4(0x700) and not engine._is_p010(0x700)


def test_frame_planes3_layout_matches_c(lib, tmp_path):
    src = tmp_path / "fp3.c"
    fields = ("y", "u", "v", "y_pitch", "u_pitch", "v_pitch")
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu%s\\n",sizeof(TuFramePlanes3)%s);'
                   'return 0;}\n' % (HEADER, " %zu" * len(fields), "".join(",offsetof(TuFramePlanes3,%s)" % f for f in fields)))
    exe = tmp_path / "fp3"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(t) for t in subprocess.check_output([str(exe)]).split()]
    P = L().TuFramePlanes3
    assert got == [C.sizeof(P)] + [getattr(P, f).offset for f in fields] == [48, 0, 8, 16, 24, 32, 40]


def codes():
    _l = L()
    return {"yuv420p": _l.TU_U8 | _l.TU_LAYOUT_YUV420P, "yuv444p": _l.TU_U8 | _l.TU_LAYOUT_YUV444P,
            "yuv444p16": _l.TU_U16 | _l.TU_LAYOUT_YUV444P}


def bad_codes():
    _l = L()
    p420, p444, p16 = codes().values()
    return (_l.TU_U16 | _l.TU_LAYOUT_YUV420P, _l.TU_F32 | _l.TU_LAYOUT_YUV444P, _l.TU_F16 | _l.TU_LAYOUT_YUV420P,
            _l.TU_BF16 | _l.TU_LAYOUT_YUV444P, p420 | _l.TU_YUV_BT2020, p444 | _l.TU_YUV_BT2020, p16 | _l.TU_YUV_BT601 | _l.TU_YUV_BT2020,
            p420 | 0x8000, p16 | 0x8000, _l.TU_U16 | _l.TU_LAYOUT_YUV420P | _l.TU_YUV_BT2020)


def frames3(B, H, W, fmt, pitch_extra=256):
    """B valid descriptors (fake, aligned addresses)"""
    s = 2 if fmt == "yuv444p16" else 1
    cw = W // 2 if fmt == "yuv420p" else W
    P = L().TuFramePlanes3
    return (P * B)(*[P(FAKE + b * (1 << 20), FAKE + b * (1 << 20) + (1 << 18), FAKE + b * (1 << 20) + (1 << 19),
                       W * s + pitch_extra, cw * s + pitch_extra, cw * s + pitch_extra) for b in range(B)])


def both_ops(lib, dense, fr, code, B, H, W, rgb=FAKE):
    return [(lib.tu_yuvp_to_rgb(dense, fr, code, rgb, B, H, W, None), L().last_error()),
            (lib.tu_rgb_to_yuvp(rgb, dense, fr, code, B, H, W, None), L().last_error())]


def expect(results, *words):
    for rc, msg in results:
        assert rc == L().TU_ERR_ARG, msg
        for w in words:
            assert w in msg, (w, msg)


def test_single_ops_reject_codes_and_arguments(lib):
    _l = L()
    for code in bad_codes() + (_l.TU_U8, _l.TU_U8 | _l.TU_LAYOUT_NV12, _l.TU_U16 | _l.TU_LAYOUT_P010, _l.TU_F16):
        expect(both_ops(lib, FAKE, None, code, 1, 4, 4), "code must be")
        expect(both_ops(lib, None, frames3(1, 4, 4, "yuv444p16"), code, 1, 4, 4), "code must be")
    for fmt, code in codes().items():
        expect(both_ops(lib, FAKE, frames3(1, 4, 4, fmt), code, 1, 4, 4), "exactly one")
        expect(both_ops(lib, None, None, code, 1, 4, 4), "exactly one")
        expect(both_ops(lib, FAKE, None, code, 0, 4, 4), "bad argument")
        expect(both_ops(lib, FAKE, None, code, 65536, 4, 4), "bad argument")
        expect(both_ops(lib, FAKE, None, code, 1, 4, 4, rgb=None), "bad argument")
        expect(both_ops(lib, FAKE, None, code, 1, 0, 4), "bad argument")
        w16 = fmt == "yuv444p16"
        # yuv420p reads and writes pairs of fp16 RGB values (4 bytes); 4:4:4 single elements
        expect(both_ops(lib, FAKE, None, code, 1, 4, 4, rgb=FAKE + (1 if fmt == "yuv444p" else 2)), "RGB buffer", "fp32" if w16 else "fp16")
        if fmt != "yuv444p":
            expect(both_ops(lib, FAKE + 1, None, code, 1, 4, 4), "dense", "2-byte aligned")
        expect(both_ops(lib, FAKE, None, code, 1, 30000, 30000), "too large")
    p420 = codes()["yuv420p"]
    for H, W in ((3, 4), (4, 5), (1, 1)):
        expect(both_ops(lib, FAKE, None, p420, 1, H, W), "yuv420p", "even")
        expect(both_ops(lib, None, frames3(1, H, W + W % 2, "yuv420p"), p420, 1, H, W), "even")


@pytest.mark.parametrize("fmt", ["yuv420p", "yuv444p", "yuv444p16"])
def test_descriptor_rejections(lib, fmt):
    code = codes()[fmt]
    B, H, W = 3, 8, 10
    s = 2 if fmt == "yuv444p16" else 1
    cw = W // 2 if fmt == "yuv420p" else W
    for field in ("y", "u", "v"):
        fr = frames3(B, H, W, fmt)
        setattr(fr[1], field, None)
        expect(both_ops(lib, None, fr, code, B, H, W), "frame 1", f"{field} is NULL")
    for field, row in (("y_pitch", W), ("u_pitch", cw), ("v_pitch", cw)):
        fr = frames3(B, H, W, fmt)
        setattr(fr[2], field, (row - 1) * s)
        expect(both_ops(lib, None, fr, code, B, H, W), "frame 2", field, "smaller than the row's %d samples" % row)
        setattr(fr[2], field, -row * s)
        expect(both_ops(lib, None, fr, code, B, H, W), "frame 2", field)
    # 2-byte alignment: the yuv420p luma plane (pairs), every yuv444p16 plane (words); yuv444p planes and yuv420p chroma take any address
    for field in ("y", "u", "v", "y_pitch", "u_pitch", "v_pitch"):
        fr = frames3(B, H, W, fmt)
        setattr(fr[0], field, getattr(fr[0], field) + 1)
        if fmt == "yuv444p16" or (fmt == "yuv420p" and field.startswith("y")):
            expect(both_ops(lib, None, fr, code, B, H, W), "frame 0", field.split("_")[0], "multiples of 2 bytes")
        else:
            msg = [m for rc, m in both_ops(lib, None, fr, code, B, H, W, rgb=None)]
            assert all("bad argument" in m for m in msg), msg      # the descriptor itself passes (the NULL RGB buffer fails first)
    # dense rows (pitch = row) are fine: only the later frame's fault is reported
    fr = frames3(B, H, W, fmt, pitch_extra=0)
    fr[2].v = None
    expect(both_ops(lib, None, fr, code, B, H, W), "frame 2", "v is NULL")
    if fmt != "yuv420p":
        expect(both_ops(lib, None, frames3(1, 70000, 8, fmt), code, 1, 70000, 8), "65535 rows")


def _weights():
    return _packed("WindowTransformer", torch.bfloat16)


def test_forward_rejections_before_any_launch(lib):
    _l = L()
    pw = _weights()
    w = C.byref(pw.struct)
    p420, p444, p16 = codes().values()
    nv12, p010 = _l.TU_U8 | _l.TU_LAYOUT_NV12, _l.TU_U16 | _l.TU_LAYOUT_P010
    B, H, W, oh, ow = 2, 72, 104, 108, 156
    P2 = _l.TuFramePlanes
    pairs = (P2 * B)(*[P2(FAKE, FAKE + 8192, 256, 256) for _ in range(B)])

    def fwd(x, xfr, i, o, ofr, oc, Hn=H, Wn=W, ohn=oh, own=ow):
        rc = lib.tu_forward_frames(w, x, xfr, i, o, ofr, oc, B, Hn, Wn, ohn, own, 0, _l.TU_BF16, 1, FAKE, 1 << 40, None)
        return rc, _l.last_error()

    xf = frames3(B, H, W, "yuv420p")
    expect([fwd(FAKE, xf, p420, FAKE, None, _l.TU_F32)], "either x or x_frames")
    expect([fwd(FAKE, None, p420, FAKE, frames3(B, oh, ow, "yuv444p"), p444)], "either out or out_frames")
    for i in (_l.TU_U8, _l.TU_F16, _l.TU_U8 | _l.TU_LAYOUT_HWC):
        expect([fwd(None, xf, i, FAKE, None, _l.TU_F32)], "x_frames", "planar YUV input")
    for o in (_l.TU_F32, _l.TU_U8 | _l.TU_LAYOUT_RGBA):
        expect([fwd(FAKE, None, p420, None, frames3(B, oh, ow, "yuv444p"), o)], "out_frames", "planar YUV output")
    # descriptors are read as the side's type: a bad one names the side, the frame and the field
    bad = frames3(B, H, W, "yuv444p16")
    bad[1].u_pitch = 2 * W - 2
    expect([fwd(None, bad, p16, FAKE, None, _l.TU_F32)], "x_frames", "frame 1", "u_pitch")
    bad = frames3(B, oh, ow, "yuv420p")
    bad[0].y += 1
    expect([fwd(None, pairs, nv12, None, bad, p420)], "out_frames", "frame 0", "y", "multiples of 2 bytes")
    # codes, sizes
    for code in bad_codes():
        expect([fwd(FAKE, None, code, FAKE, None, _l.TU_F32)], "TU_LAYOUT_YUV444P")
        expect([fwd(FAKE, None, _l.TU_F32, FAKE, None, code)], "TU_LAYOUT_YUV444P")
    expect([fwd(None, frames3(B, H + 1, W, "yuv420p"), p420, FAKE, None, _l.TU_F32, Hn=H + 1)], "yuv420p input", "even")
    expect([fwd(FAKE, None, p420, FAKE, None, p420, ohn=oh + 1)], "yuv420p output", "even")
    # tu_forward_planes takes TuFramePlanes only: never on a planar side
    rc = lib.tu_forward_planes(w, None, pairs, p444, FAKE, None, _l.TU_F32, B, H, W, oh, ow, 0, _l.TU_BF16, 1, FAKE, 1 << 40, None)
    expect([(rc, _l.last_error())], "TuFramePlanes3")
    rc = lib.tu_forward_planes(w, FAKE, None, p010, None, pairs, p16, B, H, W, oh, ow, 0, _l.TU_BF16, 1, FAKE, 1 << 40, None)
    expect([(rc, _l.last_error())], "TuFramePlanes3")
    # never a compute dtype
    for code in codes().values():
        assert lib.tu_forward_workspace_bytes(0, 1, 72, 104, 108, 156, 0, code) == 0


def _align(n):
    return (n + 1023) // 1024 * 1024


def test_workspace_sizes(lib):
    """the existing code pairs size as before; each planar side adds its planar fp16 (8-bit) / fp32 (yuv444p16) RGB frame; 0 for every
    invalid combination; a surfaces call needs exactly the dense call's workspace"""
    from tests.golden.cases import CASES
    _l = L()
    p420, p444, p16 = codes().values()
    nv12, p010, u8 = _l.TU_U8 | _l.TU_LAYOUT_NV12, _l.TU_U16 | _l.TU_LAYOUT_P010, _l.TU_U8
    plain = [_l.TU_F32, _l.TU_BF16, _l.TU_F16, u8, u8 | _l.TU_LAYOUT_HWC, u8 | _l.TU_LAYOUT_BGRA]
    packs = {}
    for name, c in CASES.items():
        H, W, oh, ow, s = _geometry(c)
        B = c["shape"][0]
        ev_in, ev_out = H % 2 == 0 and W % 2 == 0, oh % 2 == 0 and ow % 2 == 0
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
            for i in plain:
                assert q(i, _l.TU_F32) == base and q(_l.TU_F32, i) == base, (name, i)
            for yuv in (0, _l.TU_YUV_BT601 | _l.TU_YUV_FULL_RANGE):
                for code, eb in ((p444, 2), (p16, 4), (p420, 2)):
                    even = code != p420
                    assert q(code | yuv, _l.TU_F32) == (base + _align(fin * eb) if even or ev_in else 0), (name, hex(code))
                    assert q(_l.TU_F32, code | yuv) == (base + _align(fout * eb) if even or ev_out else 0), (name, hex(code))
                    assert q(code | yuv, u8 | _l.TU_LAYOUT_HWC_BGR) == q(code | yuv, _l.TU_F32), name
            assert q(p16 | _l.TU_YUV_BT2020, p16) == base + _align(fin * 4) + _align(fout * 4), name
            assert q(p444, p16) == base + _align(fin * 2) + _align(fout * 4), name
            if ev_in and ev_out:
                assert q(p420, p420) == base + _align(fin * 2) + _align(fout * 2), name
                assert q(p420, p010) == q(nv12, p010) and q(p010, p420) == q(p010, nv12), name
                assert q(nv12, p444) == base + _align(fin * 2) + _align(fout * 2), name
            for bad in bad_codes():
                assert q(bad, _l.TU_F32) == 0 and q(_l.TU_F32, bad) == 0, (name, hex(bad))
    # surfaces: one byte less than the dense query is TU_ERR_WORKSPACE from the sizing pass, before any launch
    pw = _weights()
    w = C.byref(pw.struct)
    B, H, W, oh, ow = 2, 72, 104, 108, 156
    for i, o in ((p420, p444), (p444, p420), (p16, p16), (p420, _l.TU_U8)):
        need = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, i, o)
        xf = frames3(B, H, W, {p420: "yuv420p", p444: "yuv444p", p16: "yuv444p16"}[i])
        of = frames3(B, oh, ow, {p420: "yuv420p", p444: "yuv444p", p16: "yuv444p16"}[o]) if o != _l.TU_U8 else None
        rc = lib.tu_forward_frames(w, None, xf, i, None if of else FAKE, of, o, B, H, W, oh, ow, 0, _l.TU_BF16, 1, FAKE, need - 1, None)
        assert rc == _l.TU_ERR_WORKSPACE and ("need %d bytes" % need) in _l.last_error(), (hex(i), hex(o))


# ---------------------------------------------------------------------------------------------------------------------------------
# Python
def test_plane_triples_rejections():
    from transformerupscaler_b200 import engine
    y, u = torch.zeros(8, 16, dtype=torch.uint8), torch.zeros(4, 8, dtype=torch.uint8)
    bad = [
        [],
        (y, u, u),                                                        # a triple, not a list of triples
        [(y, u)],                                                         # a pair
        [(y, u, u.numpy())],
        [(y.to(torch.uint16), u.to(torch.uint16), u.to(torch.uint16))],  # 16-bit planes for yuv420p
        [(y[None], u, u)],
        [(torch.zeros(8, 32, dtype=torch.uint8)[:, ::2], u, u)],          # non-unit stride along W
        [(y, u, torch.zeros(4, 9, dtype=torch.uint8))],                   # v is not (H/2, W/2)
        [(y, y, y)],                                                      # 4:4:4 planes for 4:2:0
        [(torch.zeros(7, 16, dtype=torch.uint8), torch.zeros(3, 8, dtype=torch.uint8), torch.zeros(3, 8, dtype=torch.uint8))],
        [(y, u, u)],                                                      # host tensors
    ]
    for fr in bad:
        with pytest.raises(ValueError):
            engine.plane_triples(fr, "yuv420p", "frames")
    with pytest.raises(ValueError):
        engine.plane_triples([(y, y, u)], "yuv444p", "frames")
    with pytest.raises(ValueError):
        engine.plane_triples([(y, y, y)], "yuv444p16", "frames")


def test_run_forward_value_errors():
    from transformerupscaler_b200 import engine
    x420 = torch.zeros(1, 12, 16, dtype=torch.uint8)
    x444 = torch.zeros(1, 3, 8, 16, dtype=torch.uint8)

    def rf(x, out_dtype=torch.uint8, **kw):
        return engine.run_forward(0, "WindowTransformer", x, (12, 24), None, True, True, out_dtype, **kw)
    with pytest.raises(ValueError, match="BT.2020"):                   # BT.2020 needs a 16-bit side and no 8-bit YUV side
        rf(x444, in_layout="yuv444p", yuv="bt2020")
    with pytest.raises(ValueError, match="BT.2020"):
        rf(x444.to(torch.uint16), torch.uint8, in_layout="yuv444p16", out_layout="yuv420p", yuv="bt2020_full")
    with pytest.raises(ValueError, match="no NV12 side"):              # the existing message where no planar side takes part
        rf(x420, torch.uint16, in_layout="nv12", out_layout="p010", yuv="bt2020")
    with pytest.raises(ValueError, match="uint16 frames"):
        rf(x444, torch.uint8, in_layout="yuv444p", out_layout="yuv444p16")
    with pytest.raises(ValueError, match="uint8 frames"):
        rf(x444, torch.uint16, in_layout="yuv444p", out_layout="yuv444p")
    with pytest.raises(ValueError, match=r"\(B, 3, H, W\)"):           # a yuv444p16 layout on uint8 data
        rf(x444, torch.uint16, in_layout="yuv444p16", out_layout="yuv444p16")
    with pytest.raises(ValueError, match=r"\(B, 3H/2, W\)"):
        rf(x444, in_layout="yuv420p")
    with pytest.raises(ValueError, match="yuv420p output frames need an even"):
        engine.run_forward(0, "WindowTransformer", x420, (13, 24), None, True, True, torch.uint8, in_layout="yuv420p",
                           out_layout="yuv420p")
    y, u = torch.zeros(8, 16, dtype=torch.uint8), torch.zeros(4, 8, dtype=torch.uint8)
    with pytest.raises(ValueError, match="triple"):                     # out= of a planar side takes triples
        rf(x420, in_layout="yuv420p", out_layout="yuv420p", out=[(y, u)])


def test_model_and_wrappers():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.models.WindowTransformer.model import TransformerModel
    from transformerupscaler_b200.pipeline import FramePipeline
    m = TransformerModel().eval()
    y, u = torch.zeros(8, 16, dtype=torch.uint8), torch.zeros(4, 8, dtype=torch.uint8)
    with pytest.raises(ValueError, match="in_layout"):
        m([(y, u, u)], in_layout="hwc", res_out=(12, 24))
    with pytest.raises((ValueError, RuntimeError)):                     # no CUDA here: the CPU check may come first
        m(torch.zeros(1, 3, 8, 8, dtype=torch.uint8), in_layout="yuv444p16", res_out=(12, 12))
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(m)([(y, u, u)], in_layout="yuv420p")
    with pytest.raises(TypeError, match="out="):
        FramePipeline(m, device=torch.device("cpu"), in_layout="yuv420p", out_layout="yuv420p", out=[(y, u, u)])


def test_resize_plumbing(monkeypatch):
    """FastTransformer's Resize path ends in tu::rgb_to_yuvp / tu::rgb_to_yuvp_planes, from fp16 (8-bit) or fp32 (yuv444p16) RGB"""
    from transformerupscaler_b200 import _lib as L, engine
    calls = []

    def fake_forward(x, handle, oh, ow, scale, cbf, code, clamp, in_layout=0):
        calls.append(("fwd", oh, ow, hex(code), hex(in_layout)))
        return torch.zeros(*engine._image_shape(x.shape[0], 3, oh, ow, code), dtype=engine._TORCH_DT[code & 0xFF])

    def fake_resize(x, oh, ow, clamp, out_code=-1, alpha=None):
        calls.append(("resize", oh, ow, hex(out_code)))
        return torch.zeros(x.shape[0], 3, oh, ow, dtype=engine._TORCH_DT[out_code & 0xFF])

    def fake_to_yuvp(x, code):
        calls.append(("to_yuvp", x.dtype, hex(code)))
        return torch.zeros(*engine._image_shape(x.shape[0], 3, x.shape[2], x.shape[3], code))

    monkeypatch.setattr(engine, "tu_forward", fake_forward)
    monkeypatch.setattr(engine, "tu_resize_aa", fake_resize)
    monkeypatch.setattr(engine, "tu_rgb_to_yuvp", fake_to_yuvp)
    p420, p16 = L.TU_U8 | L.TU_LAYOUT_YUV420P, L.TU_U16 | L.TU_LAYOUT_YUV444P
    x = torch.zeros(2, 60, 56, dtype=torch.uint8)
    out = engine.run_forward(1, "FastTransformer", x, (60, 84), None, True, True, torch.uint8, in_layout="yuv420p",
                             out_layout="yuv420p", yuv="bt601")
    assert tuple(out.shape) == (2, 90, 84)
    assert calls == [("fwd", 80, 112, hex(L.TU_F32), hex(L.TU_LAYOUT_YUV420P | L.TU_YUV_BT601)),
                     ("resize", 60, 84, hex(L.TU_F16)), ("to_yuvp", torch.float16, hex(p420 | L.TU_YUV_BT601))]
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", torch.zeros(2, 3, 40, 56, dtype=torch.uint16), (60, 84), None, True, True,
                             torch.uint16, in_layout="yuv444p16", out_layout="yuv444p16", yuv="bt2020")
    assert tuple(out.shape) == (2, 3, 60, 84)
    assert calls[1:] == [("resize", 60, 84, hex(L.TU_F32)), ("to_yuvp", torch.float32, hex(p16 | L.TU_YUV_BT2020))]


def test_fake_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    from transformerupscaler_b200 import _lib as L, engine  # noqa: F401  (registers the tu:: ops)
    p420, p444, p16 = L.TU_U8 | L.TU_LAYOUT_YUV420P, L.TU_U8 | L.TU_LAYOUT_YUV444P, L.TU_U16 | L.TU_LAYOUT_YUV444P
    with FakeTensorMode():
        x = torch.empty(2, 12, 16, dtype=torch.uint8)
        y = torch.ops.tu.forward(x, 1, 12, 18, 0, True, p444, True, L.TU_LAYOUT_YUV420P)
        assert tuple(y.shape) == (2, 3, 12, 18) and y.dtype == torch.uint8
        y = torch.ops.tu.forward(x, 1, 12, 18, 0, True, p16, True, L.TU_LAYOUT_YUV420P)
        assert tuple(y.shape) == (2, 3, 12, 18) and y.dtype == torch.uint16
        y = torch.ops.tu.forward(x, 1, 12, 18, 0, True, p420, True, L.TU_LAYOUT_YUV420P)
        assert tuple(y.shape) == (2, 18, 18) and y.dtype == torch.uint8
        planes = [torch.empty(8, 16, dtype=torch.uint8), torch.empty(4, 8, dtype=torch.uint8), torch.empty(4, 8, dtype=torch.uint8)] * 2
        y = torch.ops.tu.forward_planes(None, planes, [], 1, 12, 18, 0, True, p16, True, L.TU_LAYOUT_YUV420P)
        assert tuple(y.shape) == (2, 3, 12, 18) and y.dtype == torch.uint16
        y = torch.ops.tu.forward_planes(None, planes, planes, 1, 8, 16, 0, True, p420, True, L.TU_LAYOUT_YUV420P)
        assert tuple(y.shape) == (0,)
        f = torch.empty(2, 3, 6, 10, dtype=torch.float16)
        assert tuple(torch.ops.tu.rgb_to_yuvp(f, p420).shape) == (2, 9, 10)
        assert tuple(torch.ops.tu.rgb_to_yuvp(f, p444).shape) == (2, 3, 6, 10)
        r = torch.ops.tu.rgb_to_yuvp(f.float(), p16)
        assert tuple(r.shape) == (2, 3, 6, 10) and r.dtype == torch.uint16
        assert torch.ops.tu.rgb_to_yuvp_planes(f, planes, p420) is None
