"""CPU: 4-byte RGBA / BGRA frames (TU_U8 | TU_LAYOUT_RGBA / TU_LAYOUT_BGRA) -- the constants and the decoding of the enumerated layout
nibble, the rejections of the C ABI, the workspace query, the alpha oracle, and the Python-side errors and fake shapes.

The alpha oracle below is the definition tu_resample_alpha follows operation for operation (include/tu_b200.h states the formulas):
oracle.upscaler_oracle.bicubic_nchw on float32 codes -- its taps and weights are _cubic_taps(..., torch.float32), every product and
sum one correctly rounded fp32 tensor op -- then floor(. + 0.5) clamped to 0..255.  tests/test_gpu_rgba.py compares the kernel with
it bit for bit."""
import ctypes as C
import os
import re

import pytest
import torch

from oracle.upscaler_oracle import _cubic_taps, bicubic_nchw
from tests.test_nv12_host import _geometry, _packed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 1 << 20                      # never dereferenced: every call below fails its checks before any launch


def oracle_alpha(frames, out_h, out_w):
    """(B, H, W, 4) uint8 frames -> the (B, out_h, out_w) uint8 alpha plane of a 4-byte output"""
    a = frames[..., 3].cpu().float()[:, None]
    return torch.floor(bicubic_nchw(a, (out_h, out_w)) + 0.5).clamp(0, 255).to(torch.uint8)[:, 0]


def const_plane_codes(ks, H, W, out_h, out_w):
    """oracle_alpha of constant planes k (one per entry of ks) without materialising them: on a constant plane a row sum only
    depends on the output column's weights and the result on (column weights, row weights), so the fp32 evaluation runs over the
    distinct weight vectors.  Returns (len(ks), distinct row weights, distinct column weights) codes."""
    _, wx = _cubic_taps(W, out_w, torch.float32)
    _, wy = _cubic_taps(H, out_h, torch.float32)
    wx, wy = torch.unique(wx.t(), dim=0), torch.unique(wy.t(), dim=0)            # (nx, 4), (ny, 4)
    k = torch.tensor(ks, dtype=torch.float32)[:, None]
    acc = torch.zeros(len(ks), wx.shape[0])
    for j in range(4):
        acc = acc + k * wx[None, :, j]
    a = torch.zeros(len(ks), wy.shape[0], wx.shape[0])
    for i in range(4):
        a = a + acc[:, None, :] * wy[None, :, i, None]
    return torch.floor(a + 0.5).clamp(0, 255)


# geometries of the forward paths: 720p -> 1080p (WindowTransformer), 720p -> 4K (ResidualTransformer), FastTransformer's integer
# scales, its Resize path (x2 then down to 1080p) and ragged sizes, upscaling and downscaling
GEOMETRIES = [(720, 1280, 1080, 1920), (720, 1280, 2160, 3840)] + [(720, 1280, 720 * s, 1280 * s) for s in (2, 3, 4, 6)] + [
    (37, 53, 91, 29), (5, 7, 13, 11), (1, 1, 3, 5), (100, 80, 33, 50), (131, 189, 200, 280), (36, 52, 72, 104)]


# ---------------------------------------------------------------------------------------------------------------------------------
# the alpha oracle
def test_alpha_oracle_matches_float64_bicubic():
    """within rounding of a float64 evaluation (float64 coordinates, weights and sums): at most one code apart, and only where the
    float64 value sits within 1e-3 of a rounding boundary"""
    g = torch.Generator().manual_seed(3)
    for H, W, oh, ow in [(37, 53, 91, 29), (24, 40, 36, 60), (50, 30, 20, 70)]:
        fr = torch.randint(0, 256, (2, H, W, 4), generator=g, dtype=torch.uint8)
        got = oracle_alpha(fr, oh, ow).double()
        f64 = bicubic_nchw(fr[..., 3].double()[:, None], (oh, ow))[:, 0]
        want = torch.floor(f64 + 0.5).clamp(0, 255)
        diff = (got - want).abs()
        assert diff.max().item() <= 1
        frac = (f64 + 0.5) - torch.floor(f64 + 0.5)
        near = torch.minimum(frac, 1 - frac) < 1e-3
        assert bool((near | (diff == 0)).all())
        assert (f64.clamp(0, 255) - got).abs().max().item() < 0.5 + 1e-3


@pytest.mark.parametrize("geom", GEOMETRIES, ids=lambda g: "%dx%d-%dx%d" % g)
def test_constant_alpha_stays_exact(geom):
    """every constant plane k = 0..255 comes back as k (255 stays opaque, 0 stays transparent)"""
    codes = const_plane_codes(list(range(256)), *geom)
    want = torch.arange(256, dtype=torch.float32)[:, None, None].expand_as(codes)
    assert torch.equal(codes, want)


def test_constant_plane_shortcut_is_the_oracle():
    """the distinct-weights evaluation gives exactly what the oracle gives on materialised constant planes"""
    for H, W, oh, ow in [(37, 53, 91, 29), (6, 8, 9, 12), (5, 7, 13, 11)]:
        ks = [0, 1, 77, 128, 254, 255]
        fr = torch.zeros(len(ks), H, W, 4, dtype=torch.uint8)
        fr[..., 3] = torch.tensor(ks, dtype=torch.uint8)[:, None, None]
        full = oracle_alpha(fr, oh, ow).float()
        short = const_plane_codes(ks, H, W, oh, ow)
        for n in range(len(ks)):
            assert torch.equal(torch.unique(full[n]), torch.unique(short[n]))


def test_alpha_oracle_range_and_extremes():
    """codes stay in 0..255 on the planes that overshoot most (bicubic rings at 0 / 255 edges)"""
    g = torch.Generator().manual_seed(8)
    fr = torch.randint(0, 256, (3, 17, 23, 4), generator=g, dtype=torch.uint8)
    fr[0, ..., 3] = (torch.arange(23) % 2 * 255).to(torch.uint8)                 # a 0 / 255 column checkerboard
    fr[1, ..., 3] = ((torch.arange(17)[:, None] + torch.arange(23)) % 2 * 255).to(torch.uint8)
    a = bicubic_nchw(fr[..., 3].float()[:, None], (40, 50))
    assert a.min().item() < -0.5 and a.max().item() > 255.5                       # the clamp is exercised
    out = oracle_alpha(fr, 40, 50)
    assert out.dtype == torch.uint8 and out.shape == (3, 40, 50)


# ---------------------------------------------------------------------------------------------------------------------------------
# constants and the enumerated layout nibble
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from transformerupscaler_b200 import _lib
    return _lib.load()


def test_abi_constants_and_symbols(lib):
    from transformerupscaler_b200 import _lib, engine
    src = open(os.path.join(ROOT, "include", "tu_b200.h")).read()
    for name, val in (("TU_LAYOUT_RGBA", 0x300), ("TU_LAYOUT_BGRA", 0x500)):
        assert re.search(r"#define\s+%s\s+0x%x\b" % (name, val), src, re.I), name
        assert getattr(_lib, name) == val
    assert re.search(r"#define\s+TU_U8_RGBA\s+\(TU_U8 \| TU_LAYOUT_RGBA\)", src)
    assert re.search(r"#define\s+TU_U8_BGRA\s+\(TU_U8 \| TU_LAYOUT_BGRA\)", src)
    for n in ("tu_resample_alpha", "tu_resize_bilinear_aa_to_alpha"):
        assert hasattr(lib, n) and n in _lib.SIGNATURES
    assert engine.LAYOUTS["rgba"] == 0x300 and engine.LAYOUTS["bgra"] == 0x500
    assert engine.layout_code("bgra") == _lib.TU_LAYOUT_BGRA
    assert _lib.dtype_size(_lib.TU_U8 | _lib.TU_LAYOUT_BGRA) == 1


def test_layout_nibble_is_an_enumeration():
    """0x500 (BGRA) is never NV12 (0x400) and 0x300 (RGBA) never HWC / HWC_BGR; NV12 / P010 codes with colour bits decode as before"""
    from transformerupscaler_b200 import _lib as L, engine
    u8 = L.TU_U8
    rgba, bgra, nv12, p010 = u8 | L.TU_LAYOUT_RGBA, u8 | L.TU_LAYOUT_BGRA, u8 | L.TU_LAYOUT_NV12, L.TU_U16 | L.TU_LAYOUT_P010
    for c in (rgba, bgra):
        assert engine._is_px4(c) and not engine._is_nv12(c) and not engine._is_p010(c)
        assert engine._image_shape(2, 3, 8, 10, c) == (2, 8, 10, 4)
    for c in (u8 | L.TU_LAYOUT_HWC, u8 | L.TU_LAYOUT_HWC_BGR):
        assert not engine._is_px4(c) and engine._image_shape(2, 3, 8, 10, c) == (2, 8, 10, 3)
    for bits in (0, L.TU_YUV_BT601, L.TU_YUV_FULL_RANGE, L.TU_YUV_BT601 | L.TU_YUV_FULL_RANGE):
        assert engine._is_nv12(nv12 | bits) and not engine._is_px4(nv12 | bits) and not engine._is_p010(nv12 | bits)
        assert engine._image_shape(2, 3, 8, 10, nv12 | bits) == (2, 12, 10)
    for bits in (0, L.TU_YUV_BT601, L.TU_YUV_BT2020, L.TU_YUV_BT2020 | L.TU_YUV_FULL_RANGE):
        assert engine._is_p010(p010 | bits) and not engine._is_px4(p010 | bits) and not engine._is_nv12(p010 | bits)
        assert engine._image_shape(2, 3, 8, 10, p010 | bits) == (2, 12, 10)
    assert engine._image_shape(2, 3, 8, 10, u8) == (2, 3, 8, 10)


def test_c_side_decodes_whole_values(lib):
    """through the workspace query: a BGRA side takes no NV12 frame buffer and needs no even size (NV12 does), an RGBA pair of sides
    adds its alpha plane where an HWC pair adds nothing"""
    from transformerupscaler_b200 import _lib as L
    pw = _packed("WindowTransformer", torch.bfloat16)
    w = C.byref(pw.struct)
    u8 = L.TU_U8
    B, H, W, oh, ow = 1, 72, 104, 108, 156
    base = lib.tu_forward_workspace_bytes_for(w, B, H, W, oh, ow, 0, L.TU_BF16)

    def q(i, o, h=H, wd=W, a=oh, b=ow):
        return lib.tu_forward_workspace_bytes_io(w, B, h, wd, a, b, 0, L.TU_BF16, i, o)
    assert q(u8 | L.TU_LAYOUT_BGRA, L.TU_F32) == base
    assert q(L.TU_F32, u8 | L.TU_LAYOUT_BGRA) == base
    assert q(u8 | L.TU_LAYOUT_NV12, L.TU_F32) > base
    b_odd = lib.tu_forward_workspace_bytes_for(w, B, 71, 103, 107, 155, 0, L.TU_BF16)
    assert q(u8 | L.TU_LAYOUT_BGRA, u8 | L.TU_LAYOUT_HWC, 71, 103, 107, 155) == b_odd > 0
    assert q(u8 | L.TU_LAYOUT_NV12, L.TU_F32, 71, 103, 107, 155) == 0
    assert q(u8 | L.TU_LAYOUT_HWC, u8 | L.TU_LAYOUT_HWC) == base
    assert q(u8 | L.TU_LAYOUT_RGBA, u8 | L.TU_LAYOUT_RGBA) == base + _align(B * oh * ow)


# ---------------------------------------------------------------------------------------------------------------------------------
# rejections
def _bad_px4_codes():
    from transformerupscaler_b200 import _lib as L
    out = []
    for lay in (L.TU_LAYOUT_RGBA, L.TU_LAYOUT_BGRA):
        out += [L.TU_F32 | lay, L.TU_BF16 | lay, L.TU_F16 | lay, L.TU_U16 | lay]
        out += [L.TU_U8 | lay | bit for bit in (L.TU_YUV_BT601, L.TU_YUV_FULL_RANGE, L.TU_YUV_BT2020)]
    return out


def test_workspace_queries_reject_bad_codes(lib):
    from transformerupscaler_b200 import _lib as L
    pw = _packed("WindowTransformer", torch.bfloat16)
    w = C.byref(pw.struct)
    for bad in _bad_px4_codes():
        assert lib.tu_forward_workspace_bytes_io(w, 1, 72, 104, 108, 156, 0, L.TU_BF16, bad, L.TU_F32) == 0, hex(bad)
        assert lib.tu_forward_workspace_bytes_io(w, 1, 72, 104, 108, 156, 0, L.TU_BF16, L.TU_F32, bad) == 0, hex(bad)
        assert lib.tu_forward_workspace_bytes_io(w, 1, 72, 104, 108, 156, 0, L.TU_BF16, L.TU_U8 | L.TU_LAYOUT_RGBA, bad) == 0, hex(bad)
    for cdt in (L.TU_U8 | L.TU_LAYOUT_RGBA, L.TU_U8 | L.TU_LAYOUT_BGRA):           # never a compute dtype
        assert lib.tu_forward_workspace_bytes(0, 1, 72, 104, 108, 156, 0, cdt) == 0
        assert lib.tu_forward_workspace_bytes_for(w, 1, 72, 104, 108, 156, 0, cdt) == 0


def test_forward_rejects_bad_codes_and_frame_arrays(lib):
    """every rejection comes before anything is enqueued: TU_ERR_ARG on a CPU-only host"""
    from transformerupscaler_b200 import _lib as L
    pw = _packed("WindowTransformer", torch.bfloat16)
    w = C.byref(pw.struct)
    rgba, bgra = L.TU_U8 | L.TU_LAYOUT_RGBA, L.TU_U8 | L.TU_LAYOUT_BGRA

    def fwd(i, o, x=FAKE, xf=None, out=FAKE, of=None, cdt=L.TU_BF16):
        return lib.tu_forward_planes(w, x, xf, i, out, of, o, 1, 72, 104, 108, 156, 0, cdt, 1, FAKE, 1 << 40, None)
    for bad in _bad_px4_codes():
        assert fwd(bad, L.TU_F32) == L.TU_ERR_ARG, hex(bad)
        assert fwd(L.TU_F32, bad) == L.TU_ERR_ARG, hex(bad)
        assert lib.tu_forward(w, FAKE, bad, FAKE, L.TU_F32, 1, 72, 104, 108, 156, 0, L.TU_BF16, 1, FAKE, 1 << 40, None) == L.TU_ERR_ARG
    for c in (rgba, bgra):
        assert fwd(L.TU_F32, L.TU_F32, cdt=c) == L.TU_ERR_ARG
        planes = (L.TuFramePlanes * 1)(L.TuFramePlanes(FAKE, FAKE, 104, 104))
        assert fwd(c, L.TU_F32, x=None, xf=planes) == L.TU_ERR_ARG and "x_frames" in L.last_error()
        oplanes = (L.TuFramePlanes * 1)(L.TuFramePlanes(FAKE, FAKE, 156 * 4, 156 * 4))
        assert fwd(L.TU_F32, c, out=None, of=oplanes) == L.TU_ERR_ARG and "out_frames" in L.last_error()
        assert fwd(c, c, out=FAKE + 2) == L.TU_ERR_ARG and "aligned" in L.last_error()
    # an alpha -> alpha forward given the workspace of tu_forward_workspace_bytes_for is short by the alpha plane
    need = lib.tu_forward_workspace_bytes_io(w, 1, 72, 104, 108, 156, 0, L.TU_BF16, bgra, bgra)
    base = lib.tu_forward_workspace_bytes_for(w, 1, 72, 104, 108, 156, 0, L.TU_BF16)
    assert need > base
    rc = lib.tu_forward(w, FAKE, bgra, FAKE, bgra, 1, 72, 104, 108, 156, 0, L.TU_BF16, 1, FAKE, base, None)
    assert rc == L.TU_ERR_WORKSPACE and ("need %d bytes" % need) in L.last_error()


def test_ops_reject_bad_codes(lib):
    from transformerupscaler_b200 import _lib as L
    fin = (C.c_float * 84)()
    rgba, bgra = L.TU_U8 | L.TU_LAYOUT_RGBA, L.TU_U8 | L.TU_LAYOUT_BGRA
    for c in (rgba, bgra):
        # the 64 -> 3 tail without the fused kernel writes planar images only, as for HWC
        assert lib.tu_final_conv_add(FAKE, FAKE, FAKE, FAKE, FAKE, c, 1, 8, 8, 1, None) == L.TU_ERR_ARG
        # 4-byte outputs are 4-byte aligned
        assert lib.tu_bicubic_add_clamp(FAKE, L.TU_F32, 8, 8, None, 0, 0, FAKE + 1, c, 1, 16, 16, 1, None) == L.TU_ERR_ARG
        assert lib.tu_subpixel_conv_add(FAKE, FAKE, FAKE, 2, C.addressof(fin), FAKE, FAKE + 2, c, 1, 8, 8, 1, None) == L.TU_ERR_ARG
        assert lib.tu_resize_bilinear_aa_to(FAKE, L.TU_F32, FAKE + 3, c, 1, 8, 8, 4, 4, 1, None) == L.TU_ERR_ARG
        # and never an input of these ops
        assert lib.tu_bicubic_add_clamp(FAKE, c, 8, 8, None, 0, 0, FAKE, L.TU_F32, 1, 16, 16, 1, None) == L.TU_ERR_ARG
        assert lib.tu_stem_conv(FAKE, c, FAKE, None, FAKE, FAKE, L.TU_BF16, 1, 8, 8, None) == L.TU_ERR_ARG
        assert lib.tu_resize_bilinear_aa(FAKE, c, FAKE, 1, 8, 8, 4, 4, 1, None) == L.TU_ERR_ARG
    for bad in _bad_px4_codes():
        assert lib.tu_bicubic_add_clamp(FAKE, L.TU_F32, 8, 8, None, 0, 0, FAKE, bad, 1, 16, 16, 1, None) == L.TU_ERR_ARG, hex(bad)
        assert lib.tu_subpixel_conv_add(FAKE, FAKE, FAKE, 2, C.addressof(fin), FAKE, FAKE, bad, 1, 8, 8, 1, None) == L.TU_ERR_ARG
        assert lib.tu_resize_bilinear_aa_to(FAKE, L.TU_F32, FAKE, bad, 1, 8, 8, 4, 4, 1, None) == L.TU_ERR_ARG, hex(bad)
        assert lib.tu_resample_alpha(FAKE, bad, FAKE, 1, 8, 8, 16, 16, None) == L.TU_ERR_ARG, hex(bad)
        if bad & ~0xF00:                    # (tu_frames_to_planar takes a layout: TU_F32 | TU_LAYOUT_RGBA is the layout itself)
            assert lib.tu_frames_to_planar(FAKE, bad, FAKE, 1, 8, 8, None) == L.TU_ERR_ARG, hex(bad)
    # the alpha op takes 4-byte frames only, and the Resize takes a plane only for a 4-byte output
    for code in (L.TU_U8, L.TU_U8 | L.TU_LAYOUT_HWC, L.TU_U8 | L.TU_LAYOUT_NV12, L.TU_LAYOUT_RGBA):
        assert lib.tu_resample_alpha(FAKE, code, FAKE, 1, 8, 8, 16, 16, None) == L.TU_ERR_ARG, hex(code)
    assert lib.tu_resample_alpha(FAKE, rgba, FAKE, 65536, 8, 8, 16, 16, None) == L.TU_ERR_ARG
    assert lib.tu_resample_alpha(None, rgba, FAKE, 1, 8, 8, 16, 16, None) == L.TU_ERR_ARG
    for o in (L.TU_F32, L.TU_U8 | L.TU_LAYOUT_HWC):
        assert lib.tu_resize_bilinear_aa_to_alpha(FAKE, L.TU_F32, FAKE, FAKE, o, 1, 8, 8, 4, 4, 1, None) == L.TU_ERR_ARG
    assert lib.tu_frames_to_planar(FAKE, L.TU_LAYOUT_NV12, FAKE, 1, 8, 8, None) == L.TU_ERR_ARG


# ---------------------------------------------------------------------------------------------------------------------------------
# the workspace
def _align(n):
    return (n + 1023) // 1024 * 1024


def test_workspace_io_query(lib):
    """over the golden shapes: identical to tu_forward_workspace_bytes_for for every existing code pair and every pair with alpha on
    at most one side; larger by exactly the (B, outH, outW) alpha plane for alpha -> alpha"""
    from tests.golden.cases import CASES
    from transformerupscaler_b200 import _lib as L
    u8 = L.TU_U8
    plain = [L.TU_F32, L.TU_BF16, L.TU_F16, u8, u8 | L.TU_LAYOUT_HWC, u8 | L.TU_LAYOUT_HWC_BGR]
    px4 = [u8 | L.TU_LAYOUT_RGBA, u8 | L.TU_LAYOUT_BGRA]
    packs = {}
    for name, c in CASES.items():
        H, W, oh, ow, s = _geometry(c)
        B = c["shape"][0]
        for cdt, tdt in ((L.TU_BF16, torch.bfloat16), (L.TU_F32, torch.float32)):
            key = (c["model"], cdt)
            if key not in packs:
                packs[key] = _packed(c["model"], tdt)
            w = C.byref(packs[key].struct)
            base = lib.tu_forward_workspace_bytes_for(w, B, H, W, oh, ow, s, cdt)
            assert base > 0, name

            def q(i, o):
                return lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, i, o)
            for i in plain + px4:
                for o in plain + px4:
                    want = base + _align(B * oh * ow) if (i in px4 and o in px4) else base
                    assert q(i, o) == want, (name, hex(i), hex(o))
            if H % 2 == 0 and W % 2 == 0 and oh % 2 == 0 and ow % 2 == 0:
                nv12 = u8 | L.TU_LAYOUT_NV12
                assert q(nv12, px4[1]) == q(nv12, L.TU_F32) and q(px4[0], nv12) == q(L.TU_F32, nv12), name


# ---------------------------------------------------------------------------------------------------------------------------------
# Python
def test_run_forward_value_errors():
    from transformerupscaler_b200 import engine
    x3 = torch.zeros(1, 8, 12, 3, dtype=torch.uint8)
    x4 = torch.zeros(1, 8, 12, 4, dtype=torch.uint8)
    for lay in ("rgba", "bgra"):
        with pytest.raises(ValueError, match=r"\(B, H, W, 4\)"):                # a 3-byte frame given as 4-byte
            engine.run_forward(0, "WindowTransformer", x3, (12, 18), None, True, True, torch.uint8, in_layout=lay)
        with pytest.raises(ValueError, match=r"\(B, H, W, 4\)"):
            engine.run_forward(0, "WindowTransformer", x4.float(), (12, 18), None, True, True, torch.uint8, in_layout=lay)
        with pytest.raises(ValueError, match=r"\(B, H, W, 4\), got list"):      # frame planes are not 4-byte frames
            engine.run_forward(0, "WindowTransformer", [(x4[0, ..., 0], x4[0, :4, :, 0])], (12, 18), None, True, True, torch.uint8,
                               in_layout=lay)
        with pytest.raises(ValueError, match="uint8 frames"):                   # a 4-byte output is uint8
            engine.run_forward(0, "WindowTransformer", x4, (12, 18), None, True, True, torch.float32, in_layout=lay, out_layout=lay)
        with pytest.raises(ValueError, match="NV12 / P010"):                    # out= planes are NV12 / P010 only
            engine.run_forward(0, "WindowTransformer", x4, (12, 18), None, True, True, torch.uint8, in_layout=lay, out_layout=lay,
                               out=[(x4[0, ..., 0], x4[0, :4, :, 0])])
    with pytest.raises(ValueError, match="unknown frame layout"):
        engine.layout_code("argb")


def test_model_rejects_layouts_on_float_input():
    from transformerupscaler_b200.models.WindowTransformer.model import TransformerModel
    m = TransformerModel().eval()
    for kw in (dict(in_layout="rgba"), dict(out_layout="bgra")):
        with pytest.raises((ValueError, RuntimeError)):                         # no CUDA here: the CPU check may come first
            m(torch.rand(1, 3, 16, 16), res_out=(24, 24), **kw)


def test_forward_and_resize_plumbing(monkeypatch):
    """the stand-ins of tests/test_host_logic.py: alpha -> alpha resamples the alpha to the requested size and hands it to the
    FastTransformer Resize; the other forms call the Resize without a plane; Window / Residual go straight to tu::forward"""
    from transformerupscaler_b200 import _lib as L, engine
    calls = []

    def fake_forward(x, handle, oh, ow, scale, cbf, code, clamp, in_layout=0):
        calls.append(("fwd", oh, ow, scale, hex(code), hex(in_layout)))
        return torch.zeros(*engine._image_shape(x.shape[0], 3, oh, ow, code), dtype=engine._TORCH_DT[code & 0xFF])

    def fake_resize(x, oh, ow, clamp, out_code=-1, alpha=None):
        calls.append(("resize", oh, ow, hex(out_code), None if alpha is None else tuple(alpha.shape)))
        return torch.zeros(*engine._image_shape(x.shape[0], 3, oh, ow, out_code), dtype=engine._TORCH_DT[out_code & 0xFF])

    def fake_alpha(x, code, oh, ow):
        calls.append(("alpha", hex(code), oh, ow))
        return torch.zeros(x.shape[0], oh, ow, dtype=torch.uint8)

    monkeypatch.setattr(engine, "tu_forward", fake_forward)
    monkeypatch.setattr(engine, "tu_resize_aa", fake_resize)
    monkeypatch.setattr(engine, "tu_resample_alpha", fake_alpha)
    x = torch.zeros(2, 40, 56, 4, dtype=torch.uint8)
    bgra = L.TU_U8 | L.TU_LAYOUT_BGRA
    out = engine.run_forward(1, "FastTransformer", x, (60, 84), None, True, True, torch.uint8, in_layout="bgra", out_layout="bgra")
    assert tuple(out.shape) == (2, 60, 84, 4)
    assert calls == [("fwd", 80, 112, 2, hex(L.TU_BF16), hex(L.TU_LAYOUT_BGRA)), ("alpha", hex(bgra), 60, 84),
                     ("resize", 60, 84, hex(bgra), (2, 60, 84))]
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", x, (60, 84), None, True, True, torch.uint8, in_layout="rgba", out_layout="hwc")
    assert tuple(out.shape) == (2, 60, 84, 3) and calls[-1] == ("resize", 60, 84, hex(L.TU_U8 | L.TU_LAYOUT_HWC), None)
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", x[..., :3].contiguous(), (60, 84), None, True, True, torch.uint8, in_layout="hwc",
                             out_layout="rgba")
    assert tuple(out.shape) == (2, 60, 84, 4) and calls[-1] == ("resize", 60, 84, hex(L.TU_U8 | L.TU_LAYOUT_RGBA), None)
    calls.clear()
    out = engine.run_forward(1, "WindowTransformer", x, (60, 84), None, True, True, torch.uint8, in_layout="rgba", out_layout="rgba")
    assert tuple(out.shape) == (2, 60, 84, 4)
    assert calls == [("fwd", 60, 84, 0, hex(L.TU_U8 | L.TU_LAYOUT_RGBA), hex(L.TU_LAYOUT_RGBA))]
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", x, None, 3, True, True, torch.uint8, in_layout="bgra", out_layout="bgra")
    assert tuple(out.shape) == (2, 120, 168, 4) and [c[0] for c in calls] == ["fwd"]


def test_fake_shapes():
    """the fake kernels torch.compile traces with: (B, h, w, 4) uint8 for the new codes, (B, h, w) uint8 for the alpha plane"""
    from torch._subclasses.fake_tensor import FakeTensorMode
    from transformerupscaler_b200 import _lib as L, engine  # noqa: F401  (registers the tu:: ops)
    rgba, bgra = L.TU_U8 | L.TU_LAYOUT_RGBA, L.TU_U8 | L.TU_LAYOUT_BGRA
    with FakeTensorMode():
        x = torch.empty(2, 8, 12, 4, dtype=torch.uint8)
        y = torch.ops.tu.forward(x, 1, 12, 18, 0, True, bgra, True, L.TU_LAYOUT_BGRA)
        assert tuple(y.shape) == (2, 12, 18, 4) and y.dtype == torch.uint8
        y = torch.ops.tu.forward(x, 1, 12, 18, 0, True, L.TU_U8 | L.TU_LAYOUT_HWC, True, L.TU_LAYOUT_RGBA)
        assert tuple(y.shape) == (2, 12, 18, 3)
        y = torch.ops.tu.forward_planes(x, [], [], 1, 12, 18, 0, True, rgba, True, L.TU_LAYOUT_RGBA)
        assert tuple(y.shape) == (2, 12, 18, 4)
        a = torch.ops.tu.resample_alpha(x, rgba, 12, 18)
        assert tuple(a.shape) == (2, 12, 18) and a.dtype == torch.uint8
        f = torch.empty(2, 3, 16, 24, dtype=torch.bfloat16)
        r = torch.ops.tu.resize_aa(f, 12, 18, True, bgra, a)
        assert tuple(r.shape) == (2, 12, 18, 4) and r.dtype == torch.uint8
        r = torch.ops.tu.resize_aa(f, 12, 18, True, -1)
        assert tuple(r.shape) == (2, 3, 12, 18)
