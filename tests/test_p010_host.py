"""CPU: P010 video frames (TU_U16 | TU_LAYOUT_P010) -- the conversion oracle, its agreement with a float64 evaluation of the
defining equations (BT.709, BT.601, BT.2020 / BT.2100), the exact endpoints, the identity with the NV12 oracle, the low bits of the
16-bit words, the C-ABI constants and symbols, the rejections, and the workspace query tu_forward_workspace_bytes_io.

The oracle functions below are the definition the kernels of csrc/resample.cu follow operation for operation (include/tu_b200.h
states the formulas): plain fp32 torch ops on the CPU, each one correctly rounded, no fused multiply-add.  tests/test_gpu_p010.py
compares the kernels with them bit for bit."""
import ctypes as C
import os
import re

import pytest
import torch

from tests.test_nv12_host import _div, _geometry, _packed, _upsample, oracle_nv12_to_rgb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLOURS10 = ("bt709", "bt601", "bt2020", "bt709_full", "bt601_full", "bt2020_full")
SPECIAL = (0, 64, 512, 940, 960, 1023)
MATRIX = {"bt709": (0.2126, 0.0722), "bt601": (0.299, 0.114), "bt2020": (0.2627, 0.0593)}


def _params(yuv):
    """(Kr, Kb, yo, ys, cs) of a colour name, in float64"""
    kr, kb = MATRIX[yuv.split("_")[0]]
    full = yuv.endswith("_full")
    return kr, kb, (0.0 if full else 64.0), (1023.0 if full else 876.0), (1023.0 if full else 896.0)


def coefficients10(yuv):
    """every coefficient computed in float64 and rounded once to float32 (0-dim tensors)"""
    kr, kb, yo, ys, cs = _params(yuv)
    kg = 1.0 - kr - kb
    v = dict(yo=yo, ys=ys, cs=cs,
             a_rv=2 * (1 - kr), a_bu=2 * (1 - kb), a_gu=-2 * (1 - kb) * kb / kg, a_gv=-2 * (1 - kr) * kr / kg,
             kr=kr, kg=kg, kb=kb, cb_r=-kr / (2 * (1 - kb)), cb_g=-kg / (2 * (1 - kb)), cr_g=-kg / (2 * (1 - kr)),
             cr_b=-kb / (2 * (1 - kr)))
    return {k: torch.tensor(x, dtype=torch.float32) for k, x in v.items()}


def words_to_codes(p010):
    """uint16 words -> int32 10-bit codes (the high 10 bits)"""
    return p010.cpu().to(torch.int32) >> 6


def codes_to_words(codes):
    return (codes.to(torch.int32) << 6).to(torch.uint16)


def oracle_p010_to_rgb(p010, yuv="bt709"):
    """P010 frames (B, 3H/2, W) uint16 -> planar RGB (B, 3, H, W) fp32 clamped to [0, 1]"""
    f = words_to_codes(p010)
    B, R, W = f.shape
    H = R * 2 // 3
    k = coefficients10(yuv)
    y = f[:, :H].float()
    ch = f[:, H:].reshape(B, H // 2, W // 2, 2).float()
    yn = _div(y - k["yo"], k["ys"])
    un = _div(_upsample(ch[..., 0], H, W) - 512.0, k["cs"])
    vn = _div(_upsample(ch[..., 1], H, W) - 512.0, k["cs"])
    r = yn + k["a_rv"] * vn
    g = (yn + k["a_gu"] * un) + k["a_gv"] * vn
    b = yn + k["a_bu"] * un
    return torch.stack([r, g, b], 1).clamp(0, 1)


def _code10(v):
    return torch.floor(v + 0.5).clamp(0, 1023).to(torch.int32)


def oracle_rgb_to_p010(rgb, yuv="bt709"):
    """planar RGB (B, 3, H, W) fp32 -> P010 frames (B, 3H/2, W) uint16 (codes << 6)"""
    p = rgb.cpu().float()
    B, _, H, W = p.shape
    k = coefficients10(yuv)
    yl = (k["kr"] * p[:, 0] + k["kg"] * p[:, 1]) + k["kb"] * p[:, 2]
    vs = p[:, :, 0::2] + p[:, :, 1::2]                          # column sums of the row pairs, (B, 3, H/2, W)
    c1, c2 = vs[..., 0::2], vs[..., 1::2]                       # columns 2j, 2j+1
    c0 = torch.cat([c1[..., :1], c2[..., :-1]], -1)             # column 2j-1, clamped at 0
    bar = ((c0 + 2 * c1) + c2) * 0.125
    cb = (k["cb_r"] * bar[:, 0] + k["cb_g"] * bar[:, 1]) + 0.5 * bar[:, 2]
    cr = (0.5 * bar[:, 0] + k["cr_g"] * bar[:, 1]) + k["cr_b"] * bar[:, 2]
    Y = _code10(k["ys"] * yl + k["yo"])
    uv = torch.stack([_code10(k["cs"] * cb + 512.0), _code10(k["cs"] * cr + 512.0)], -1).reshape(B, H // 2, W)
    return codes_to_words(torch.cat([Y, uv], 1))


def chroma_lattice():
    """(U, V) codes: a coprime-stride lattice (strides 33 and 31) over 0..1023 plus the special codes, every pair of the two"""
    us = sorted(set(range(0, 1024, 33)) | set(SPECIAL))
    vs = sorted(set(range(0, 1024, 31)) | set(SPECIAL))
    return [(u, v) for u in us for v in vs]


def flat_chroma_frames10(H=32, W=32, pairs=None):
    """P010 words: frame n has chroma pairs[n] everywhere and luma 0..1023 over its first 1024 pixels (every Y code), so the chroma
    upsampling sees flat planes"""
    assert H * W >= 1024
    pairs = chroma_lattice() if pairs is None else pairs
    n = len(pairs)
    y = torch.arange(H * W, dtype=torch.int32) % 1024
    f = torch.empty(n, H * 3 // 2, W, dtype=torch.int32)
    f[:, :H] = y.reshape(H, W)
    ch = torch.tensor(pairs, dtype=torch.int32)                  # (n, 2)
    f[:, H:] = ch[:, None, None, :].expand(n, H // 2, W // 2, 2).reshape(n, H // 2, W)
    return codes_to_words(f)


def f64_ycc_to_rgb(Y, U, V, yuv):
    """the defining equations in float64 (flat chroma): codes -> R, G, B clamped to [0, 1]"""
    kr, kb, yo, ys, cs = _params(yuv)
    kg = 1.0 - kr - kb
    y, u, v = (Y - yo) / ys, (U - 512.0) / cs, (V - 512.0) / cs
    r = y + 2 * (1 - kr) * v
    g = y - 2 * (1 - kb) * kb / kg * u - 2 * (1 - kr) * kr / kg * v
    b = y + 2 * (1 - kb) * u
    return torch.stack([r, g, b], 1).clamp(0, 1)


# ---------------------------------------------------------------------------------------------------------------------------------
# the oracle
@pytest.mark.parametrize("yuv", COLOURS10)
def test_oracle_to_rgb_matches_float64_equations(yuv):
    """every Y code, the (U, V) lattice: within one 10-bit code of the float64 result (in fact far closer)"""
    f = flat_chroma_frames10()
    got = oracle_p010_to_rgb(f, yuv).reshape(f.shape[0], 3, -1)[..., :1024].double()
    codes = words_to_codes(f)
    Y = codes[:, :32].reshape(f.shape[0], -1)[:, :1024].double()
    U = codes[:, 32, 0].double()[:, None].expand_as(Y)
    V = codes[:, 32, 1].double()[:, None].expand_as(Y)
    want = f64_ycc_to_rgb(Y, U, V, yuv)
    err = (got - want).abs().max().item()
    assert err * 1023 <= 1
    assert err < 1e-6


@pytest.mark.parametrize("yuv", COLOURS10)
def test_oracle_to_p010_matches_float64_equations(yuv):
    """random colours on flat 2x2 blocks (the chroma filter sees flat columns): codes within one of the float64 rounding"""
    kr, kb, yo, ys, cs = _params(yuv)
    kg = 1.0 - kr - kb
    g = torch.Generator().manual_seed(5)
    n = 8192
    col = torch.rand(n, 3, generator=g, dtype=torch.float64)
    img = col.float()[:, :, None, None].expand(n, 3, 2, 2).contiguous()
    got = words_to_codes(oracle_rgb_to_p010(img, yuv))                    # (n, 3, 2)
    c = img[:, :, 0, 0].double()
    yl = kr * c[:, 0] + kg * c[:, 1] + kb * c[:, 2]
    cb = (c[:, 2] - yl) / (2 * (1 - kb))
    cr = (c[:, 0] - yl) / (2 * (1 - kr))
    ccs = 1023.0 if yuv.endswith("_full") else 896.0
    want_y = torch.floor(ys * yl + yo + 0.5).clamp(0, 1023)
    want_u = torch.floor(ccs * cb + 512 + 0.5).clamp(0, 1023)
    want_v = torch.floor(ccs * cr + 512 + 0.5).clamp(0, 1023)
    assert (got[:, :2].reshape(n, 4).double() - want_y[:, None]).abs().max().item() <= 1
    assert (got[:, 2, 0].double() - want_u).abs().max().item() <= 1
    assert (got[:, 2, 1].double() - want_v).abs().max().item() <= 1


@pytest.mark.parametrize("yuv", COLOURS10)
def test_exact_endpoints(yuv):
    full = yuv.endswith("_full")
    lo, hi = (0, 1023) if full else (64, 940)
    f = torch.full((2, 3, 2), 512, dtype=torch.int32)
    f[0, :2], f[1, :2] = lo, hi
    f = codes_to_words(f)
    rgb = oracle_p010_to_rgb(f, yuv)
    assert torch.equal(rgb[0], torch.zeros(3, 2, 2)) and torch.equal(rgb[1], torch.ones(3, 2, 2))
    assert torch.equal(oracle_rgb_to_p010(rgb, yuv), f)


@pytest.mark.parametrize("yuv", ["bt709", "bt601"])
def test_identity_with_nv12_oracle(yuv):
    """limited range: P010 words = NV12 codes << 8 give the NV12 oracle's RGB bit for bit after .half() -- 4 (C - 128) / (4 * 224) is
    the same real quotient as (C - 128) / 224, so it rounds to the same float, and every step before it is exact"""
    g = torch.Generator().manual_seed(9)
    nv12 = torch.randint(0, 256, (4, 24, 34), generator=g, dtype=torch.uint8)
    p010 = (nv12.to(torch.int32) << 8).to(torch.uint16)
    assert torch.equal(oracle_p010_to_rgb(p010, yuv).half(), oracle_nv12_to_rgb(nv12, yuv).half())
    assert torch.equal(oracle_p010_to_rgb(p010, yuv), oracle_nv12_to_rgb(nv12, yuv))


def test_low_bits_ignored_and_zero_on_output():
    g = torch.Generator().manual_seed(4)
    codes = torch.randint(0, 1024, (3, 12, 10), generator=g, dtype=torch.int32)
    clean = codes_to_words(codes)
    dirty = ((codes << 6) | torch.randint(0, 64, codes.shape, generator=g, dtype=torch.int32)).to(torch.uint16)
    for yuv in COLOURS10:
        rgb = oracle_p010_to_rgb(dirty, yuv)
        assert torch.equal(rgb, oracle_p010_to_rgb(clean, yuv))
        out = oracle_rgb_to_p010(rgb, yuv).to(torch.int32)
        assert int((out & 63).max()) == 0 and int(out.max()) <= 1023 << 6


def test_upsampling_sums_are_exact():
    """the largest chroma sums (8 * 1023) and their quarter / eighth steps are exact in fp32: the upsampled planes equal a float64
    evaluation"""
    g = torch.Generator().manual_seed(2)
    c = torch.randint(0, 1024, (2, 6, 7), generator=g).float()
    c[0] = 1023.0
    up = _upsample(c, 12, 14)
    assert torch.equal(up.double(), _upsample(c.double(), 12, 14))


# ---------------------------------------------------------------------------------------------------------------------------------
# the C ABI
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from transformerupscaler_b200 import _lib
    return _lib.load()


def test_abi_constants_and_symbols(lib):
    from transformerupscaler_b200 import _lib, engine
    src = open(os.path.join(ROOT, "include", "tu_b200.h")).read()
    for name, val in (("TU_LAYOUT_P010", 0x800), ("TU_YUV_BT2020", 0x4000)):
        assert re.search(r"#define\s+%s\s+0x%x\b" % (name, val), src, re.I), name
        assert getattr(_lib, name) == val
    assert re.search(r"#define\s+TU_U16\s+4\b", src) and _lib.TU_U16 == 4
    assert re.search(r"#define\s+TU_U16_P010\s+\(TU_U16 \| TU_LAYOUT_P010\)", src)
    for n in ("tu_p010_to_rgb", "tu_rgb_to_p010"):
        assert hasattr(lib, n) and n in _lib.SIGNATURES
    assert engine.LAYOUTS["p010"] == _lib.TU_LAYOUT_P010
    assert set(engine.YUV) == {"bt709", "bt601", "bt709_full", "bt601_full"}
    assert engine.yuv_code("bt2020") == _lib.TU_YUV_BT2020
    assert engine.yuv_code("bt2020_full") == _lib.TU_YUV_BT2020 | _lib.TU_YUV_FULL_RANGE
    p010 = _lib.TU_U16 | _lib.TU_LAYOUT_P010
    assert _lib.dtype_size(p010 | _lib.TU_YUV_BT2020) == 2 and _lib.dtype_size(_lib.TU_U16) == 2
    assert engine._is_p010(p010) and not engine._is_nv12(p010) and not engine._is_p010(_lib.TU_U8 | _lib.TU_LAYOUT_NV12)
    assert engine._image_shape(2, 3, 8, 10, p010 | _lib.TU_YUV_BT2020) == (2, 12, 10)
    assert engine._DT[torch.uint16] == _lib.TU_U16 and engine._TORCH_DT[_lib.TU_U16] == torch.uint16


def _bad_p010_codes():
    from transformerupscaler_b200 import _lib as L
    p010 = L.TU_U16 | L.TU_LAYOUT_P010
    return (L.TU_U16, L.TU_U16 | L.TU_YUV_BT2020, L.TU_U8 | L.TU_LAYOUT_P010, L.TU_F32 | L.TU_LAYOUT_P010,
            p010 | L.TU_YUV_BT601 | L.TU_YUV_BT2020, L.TU_U16 | L.TU_LAYOUT_NV12, p010 | L.TU_LAYOUT_NV12, p010 | 0x8000,
            L.TU_U8 | L.TU_LAYOUT_NV12, L.TU_U16 | L.TU_LAYOUT_HWC)


def test_conversion_ops_reject_bad_codes_and_sizes_without_gpu(lib):
    """argument checks come before any launch: bad codes, odd sizes, too many frames and misaligned buffers return TU_ERR_ARG on a
    CPU-only host too"""
    from transformerupscaler_b200 import _lib as L
    p010 = L.TU_U16 | L.TU_LAYOUT_P010
    fake = 1 << 20                                                   # never dereferenced: every call below fails its checks
    for code in _bad_p010_codes():
        assert lib.tu_p010_to_rgb(fake, code, fake, 1, 4, 4, None) == L.TU_ERR_ARG, hex(code)
        assert lib.tu_rgb_to_p010(fake, fake, code, 1, 4, 4, None) == L.TU_ERR_ARG, hex(code)
    for H, W in ((3, 4), (4, 5)):
        assert lib.tu_p010_to_rgb(fake, p010, fake, 1, H, W, None) == L.TU_ERR_ARG
        assert lib.tu_rgb_to_p010(fake, fake, p010, 1, H, W, None) == L.TU_ERR_ARG
        assert "even" in L.last_error()
    assert lib.tu_p010_to_rgb(fake, p010, fake, 65536, 4, 4, None) == L.TU_ERR_ARG
    assert lib.tu_rgb_to_p010(fake, fake, p010, 0, 4, 4, None) == L.TU_ERR_ARG
    assert lib.tu_p010_to_rgb(fake + 2, p010, fake, 1, 4, 4, None) == L.TU_ERR_ARG          # P010 buffer 4-byte aligned
    assert lib.tu_rgb_to_p010(fake + 4, fake, p010, 1, 4, 4, None) == L.TU_ERR_ARG          # RGB buffer 8-byte aligned
    assert "aligned" in L.last_error()
    # BT.2020 is P010 only: the NV12 ops reject it, and the P010 codes
    nv12 = L.TU_U8 | L.TU_LAYOUT_NV12
    for code in (nv12 | L.TU_YUV_BT2020, p010, p010 | L.TU_YUV_BT2020):
        assert lib.tu_nv12_to_rgb(fake, code, fake, 1, 4, 4, None) == L.TU_ERR_ARG
        assert lib.tu_rgb_to_nv12(fake, fake, code, 1, 4, 4, None) == L.TU_ERR_ARG


def test_other_image_entry_points_reject_u16_without_gpu(lib):
    """TU_U16 is a P010 word only: no other entry point reads it as some other dtype"""
    from transformerupscaler_b200 import _lib as L
    fake = 1 << 20
    fin = (C.c_float * 84)()
    for code in (L.TU_U16, L.TU_U16 | L.TU_LAYOUT_P010):
        assert lib.tu_stem_conv(fake, code, fake, None, fake, fake, L.TU_BF16, 1, 8, 8, None) == L.TU_ERR_ARG
        assert lib.tu_conv12_fused(fake, code, fake, fake, fake, fake, fake, 1, 8, 8, None) == L.TU_ERR_ARG
        assert lib.tu_bicubic_add_clamp(fake, code, 8, 8, None, 0, 0, fake, L.TU_F32, 1, 16, 16, 1, None) == L.TU_ERR_ARG
        assert lib.tu_bicubic_add_clamp(fake, L.TU_F32, 8, 8, None, 0, 0, fake, code, 1, 16, 16, 1, None) == L.TU_ERR_ARG
        assert lib.tu_subpixel_conv_add(fake, fake, fake, 2, C.addressof(fin), fake, fake, code, 1, 8, 8, 1, None) == L.TU_ERR_ARG
        assert lib.tu_final_conv_add(fake, fake, fake, fake, fake, code, 1, 8, 8, 1, None) == L.TU_ERR_ARG
        assert lib.tu_resize_bilinear_aa(fake, code, fake, 1, 8, 8, 4, 4, 1, None) == L.TU_ERR_ARG
        assert lib.tu_resize_bilinear_aa_to(fake, code, fake, L.TU_F32, 1, 8, 8, 4, 4, 1, None) == L.TU_ERR_ARG
        assert lib.tu_resize_bilinear_aa_to(fake, L.TU_F32, fake, code, 1, 8, 8, 4, 4, 1, None) == L.TU_ERR_ARG
        assert lib.tu_frames_to_planar(fake, code, fake, 1, 8, 8, None) == L.TU_ERR_ARG
    # and never a compute dtype
    assert lib.tu_forward_workspace_bytes(0, 1, 72, 104, 108, 156, 0, L.TU_U16) == 0


def _align(n):
    return (n + 1023) // 1024 * 1024


def test_workspace_io_query(lib):
    """exactly the old sizes for every pair of existing codes (NV12 included: base + its fp16 frames); a P010 side adds its planar
    fp32 frames; 0 for every invalid combination"""
    from tests.golden.cases import CASES
    from transformerupscaler_b200 import _lib as L
    u8, nv12, p010 = L.TU_U8, L.TU_U8 | L.TU_LAYOUT_NV12, L.TU_U16 | L.TU_LAYOUT_P010
    plain = [L.TU_F32, L.TU_BF16, L.TU_F16, u8, u8 | L.TU_LAYOUT_HWC, u8 | L.TU_LAYOUT_HWC_BGR]
    packs = {}
    for name, c in CASES.items():
        H, W, oh, ow, s = _geometry(c)
        B = c["shape"][0]
        ev_in, ev_out = H % 2 == 0 and W % 2 == 0, oh % 2 == 0 and ow % 2 == 0
        fin, fout = B * 3 * H * W, B * 3 * oh * ow
        for cdt, tdt in ((L.TU_BF16, torch.bfloat16), (L.TU_F32, torch.float32)):
            key = (c["model"], cdt)
            if key not in packs:
                packs[key] = _packed(c["model"], tdt)
            w = C.byref(packs[key].struct)
            base = lib.tu_forward_workspace_bytes_for(w, B, H, W, oh, ow, s, cdt)
            assert base > 0, name

            def q(i, o):
                return lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, i, o)
            for i in plain:
                for o in plain:
                    assert q(i, o) == base, (name, i, o)
            for yuv in (0, L.TU_YUV_BT601 | L.TU_YUV_FULL_RANGE):
                if ev_in:
                    assert q(nv12 | yuv, L.TU_F32) == base + _align(fin * 2), name
                if ev_out:
                    assert q(L.TU_F32, nv12 | yuv) == base + _align(fout * 2), name
                if ev_in and ev_out:
                    assert q(nv12 | yuv, nv12 | yuv) == base + _align(fin * 2) + _align(fout * 2), name
            for yuv in (0, L.TU_YUV_BT601, L.TU_YUV_BT2020 | L.TU_YUV_FULL_RANGE):
                n_in, n_out, n_both = q(p010 | yuv, L.TU_F32), q(L.TU_F32, p010 | yuv), q(p010 | yuv, p010 | yuv)
                if ev_in:
                    assert n_in == base + _align(fin * 4) and n_in >= base + fin * 4, name
                else:
                    assert n_in == 0 and "even" in L.last_error(), name
                if ev_out:
                    assert n_out == base + _align(fout * 4) and n_out >= base + fout * 4, name
                else:
                    assert n_out == 0, name
                if ev_in and ev_out:
                    assert n_both == base + _align(fin * 4) + _align(fout * 4), name
                    assert q(nv12, p010 | yuv) == base + _align(fin * 2) + _align(fout * 4), name
                    assert q(p010 | yuv, nv12) == base + _align(fin * 4) + _align(fout * 2), name
                    assert q(p010 | yuv, u8 | L.TU_LAYOUT_HWC_BGR) == n_in, name
                    assert q(u8, p010 | yuv) == n_out, name
            for bad in [b for b in _bad_p010_codes() if b != nv12] + [nv12 | L.TU_YUV_BT2020, L.TU_F32 | L.TU_YUV_BT2020]:
                assert q(bad, L.TU_F32) == 0 and q(L.TU_F32, bad) == 0, (name, hex(bad))
