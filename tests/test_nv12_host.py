"""CPU: NV12 video frames (TU_U8 | TU_LAYOUT_NV12) -- the conversion oracle, its agreement with OpenCV, the exact endpoints, the
C-ABI constants and symbols, and the workspace query tu_forward_workspace_bytes_io.

The oracle functions below are the definition the kernels of csrc/resample.cu follow operation for operation (include/tu_b200.h
states the formulas): plain fp32 torch ops on the CPU, each one correctly rounded, no fused multiply-add.  tests/test_gpu_nv12.py
compares the kernels with them bit for bit."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLOURS = ("bt709", "bt601", "bt709_full", "bt601_full")


def coefficients(yuv):
    """every coefficient computed in float64 and rounded once to float32 (0-dim tensors)"""
    bt601, full = yuv.startswith("bt601"), yuv.endswith("_full")
    kr, kb = (0.299, 0.114) if bt601 else (0.2126, 0.0722)
    kg = 1.0 - kr - kb
    v = dict(yo=0.0 if full else 16.0, ys=255.0 if full else 219.0, cs=255.0 if full else 224.0,
             a_rv=2 * (1 - kr), a_bu=2 * (1 - kb), a_gu=-2 * (1 - kb) * kb / kg, a_gv=-2 * (1 - kr) * kr / kg,
             kr=kr, kg=kg, kb=kb, cb_r=-kr / (2 * (1 - kb)), cb_g=-kg / (2 * (1 - kb)), cr_g=-kg / (2 * (1 - kr)),
             cr_b=-kb / (2 * (1 - kr)))
    return {k: torch.tensor(x, dtype=torch.float32) for k, x in v.items()}


def _div(a, d):
    """a / d elementwise against a full tensor (a true division, whatever a scalar divisor's fast path would do)"""
    return a / torch.full_like(a, float(d))


def _upsample(c, H, W):
    """(B, H/2, W/2) chroma codes -> (B, H, W), bilinear with type-0 siting, edges clamped (exact in fp32)"""
    prev = torch.cat([c[:, :1], c[:, :-1]], 1)
    nxt = torch.cat([c[:, 1:], c[:, -1:]], 1)
    rows = torch.stack([0.25 * prev + 0.75 * c, 0.75 * c + 0.25 * nxt], 2).reshape(c.shape[0], H, W // 2)
    right = torch.cat([rows[..., 1:], rows[..., -1:]], 2)
    return torch.stack([rows, 0.5 * rows + 0.5 * right], 3).reshape(c.shape[0], H, W)


def oracle_nv12_to_rgb(nv12, yuv="bt709"):
    """NV12 frames (B, 3H/2, W) uint8 -> planar RGB (B, 3, H, W) fp32 clamped to [0, 1] (the kernel stores this rounded to fp16)"""
    f = nv12.cpu()
    B, R, W = f.shape
    H = R * 2 // 3
    k = coefficients(yuv)
    y = f[:, :H].float()
    ch = f[:, H:].reshape(B, H // 2, W // 2, 2).float()
    yn = _div(y - k["yo"], k["ys"])
    un = _div(_upsample(ch[..., 0], H, W) - 128.0, k["cs"])
    vn = _div(_upsample(ch[..., 1], H, W) - 128.0, k["cs"])
    r = yn + k["a_rv"] * vn
    g = (yn + k["a_gu"] * un) + k["a_gv"] * vn
    b = yn + k["a_bu"] * un
    return torch.stack([r, g, b], 1).clamp(0, 1)


def _code(v):
    return torch.floor(v + 0.5).clamp(0, 255).to(torch.uint8)


def oracle_rgb_to_nv12(rgb, yuv="bt709"):
    """planar RGB (B, 3, H, W) (fp16 values, widened exactly) -> NV12 frames (B, 3H/2, W) uint8"""
    p = rgb.cpu().float()
    B, _, H, W = p.shape
    k = coefficients(yuv)
    yl = (k["kr"] * p[:, 0] + k["kg"] * p[:, 1]) + k["kb"] * p[:, 2]
    vs = p[:, :, 0::2] + p[:, :, 1::2]                          # column sums of the row pairs, (B, 3, H/2, W)
    c1, c2 = vs[..., 0::2], vs[..., 1::2]                       # columns 2j, 2j+1
    c0 = torch.cat([c1[..., :1], c2[..., :-1]], -1)             # column 2j-1, clamped at 0
    bar = ((c0 + 2 * c1) + c2) * 0.125
    cb = (k["cb_r"] * bar[:, 0] + k["cb_g"] * bar[:, 1]) + 0.5 * bar[:, 2]
    cr = (0.5 * bar[:, 0] + k["cr_g"] * bar[:, 1]) + k["cr_b"] * bar[:, 2]
    Y = _code(k["ys"] * yl + k["yo"])
    uv = torch.stack([_code(k["cs"] * cb + 128.0), _code(k["cs"] * cr + 128.0)], -1).reshape(B, H // 2, W)
    return torch.cat([Y, uv], 1)


def flat_chroma_frames(H=16, W=16):
    """every (Y, U, V) triple: frame u*256 + v has chroma (u, v) everywhere and luma 0..255 over its first 256 pixels, so the
    chroma upsampling sees flat planes"""
    assert H * W >= 256
    n = 256 * 256
    y = torch.arange(H * W) % 256
    f = torch.empty(n, H * 3 // 2, W, dtype=torch.uint8)
    f[:, :H] = y.reshape(H, W).to(torch.uint8)
    uv = torch.arange(n)
    ch = torch.stack([uv // 256, uv % 256], -1).to(torch.uint8)          # (n, 2)
    f[:, H:] = ch[:, None, None, :].expand(n, H // 2, W // 2, 2).reshape(n, H // 2, W)
    return f


# ---------------------------------------------------------------------------------------------------------------------------------
# the oracle
@pytest.mark.parametrize("yuv", COLOURS)
def test_exact_endpoints(yuv):
    full = yuv.endswith("_full")
    lo, hi = (0, 255) if full else (16, 235)
    f = torch.full((2, 3, 2), 128, dtype=torch.uint8)
    f[0, :2], f[1, :2] = lo, hi
    rgb = oracle_nv12_to_rgb(f, yuv)
    assert torch.equal(rgb[0], torch.zeros(3, 2, 2)) and torch.equal(rgb[1], torch.ones(3, 2, 2))
    assert torch.equal(rgb.half().float(), rgb)
    back = oracle_rgb_to_nv12(rgb.half(), yuv)
    assert torch.equal(back, f)


def test_upsampling_siting():
    """type-0 siting: a chroma step between rows 1 and 2 of the chroma plane shows up with weights 1/4, 3/4 on luma rows 2i / 2i+1,
    and co-sited columns keep the sample while odd columns average their two neighbours"""
    c = torch.tensor([[[0.0, 8.0], [64.0, 8.0]]])                     # (1, 2, 2)
    u = _upsample(c, 4, 4)[0]
    assert u[:, 0].tolist() == [0.0, 16.0, 48.0, 64.0]
    assert u[0].tolist() == [0.0, 4.0, 8.0, 8.0]


def test_oracle_matches_opencv_bt601_limited():
    cv2 = pytest.importorskip("cv2")
    # NV12 -> RGB over every legal (Y, U, V) triple (OpenCV clamps Y < 16 before its matrix: compare legal codes only)
    f = flat_chroma_frames()
    ours = oracle_nv12_to_rgb(f, "bt601")                              # (n, 3, 16, 16)
    y = f[:, :16].reshape(-1, 256)[:, :256]
    uv = f[:, 16, :2]
    legal = ((uv >= 16) & (uv <= 240)).all(1)
    ocv = np.stack([cv2.cvtColor(np.ascontiguousarray(fr), cv2.COLOR_YUV2RGB_NV12) for fr in f[legal].numpy()])   # (m, 16, 16, 3)
    o = torch.from_numpy(ocv).permute(0, 3, 1, 2).reshape(-1, 3, 256)
    q = torch.floor(ours[legal].reshape(-1, 3, 256) * 255 + 0.5)
    ly = ((y[legal] >= 16) & (y[legal] <= 235))[:, None, :].expand_as(q)
    assert (q - o.float()).abs()[ly].max().item() <= 1
    # RGB -> NV12: random colours on flat 2x2 blocks (the chroma filter then sees flat columns)
    g = torch.Generator().manual_seed(3)
    n = 4096
    col = torch.randint(0, 256, (n, 3), generator=g, dtype=torch.uint8)
    img = col[:, :, None, None].expand(n, 3, 2, 2).contiguous()
    ours = oracle_rgb_to_nv12((img.float() / 255).half(), "bt601")     # (n, 3, 2)
    yuv = np.stack([cv2.cvtColor(np.ascontiguousarray(im.permute(1, 2, 0).numpy()), cv2.COLOR_RGB2YUV_I420) for im in img])  # (n, 3, 2)
    assert (ours[:, :2].int() - torch.from_numpy(yuv[:, :2]).int()).abs().max().item() <= 1            # Y
    ocv_uv = torch.from_numpy(np.stack([yuv[:, 2, 0], yuv[:, 2, 1]], 1)).int()                           # I420: U then V
    assert (ours[:, 2].int() - ocv_uv).abs().max().item() <= 1


def test_fp16_intermediate_keeps_codes():
    """the forward converts through planar fp16: NV12 -> fp16 RGB -> NV12 moves a legal code by at most one (fp16 keeps 11 bits
    on [0, 1], under 0.06 of a code, and the chroma filter of flat frames is the identity)"""
    f = flat_chroma_frames()[::97]
    for yuv in COLOURS:
        back = oracle_rgb_to_nv12(oracle_nv12_to_rgb(f, yuv).half(), yuv)
        lo, hi = (0, 255) if yuv.endswith("_full") else (16, 235)
        yv = f[:, :16]
        legal_y = (yv >= lo) & (yv <= hi)
        rgb = oracle_nv12_to_rgb(f, yuv)
        inside = ((rgb > 0) & (rgb < 1)).all(1)                      # no channel clipped
        m = legal_y & inside
        assert (back[:, :16].int() - yv.int()).abs()[m].max().item() <= 1, yuv


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
    for name, val in (("TU_LAYOUT_NV12", 0x400), ("TU_YUV_BT601", 0x1000), ("TU_YUV_FULL_RANGE", 0x2000)):
        assert re.search(r"#define\s+%s\s+0x%x\b" % (name, val), src, re.I), name
        assert getattr(_lib, name) == val
    for n in ("tu_nv12_to_rgb", "tu_rgb_to_nv12", "tu_forward_workspace_bytes_io"):
        assert hasattr(lib, n) and n in _lib.SIGNATURES
    assert engine.LAYOUTS["nv12"] == _lib.TU_LAYOUT_NV12
    assert set(engine.YUV) == set(COLOURS)
    nv12 = _lib.TU_U8 | _lib.TU_LAYOUT_NV12
    for yuv in COLOURS:
        code = nv12 | engine.yuv_code(yuv)
        assert _lib.dtype_size(code) == 1
    # the existing codes decode as before: interleaved layouts in bits 8..9, never the NV12 bit
    assert _lib.TU_LAYOUT_HWC >> 8 == 1 and _lib.TU_LAYOUT_HWC_BGR >> 8 == 2
    assert not engine._is_nv12(_lib.TU_U8 | _lib.TU_LAYOUT_HWC_BGR) and engine._is_nv12(nv12 | _lib.TU_YUV_FULL_RANGE)
    assert engine._image_shape(2, 3, 8, 10, nv12 | _lib.TU_YUV_BT601) == (2, 12, 10)
    assert engine._image_shape(2, 3, 8, 10, _lib.TU_U8 | _lib.TU_LAYOUT_HWC) == (2, 8, 10, 3)
    assert engine._image_shape(2, 3, 8, 10, _lib.TU_F16) == (2, 3, 8, 10)


def test_conversion_ops_reject_bad_codes_and_sizes_without_gpu(lib):
    """argument checks come before any launch: bad codes and odd sizes return TU_ERR_ARG on a CPU-only host too"""
    from transformerupscaler_b200 import _lib
    nv12 = _lib.TU_U8 | _lib.TU_LAYOUT_NV12
    fake = 1 << 20                                                   # never dereferenced: every call below fails its checks
    for code in (_lib.TU_U8, _lib.TU_F32 | _lib.TU_LAYOUT_NV12, _lib.TU_U8 | _lib.TU_YUV_BT601, nv12 | 0x4000,
                 _lib.TU_U8 | _lib.TU_LAYOUT_HWC):
        assert lib.tu_nv12_to_rgb(fake, code, fake, 1, 4, 4, None) == _lib.TU_ERR_ARG
        assert lib.tu_rgb_to_nv12(fake, fake, code, 1, 4, 4, None) == _lib.TU_ERR_ARG
    for H, W in ((3, 4), (4, 5)):
        assert lib.tu_nv12_to_rgb(fake, nv12, fake, 1, H, W, None) == _lib.TU_ERR_ARG
        assert lib.tu_rgb_to_nv12(fake, fake, nv12, 1, H, W, None) == _lib.TU_ERR_ARG
        assert "even" in _lib.last_error()
    assert lib.tu_nv12_to_rgb(fake, nv12, fake, 1, 0, 4, None) == _lib.TU_ERR_ARG


def _packed(model, dt):
    from oracle.weights import synth_state_dict
    from transformerupscaler_b200.packing import PackedWeights
    return PackedWeights(model, synth_state_dict(model, 1), dt, torch.device("cpu"))


def _geometry(c):
    """(H, W, outH, outW, scale) of a golden case, the way engine.run_forward computes them"""
    import math
    _, _, H, W = c["shape"]
    kw = c["kw"]
    if "upscale_factor" in kw:
        f = kw["upscale_factor"]
        return H, W, H * f, W * f, f
    oh, ow = kw["res_out"]
    if c["model"] != "FastTransformer":
        return H, W, oh, ow, 0
    s = math.ceil(max(oh / H, ow / W))
    return H, W, H * s, W * s, s


def test_workspace_io_query(lib):
    from tests.golden.cases import CASES
    from transformerupscaler_b200 import _lib
    u8, nv12 = _lib.TU_U8, _lib.TU_U8 | _lib.TU_LAYOUT_NV12
    plain = [_lib.TU_F32, _lib.TU_BF16, _lib.TU_F16, u8, u8 | _lib.TU_LAYOUT_HWC, u8 | _lib.TU_LAYOUT_HWC_BGR]
    packs = {}
    for name, c in CASES.items():
        H, W, oh, ow, s = _geometry(c)
        B = c["shape"][0]
        for cdt, tdt in ((_lib.TU_BF16, torch.bfloat16), (_lib.TU_F32, torch.float32)):
            key = (c["model"], cdt)
            if key not in packs:
                packs[key] = _packed(c["model"], tdt)
            w = C.byref(packs[key].struct)
            base = lib.tu_forward_workspace_bytes_for(w, B, H, W, oh, ow, s, cdt)
            assert base > 0, name
            for i in plain:
                for o in plain:
                    assert lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, i, o) == base, (name, i, o)
            ev_in, ev_out = H % 2 == 0 and W % 2 == 0, oh % 2 == 0 and ow % 2 == 0
            for yuv in (0, _lib.TU_YUV_BT601 | _lib.TU_YUV_FULL_RANGE):
                n_in = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, nv12 | yuv, _lib.TU_F32)
                n_out = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, _lib.TU_F32, nv12 | yuv)
                n_both = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, nv12 | yuv, nv12 | yuv)
                if ev_in:
                    assert n_in >= base + B * 3 * H * W * 2, name
                else:
                    assert n_in == 0 and "even" in _lib.last_error(), name
                if ev_out:
                    assert n_out >= base + B * 3 * oh * ow * 2, name
                if ev_in and ev_out:
                    assert n_both > max(n_in, n_out), name
            # an NV12 bit on a float code, colour bits without NV12: rejected (size 0)
            assert lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, _lib.TU_F32 | _lib.TU_LAYOUT_NV12, _lib.TU_F32) == 0
            assert lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, s, cdt, _lib.TU_F32, u8 | _lib.TU_YUV_BT601) == 0
