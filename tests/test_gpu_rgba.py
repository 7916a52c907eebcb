"""GPU: 4-byte RGBA / BGRA frames at both ends of the forward (csrc/resample.cu, csrc/subpixel_tail.cu).

Every comparison is bitwise.  An RGBA / BGRA input gives the forward of the same pixels given as HWC / HWC_BGR (random alpha, so the
alpha provably does not reach R, G, B); the R, G, B bytes of an RGBA / BGRA output are those of the HWC / HWC_BGR output; the alpha
bytes are the oracle of tests/test_rgba_host.py (both sides 4-byte) or 255.  Outputs written through the C ABI start from two
different sentinel fills and must come out identical: every byte of every pixel is written, alpha included."""
import ctypes as C

import pytest
import torch

from oracle.weights import synth_frames
from tests.golden.cases import CASES, FULLSIZE
from tests.test_gpu_models import build
from tests.test_gpu_p010 import natural_nv12, natural_p010
from tests.test_rgba_host import oracle_alpha

pytestmark = pytest.mark.gpu

U8, U16 = torch.uint8, torch.uint16
DEV = torch.device("cuda:0")
PAIRS = (("rgba", "hwc"), ("bgra", "hwc_bgr"))


def _L():
    from transformerupscaler_b200 import _lib
    return _lib, _lib.load()


def st():
    return torch.cuda.current_stream().cuda_stream


def frames4(B, H, W, seed):
    """natural RGB content (what a capture holds) with a random alpha byte per pixel"""
    g = torch.Generator().manual_seed(seed)
    x = torch.empty(B, H, W, 4, dtype=U8)
    x[..., :3] = (synth_frames(B, H, W, seed=seed) * 255).round().to(U8).permute(0, 2, 3, 1)
    x[..., 3] = torch.randint(0, 256, (B, H, W), generator=g, dtype=torch.int32).to(U8)
    return x


def code(layout):
    from transformerupscaler_b200 import _lib, engine
    return _lib.TU_U8 | engine.layout_code(layout)


_models = {}


def _model(name):
    c = CASES[name]
    key = (c["model"], c["wseed"])
    if key not in _models:
        _models[key] = build(c["model"], c["wseed"])[0]
    return _models[key]


def _run(M, x, kw, bf16, **lk):
    from transformerupscaler_b200 import engine
    h = M._packed(bf16, x.device)
    return engine.run_forward(h, M.ENGINE_MODEL, x, kw.get("res_out", (1080, 1920)), kw.get("upscale_factor"),
                              kw.get("require_ratio", True), bf16, U8, **lk)


def _c_forward(M, x, in_code, out_code, oh, ow, scale, bf16, fill):
    """tu_forward straight through the C ABI into an output buffer pre-filled with `fill`"""
    from transformerupscaler_b200 import engine
    L, lib = _L()
    pw = engine._REGISTRY[M._packed(bf16, x.device)]
    w = C.byref(pw.struct)
    B, H, W = x.shape[0], x.shape[1], x.shape[2]
    cdt = L.TU_BF16 if bf16 else L.TU_F32
    out = torch.full(engine._image_shape(B, 3, oh, ow, out_code), fill, dtype=U8, device=x.device)
    n = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, scale, cdt, in_code, out_code)
    assert n > 0, L.last_error()
    ws = torch.empty(n, dtype=U8, device=x.device)
    L.check(lib.tu_forward(w, x.data_ptr(), in_code, out.data_ptr(), out_code, B, H, W, oh, ow, scale, cdt, 1, ws.data_ptr(), n, st()))
    return out


def _geom(c, H, W):
    kw = c["kw"]
    if "upscale_factor" in kw:
        f = kw["upscale_factor"]
        return H * f, W * f, (f if c["model"] == "FastTransformer" else 0)
    return kw["res_out"][0], kw["res_out"][1], 0


def check_forward(M, c, x4, bf16, kw=None):
    """every claim of the module docstring for one model / case / path, both byte orders"""
    kw = kw or c["kw"]
    x4 = x4.to(DEV)
    B, H, W, _ = x4.shape
    direct = "res_out" not in kw or M.ENGINE_MODEL != "FastTransformer"
    oh, ow, scale = _geom(dict(c, kw=kw), H, W)
    a_want = None
    with torch.no_grad():
        for l4, l3 in PAIRS:
            x3 = x4[..., :3].contiguous()
            ref = _run(M, x3, kw, bf16, in_layout=l3, out_layout=l3)
            got = _run(M, x4, kw, bf16, in_layout=l4, out_layout=l4)                  # alpha -> alpha
            assert got.shape == ref.shape[:3] + (4,) and got.dtype == U8
            assert torch.equal(got[..., :3], ref), (l4, "rgb")
            if a_want is None:
                a_want = oracle_alpha(x4, got.shape[1], got.shape[2]).to(DEV)
            assert torch.equal(got[..., 3], a_want), (l4, "alpha")
            opaque = _run(M, x3, kw, bf16, in_layout=l3, out_layout=l4)              # no alpha in: 255
            assert torch.equal(opaque[..., :3], ref) and bool((opaque[..., 3] == 255).all()), (l4, "opaque")
            assert torch.equal(_run(M, x4, kw, bf16, in_layout=l4, out_layout=l3), ref), (l4, "dropped")
            planar = _run(M, x4, kw, bf16, in_layout=l4)                              # 4-byte in, uint8 CHW out
            assert torch.equal(planar, _run(M, x3, kw, bf16, in_layout=l3)), (l4, "chw")
            if direct:                                                                # every byte written (two sentinels)
                xd = x4
                s0 = _c_forward(M, xd, code(l4), code(l4), oh, ow, scale, bf16, 0x00)
                s1 = _c_forward(M, xd, code(l4), code(l4), oh, ow, scale, bf16, 0xFF)
                assert torch.equal(s0, got) and torch.equal(s1, got), (l4, "sentinel")
                s0 = _c_forward(M, xd[..., :3].contiguous(), code(l3), code(l4), oh, ow, scale, bf16, 0x00)
                assert torch.equal(s0, opaque), (l4, "sentinel opaque")


# ---------------------------------------------------------------------------------------------------------------------------------
# the single ops
@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 5, 7), (1, 3, 6), (3, 4, 6), (2, 33, 1279), (1, 720, 1280)])
def test_frames_to_planar_drops_alpha(shape):
    L, lib = _L()
    B, H, W = shape
    x4 = frames4(B, H, W, seed=H * 31 + W).to(DEV)
    x3 = x4[..., :3].contiguous()
    for lay4, lay3 in ((L.TU_LAYOUT_RGBA, L.TU_LAYOUT_HWC), (L.TU_LAYOUT_BGRA, L.TU_LAYOUT_HWC_BGR)):
        for off in (0, 1):                                                  # aligned words, and the byte path at an odd address
            buf = torch.zeros(B * H * W * 4 + 4, dtype=U8, device=DEV)
            buf[off:off + x4.numel()] = x4.reshape(-1)
            got = torch.full((B, 3, H, W), 0x5A, dtype=U8, device=DEV)
            want = torch.full((B, 3, H, W), 0xA5, dtype=U8, device=DEV)
            L.check(lib.tu_frames_to_planar(buf.data_ptr() + off, lay4, got.data_ptr(), B, H, W, st()))
            L.check(lib.tu_frames_to_planar(x3.data_ptr(), lay3, want.data_ptr(), B, H, W, st()))
            assert torch.equal(got, want), (hex(lay4), off)


ALPHA_GEOMS = [(1, 1, 1, 3, 5), (2, 5, 7, 13, 11), (1, 37, 53, 91, 29), (2, 100, 80, 33, 50), (1, 131, 189, 200, 280), (3, 6, 9, 6, 9),
               (8, 720, 1280, 1080, 1920), (2, 720, 1280, 2160, 3840)] + [(1, 720, 1280, 720 * s, 1280 * s) for s in (2, 3, 4, 6)]


@pytest.mark.parametrize("geom", ALPHA_GEOMS, ids=lambda g: "%dx%dx%d-%dx%d" % g)
def test_resample_alpha_matches_oracle(geom):
    L, lib = _L()
    B, H, W, oh, ow = geom
    x4 = frames4(B, H, W, seed=H + W + oh)
    x4[0, ..., 3] = ((torch.arange(H)[:, None] + torch.arange(W)) % 2 * 255).to(U8)        # the largest overshoots
    xd = x4.to(DEV)
    for lay in (L.TU_LAYOUT_RGBA, L.TU_LAYOUT_BGRA):
        out = torch.full((B, oh, ow), 0x5A, dtype=U8, device=DEV)
        L.check(lib.tu_resample_alpha(xd.data_ptr(), L.TU_U8 | lay, out.data_ptr(), B, H, W, oh, ow, st()))
        assert torch.equal(out.cpu(), oracle_alpha(x4, oh, ow)), hex(lay)
    # constant planes stay exact
    for k in (0, 1, 128, 255):
        xd[..., 3] = k
        out = torch.empty((B, oh, ow), dtype=U8, device=DEV)
        L.check(lib.tu_resample_alpha(xd.data_ptr(), L.TU_U8 | L.TU_LAYOUT_RGBA, out.data_ptr(), B, H, W, oh, ow, st()))
        assert bool((out == k).all()), k


def test_resize_alpha_op_and_opaque_ops():
    """tu_resize_bilinear_aa_to_alpha: the RGB bytes of the HWC output, alpha from the plane or 255, every byte written; the ops that
    write HWC write alpha 255 through their unchanged signatures"""
    from transformerupscaler_b200 import engine
    L, lib = _L()
    g = torch.Generator().manual_seed(4)
    x = torch.rand(2, 3, 40, 58, generator=g).to(DEV)
    plane = torch.randint(0, 256, (2, 27, 37), generator=g, dtype=torch.int32).to(U8).to(DEV)
    for l4, l3 in PAIRS:
        ref = engine.tu_resize_aa(x, 27, 37, True, code(l3))
        for fill in (0x00, 0xFF):
            for a in (plane, None):
                out = torch.full((2, 27, 37, 4), fill, dtype=U8, device=DEV)
                L.check(lib.tu_resize_bilinear_aa_to_alpha(x.data_ptr(), L.TU_F32, None if a is None else a.data_ptr(), out.data_ptr(),
                                                           code(l4), 2, 40, 58, 27, 37, 1, st()))
                assert torch.equal(out[..., :3], ref) and torch.equal(out[..., 3], plane if a is not None else torch.full_like(plane, 255))
        assert torch.equal(engine.tu_resize_aa(x, 27, 37, True, code(l4), plane)[..., 3], plane)
        out = torch.full((2, 27, 37, 4), 7, dtype=U8, device=DEV)
        L.check(lib.tu_resize_bilinear_aa_to(x.data_ptr(), L.TU_F32, out.data_ptr(), code(l4), 2, 40, 58, 27, 37, 1, st()))
        assert torch.equal(out[..., :3], ref) and bool((out[..., 3] == 255).all())
        # tu_bicubic_add_clamp (pair kernel at even widths, strip kernel at odd ones) with alpha 255
        for ow in (90, 91):
            ref = torch.empty(2, 60, ow, 3, dtype=U8, device=DEV)
            L.check(lib.tu_bicubic_add_clamp(x.data_ptr(), L.TU_F32, 40, 58, None, 0, 0, ref.data_ptr(), code(l3), 2, 60, ow, 1, st()))
            out = torch.full((2, 60, ow, 4), 3, dtype=U8, device=DEV)
            L.check(lib.tu_bicubic_add_clamp(x.data_ptr(), L.TU_F32, 40, 58, None, 0, 0, out.data_ptr(), code(l4), 2, 60, ow, 1, st()))
            assert torch.equal(out[..., :3], ref) and bool((out[..., 3] == 255).all()), (l4, ow)


# ---------------------------------------------------------------------------------------------------------------------------------
# whole forwards
FWD_CASES = ["window_72x104_r1p5", "window_64x80_x2", "window_131x189_odd", "fast_40x56_x2", "fast_40x56_x3", "fast_40x56_x4",
             "fast_24x32_x6", "fast_36x52_x2_reflect", "fast_40x56_res60x84", "residual_720p_1080p"]


@pytest.mark.parametrize("name", FWD_CASES)
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forward_rgba(name, path):
    c = CASES[name]
    B, _, H, W = c["shape"]
    check_forward(_model(name), c, frames4(B, H, W, seed=c["xseed"]), path == "bf16")


@pytest.mark.parametrize("factor", [3, 4, 6])
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forward_rgba_row_schedules(factor, path):
    """row schedules 3, 4, 6 of the bicubic kernel (0 and 2 run in test_forward_rgba: x1.5 and x2 WindowTransformer cases)"""
    from transformerupscaler_b200 import _lib
    assert _lib.load().tu_bicubic_row_schedule(64, 32, 64 * factor) == factor
    c = CASES["window_64x80_x2"]
    check_forward(_model("window_64x80_x2"), c, frames4(2, 64, 80, seed=40 + factor), path == "bf16", kw=dict(upscale_factor=factor))


@pytest.mark.parametrize("key,val", [("bicubic_tile", 1), ("bicubic_tile", 2), ("bicubic_pair", 1), ("bicubic_pair", 0)])
@pytest.mark.parametrize("name", ["window_72x104_r1p5", "window_64x80_x2"])
def test_forward_rgba_bicubic_variants(key, val, name):
    """both tile sizes of the row-schedule kernel, and the pair and strip kernels"""
    L, lib = _L()
    default = {"bicubic_tile": 0, "bicubic_pair": 2}[key]
    c = CASES[name]
    B, _, H, W = c["shape"]
    try:
        assert lib.tu_debug_set(key.encode(), val) == 0
        for bf16 in (True, False):
            check_forward(_model(name), c, frames4(B, H, W, seed=c["xseed"] + val), bf16)
    finally:
        lib.tu_debug_set(key.encode(), default)


@pytest.mark.parametrize("name", ["window_72x104_r1p5", "fast_36x52_x2_reflect", "fast_40x56_res60x84", "residual_720p_1080p"])
def test_forward_rgba_mixed_sides(name):
    """NV12 surfaces -> BGRA, P010 -> RGBA, RGBA -> NV12 / P010 / CHW (alpha dropped)"""
    c = CASES[name]
    B, _, H, W = c["shape"]
    M = _model(name)
    kw = c["kw"]
    with torch.no_grad():
        n = natural_nv12(B, H, W, seed=c["xseed"] + 5).to(DEV)
        planes = [(f[:H].clone(), f[H:].clone()) for f in n]
        got = M(planes, in_layout="nv12", out_layout="bgra", **kw)
        ref = M(n, in_layout="nv12", out_layout="hwc_bgr", **kw)
        assert got.shape == ref.shape[:3] + (4,) and torch.equal(got[..., :3], ref) and bool((got[..., 3] == 255).all())
        f = natural_p010(B, H, W, seed=c["xseed"] + 6, yuv="bt2020").to(DEV)
        got = M(f, in_layout="p010", out_layout="rgba", yuv="bt2020", **kw)
        ref = M(f, in_layout="p010", out_layout="hwc", yuv="bt2020", **kw)
        assert got.dtype == U8 and torch.equal(got[..., :3], ref) and bool((got[..., 3] == 255).all())
        x4 = frames4(B, H, W, seed=c["xseed"] + 7).to(DEV)
        x3 = x4[..., :3].contiguous()
        assert torch.equal(M(x4, in_layout="rgba", out_layout="nv12", **kw), M(x3, in_layout="hwc", out_layout="nv12", **kw))
        got = M(x4, in_layout="bgra", out_layout="p010", yuv="bt2020_full", **kw)
        assert got.dtype == U16 and torch.equal(got, M(x3, in_layout="hwc_bgr", out_layout="p010", yuv="bt2020_full", **kw))
        assert torch.equal(M(x4, in_layout="rgba", **kw), M(x3, in_layout="hwc", **kw))


@pytest.mark.parametrize("name", ["window_720p_1080p_b8", "residual_720p_4k"])
def test_fullsize_bgra_to_bgra(name):
    c = FULLSIZE[name]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    x4 = frames4(B, H, W, seed=c["xseed"])
    xd = x4.to(DEV)
    with torch.no_grad():
        got = _run(M, xd, c["kw"], True, in_layout="bgra", out_layout="bgra")
        ref = _run(M, xd[..., :3].contiguous(), c["kw"], True, in_layout="hwc_bgr", out_layout="hwc_bgr")
    oh, ow = c["kw"]["res_out"]
    assert got.shape == (B, oh, ow, 4) and torch.equal(got[..., :3], ref)
    del ref
    assert torch.equal(got[..., 3].cpu(), oracle_alpha(x4, oh, ow))


def test_rejections():
    M = _model("window_72x104_r1p5")
    with torch.no_grad():
        with pytest.raises(ValueError):                                     # a 3-byte frame given as RGBA
            M(torch.zeros(1, 72, 104, 3, dtype=U8, device=DEV), in_layout="rgba", res_out=(108, 156))
        with pytest.raises(ValueError):                                     # layouts on float input
            M(torch.zeros(1, 3, 72, 104, device=DEV), out_layout="bgra", res_out=(108, 156))
        with pytest.raises(ValueError):
            M(torch.zeros(1, 72, 104, 4, device=DEV), in_layout="rgba", res_out=(108, 156))


# ---------------------------------------------------------------------------------------------------------------------------------
# wrappers
def test_rgba_graphed_model_frame_pipeline_and_compile():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M = _model("window_72x104_r1p5")
    kw = dict(res_out=(108, 156), in_layout="bgra", out_layout="bgra")
    xs = [frames4(2, 72, 104, seed=700 + i) for i in range(5)]
    with torch.no_grad():
        eager = [M(x.to(DEV), **kw).clone() for x in xs]
    assert eager[0].shape == (2, 108, 156, 4) and eager[0].dtype == U8
    assert torch.equal(eager[0][..., 3].cpu(), oracle_alpha(xs[0], 108, 156))
    G = GraphedModel(M)
    for x, e in zip(xs, eager):
        assert torch.equal(G(x.to(DEV), **kw), e)
    hin = [x.pin_memory() for x in xs]
    hout = [torch.zeros((2, 108, 156, 4), dtype=U8).pin_memory() for _ in xs]
    assert all(t.is_pinned() for t in hin + hout)
    pipe = FramePipeline(M, depth=3, device=DEV, compute_streams=2, **kw)
    for a, b in zip(hin, hout):
        pipe.submit(a, b)
    pipe.drain()
    for b, e in zip(hout, eager):
        assert torch.equal(b, e.cpu())
    # torch.compile traces tu::forward, tu::resample_alpha and tu::resize_aa through their fake kernels
    Mf = _model("fast_40x56_res60x84")
    x4 = frames4(1, 40, 56, seed=3).to(DEV)
    with torch.no_grad():
        assert torch.equal(torch.compile(M)(xs[0].to(DEV), **kw), eager[0])
        want = Mf(x4, in_layout="rgba", out_layout="rgba", res_out=(60, 84))
        got = torch.compile(Mf)(x4, in_layout="rgba", out_layout="rgba", res_out=(60, 84))
        assert got.shape == (1, 60, 84, 4) and torch.equal(got, want)
        assert torch.equal(got[..., 3].cpu(), oracle_alpha(x4.cpu(), 60, 84))
