"""GPU: NV12 video frames at both ends of the forward (tu_nv12_to_rgb / tu_rgb_to_nv12, csrc/resample.cu).

Every comparison is bitwise.  The conversion kernels equal the fp32 oracle of tests/test_nv12_host.py; a forward with an NV12 side
equals the composition of that oracle with the fp16 image path: NV12 in = the forward of oracle_nv12_to_rgb(x).half(), NV12 out =
oracle_rgb_to_nv12 of the fp16 output."""
import ctypes as C

import pytest
import torch

from oracle.weights import synth_frames
from tests.golden.cases import CASES, FULLSIZE
from tests.test_gpu_models import build
from tests.test_nv12_host import COLOURS, flat_chroma_frames, oracle_nv12_to_rgb, oracle_rgb_to_nv12

pytestmark = pytest.mark.gpu

F32, F16, U8 = torch.float32, torch.float16, torch.uint8
DEV = torch.device("cuda:0")


def _lib():
    from transformerupscaler_b200 import _lib
    return _lib, _lib.load()


def nv12_code(yuv):
    from transformerupscaler_b200 import _lib, engine
    return _lib.TU_U8 | _lib.TU_LAYOUT_NV12 | engine.yuv_code(yuv)


def k_nv12_to_rgb(f, yuv):
    _l, lib = _lib()
    B, R, W = f.shape
    H = R * 2 // 3
    out = torch.empty(B, 3, H, W, dtype=F16, device=f.device)
    _l.check(lib.tu_nv12_to_rgb(f.data_ptr(), nv12_code(yuv), out.data_ptr(), B, H, W, torch.cuda.current_stream().cuda_stream))
    return out


def k_rgb_to_nv12(x, yuv):
    _l, lib = _lib()
    B, _, H, W = x.shape
    out = torch.empty(B, 3 * H // 2, W, dtype=U8, device=x.device)
    _l.check(lib.tu_rgb_to_nv12(x.data_ptr(), out.data_ptr(), nv12_code(yuv), B, H, W, torch.cuda.current_stream().cuda_stream))
    return out


def random_nv12(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (B, 3 * H // 2, W), generator=g, dtype=U8)


def natural_nv12(B, H, W, seed, yuv="bt709"):
    """NV12 frames of smooth synthetic content (what a decoder hands out), made with the oracle"""
    return oracle_rgb_to_nv12(synth_frames(B, H, W, seed=seed).half(), yuv)


SIZES = [(H, W) for H in (2, 720) for W in (2, 6, 10, 1280)]


# ---------------------------------------------------------------------------------------------------------------------------------
# the conversion kernels
@pytest.mark.parametrize("yuv", COLOURS)
@pytest.mark.parametrize("hw", SIZES)
def test_nv12_to_rgb_kernel_matches_oracle(yuv, hw):
    H, W = hw
    f = random_nv12(3, H, W, seed=H * 7 + W)                              # every code, illegal ones included
    got = k_nv12_to_rgb(f.to(DEV), yuv).cpu()
    assert torch.equal(got, oracle_nv12_to_rgb(f, yuv).half())


@pytest.mark.parametrize("yuv", COLOURS)
def test_nv12_to_rgb_kernel_every_yuv_triple(yuv):
    f = flat_chroma_frames()                                              # 65536 frames 16 x 16: every (Y, U, V)
    for part in f.split(32768):                                           # a launch takes up to 65535 frames
        got = k_nv12_to_rgb(part.to(DEV), yuv).cpu()
        assert torch.equal(got, oracle_nv12_to_rgb(part, yuv).half())


@pytest.mark.parametrize("yuv", COLOURS)
@pytest.mark.parametrize("hw", SIZES)
def test_rgb_to_nv12_kernel_matches_oracle(yuv, hw):
    H, W = hw
    g = torch.Generator().manual_seed(H * 11 + W)
    x = (torch.rand(3, 3, H, W, generator=g) * 1.6 - 0.3).half()           # values outside [0, 1] too
    got = k_rgb_to_nv12(x.to(DEV), yuv).cpu()
    assert torch.equal(got, oracle_rgb_to_nv12(x, yuv))


# ---------------------------------------------------------------------------------------------------------------------------------
# whole forward
def _even(name):
    _, _, H, W = CASES[name]["shape"]
    return H % 2 == 0 and W % 2 == 0


def _run(M, x, kw, bf16, out_dtype, clamp=True, **lk):
    from transformerupscaler_b200 import engine
    h = M._packed(bf16, x.device)
    return engine.run_forward(h, M.ENGINE_MODEL, x, kw.get("res_out", (1080, 1920)), kw.get("upscale_factor"),
                              kw.get("require_ratio", True), bf16, out_dtype, clamp=clamp, **lk)


_models = {}


def _model(name):
    c = CASES[name]
    key = (c["model"], c["wseed"], c.get("gain", 1.0))
    if key not in _models:
        _models[key] = build(c["model"], c["wseed"], c.get("gain", 1.0))[0]
    return _models[key]


@pytest.mark.parametrize("name", [n for n in CASES if _even(n)])
@pytest.mark.parametrize("path", ["bf16", "fp32"])
@pytest.mark.parametrize("yuv", ["bt709", "bt601_full"])
def test_forward_nv12_input_is_the_fp16_forward_of_the_converted_frame(name, path, yuv):
    c = CASES[name]
    B, _, H, W = c["shape"]
    M = _model(name)
    bf16 = path == "bf16"
    f = natural_nv12(B, H, W, seed=c["xseed"], yuv=yuv).to(DEV)
    rgb = oracle_nv12_to_rgb(f, yuv).half().to(DEV)
    with torch.no_grad():
        for clamp in (False, True):
            for D in (F32, F16, U8):
                got = _run(M, f, c["kw"], bf16, D, clamp, in_layout="nv12", yuv=yuv)
                want = _run(M, rgb, c["kw"], bf16, D, clamp)
                assert got.dtype == D and torch.equal(got, want), (clamp, D)


OUT_CASES = ["window_72x104_r1p5", "window_64x80_x2", "residual_720p_1080p", "fast_40x56_x2", "fast_40x56_x3", "fast_40x56_x4",
             "fast_24x32_x6", "fast_40x56_res60x84"]


@pytest.mark.parametrize("name", OUT_CASES)
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forward_nv12_output_is_the_converted_fp16_output(name, path):
    c = CASES[name]
    B, _, H, W = c["shape"]
    M = _model(name)
    bf16 = path == "bf16"
    x = synth_frames(B, H, W, seed=c["xseed"]).to(DEV)
    with torch.no_grad():
        for yuv in ("bt709", "bt601_full"):
            for clamp in (False, True):
                got = _run(M, x, c["kw"], bf16, U8, clamp, out_layout="nv12", yuv=yuv)
                want = oracle_rgb_to_nv12(_run(M, x, c["kw"], bf16, F16, clamp), yuv)
                assert got.dtype == U8 and torch.equal(got.cpu(), want), (yuv, clamp)


@pytest.mark.parametrize("name", ["window_72x104_r1p5", "fast_36x52_x2_reflect", "fast_40x56_res60x84", "residual_720p_1080p"])
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forward_nv12_to_nv12_and_to_hwc_bgr(name, path):
    c = CASES[name]
    B, _, H, W = c["shape"]
    M = _model(name)
    M.engine_precision = path
    try:
        bf16 = path == "bf16"
        f = natural_nv12(B, H, W, seed=c["xseed"] + 1, yuv="bt601").to(DEV)
        rgb = oracle_nv12_to_rgb(f, "bt601").half().to(DEV)
        with torch.no_grad():
            got = M(f, in_layout="nv12", out_layout="nv12", yuv="bt601", **c["kw"])
            assert got.dtype == U8
            assert torch.equal(got.cpu(), oracle_rgb_to_nv12(_run(M, rgb, c["kw"], bf16, F16), "bt601"))
            bgr = M(f, in_layout="nv12", out_layout="hwc_bgr", yuv="bt601", **c["kw"])
            assert torch.equal(bgr, _run(M, rgb, c["kw"], bf16, U8, out_layout="hwc_bgr"))
            planar = M(f, in_layout="nv12", yuv="bt601", **c["kw"])          # NV12 in, uint8 CHW out
            assert planar.dtype == U8 and torch.equal(planar, _run(M, rgb, c["kw"], bf16, U8))
    finally:
        M.engine_precision = None


@pytest.mark.parametrize("name", ["window_720p_1080p_b8", "residual_720p_4k"])
def test_fullsize_nv12_to_nv12_bf16(name):
    """the row-schedule bicubic kernel on fp16 frames at the BASELINE sizes"""
    c = FULLSIZE[name]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    f = natural_nv12(B, H, W, seed=c["xseed"]).to(DEV)
    with torch.no_grad():
        got = _run(M, f, c["kw"], True, U8, in_layout="nv12", out_layout="nv12").cpu()
        mid = _run(M, oracle_nv12_to_rgb(f).half().to(DEV), c["kw"], True, F16)
    want = oracle_rgb_to_nv12(mid)
    del mid
    torch.cuda.empty_cache()
    oh, ow = c["kw"]["res_out"]
    assert got.shape == (B, 3 * oh // 2, ow) and torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------------------------------------
# rejections
def test_nv12_rejections():
    from transformerupscaler_b200 import _lib as L
    lib = L.load()
    c = CASES["window_131x189_odd"]
    M = _model("window_131x189_odd")
    with torch.no_grad():
        with pytest.raises(ValueError):                                   # (1, 196, 189): not a (B, 3H/2, W) buffer, odd W
            M(torch.zeros(1, 196, 189, dtype=U8, device=DEV), in_layout="nv12", **c["kw"])
        with pytest.raises(ValueError):                                   # 3H/2 rows, but H = 130 rows with an odd W
            M(torch.zeros(1, 195, 189, dtype=U8, device=DEV), in_layout="nv12", **c["kw"])
        f = natural_nv12(1, 72, 104, seed=1).to(DEV)
        M72 = _model("window_72x104_r1p5")
        with pytest.raises(ValueError):
            M72(f, in_layout="nv12", out_layout="nv12", res_out=(108, 157))
        with pytest.raises(ValueError):
            M72(f, in_layout="nv12", out_layout="nv12", res_out=(109, 156))
        with pytest.raises(ValueError):                                   # a colour without an NV12 side
            M72(torch.zeros(1, 3, 72, 104, dtype=U8, device=DEV), res_out=(108, 156), yuv="bt601")
        with pytest.raises(ValueError):
            M72(f, in_layout="nv12", yuv="bt2020")
        with pytest.raises(ValueError):                                   # NV12 is a uint8 frame layout
            M72(torch.zeros(1, 3, 72, 104, device=DEV), out_layout="nv12", res_out=(108, 156))
    # the C ABI
    h = M72._packed(True, DEV)
    from transformerupscaler_b200 import engine
    pw = engine._REGISTRY[h]
    w = C.byref(pw.struct)
    out = torch.empty(1, 162, 156, dtype=U8, device=DEV)
    nv12 = L.TU_U8 | L.TU_LAYOUT_NV12
    st = torch.cuda.current_stream().cuda_stream
    need = lib.tu_forward_workspace_bytes_io(w, 1, 72, 104, 108, 156, 0, L.TU_BF16, nv12, nv12)
    old = lib.tu_forward_workspace_bytes_for(w, 1, 72, 104, 108, 156, 0, L.TU_BF16)
    assert need > old > 0
    ws = torch.empty(need, dtype=U8, device=DEV)
    xf = torch.zeros(1, 3, 72, 104, device=DEV)
    assert lib.tu_forward(w, xf.data_ptr(), L.TU_F32 | L.TU_LAYOUT_NV12, out.data_ptr(), nv12, 1, 72, 104, 108, 156, 0, L.TU_BF16, 1,
                          ws.data_ptr(), need, st) == L.TU_ERR_ARG                     # NV12 bit on a float base
    assert lib.tu_forward(w, f.data_ptr(), nv12, out.data_ptr(), L.TU_F32 | L.TU_LAYOUT_NV12, 1, 72, 104, 108, 156, 0, L.TU_BF16, 1,
                          ws.data_ptr(), need, st) == L.TU_ERR_ARG
    assert lib.tu_forward(w, f.data_ptr(), L.TU_U8 | L.TU_YUV_BT601, out.data_ptr(), nv12, 1, 72, 104, 108, 156, 0, L.TU_BF16, 1,
                          ws.data_ptr(), need, st) == L.TU_ERR_ARG                     # colour bits without NV12
    assert lib.tu_forward(w, f.data_ptr(), nv12, out.data_ptr(), L.TU_U8 | L.TU_LAYOUT_HWC | L.TU_YUV_FULL_RANGE, 1, 72, 104, 108, 156, 0,
                          L.TU_BF16, 1, ws.data_ptr(), need, st) == L.TU_ERR_ARG
    assert lib.tu_forward(w, f.data_ptr(), nv12, out.data_ptr(), nv12, 1, 72, 104, 108, 156, 0, L.TU_BF16, 1,
                          ws.data_ptr(), old, st) == L.TU_ERR_WORKSPACE                # sized by the old query
    assert lib.tu_forward(w, f.data_ptr(), nv12, out.data_ptr(), nv12, 1, 72, 104, 108, 156, 0, L.TU_BF16, 1,
                          ws.data_ptr(), need, st) == 0
    torch.cuda.synchronize()
    with torch.no_grad():
        assert torch.equal(out, _run(M72, f, dict(res_out=(108, 156)), True, U8, in_layout="nv12", out_layout="nv12"))


# ---------------------------------------------------------------------------------------------------------------------------------
# wrappers
def test_nv12_graphed_model_frame_pipeline_and_compile():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M = _model("window_72x104_r1p5")
    kw = dict(res_out=(108, 156), in_layout="nv12", out_layout="nv12", yuv="bt709_full")
    xs = [natural_nv12(2, 72, 104, seed=600 + i, yuv="bt709_full") for i in range(5)]
    with torch.no_grad():
        eager = [M(x.to(DEV), **kw).clone() for x in xs]
    assert eager[0].shape == (2, 162, 156) and eager[0].dtype == U8
    G = GraphedModel(M)
    for x, e in zip(xs, eager):
        assert torch.equal(G(x.to(DEV), **kw), e)
    hin = [x.pin_memory() for x in xs]
    hout = [torch.zeros((2, 162, 156), dtype=U8).pin_memory() for _ in xs]
    pipe = FramePipeline(M, depth=3, device=DEV, compute_streams=2, **kw)
    for a, b in zip(hin, hout):
        pipe.submit(a, b)
    pipe.drain()
    for b, e in zip(hout, eager):
        assert torch.equal(b, e.cpu())
    # torch.compile traces tu::forward through its fake kernel (NV12 output shape) and returns the eager result
    Mf = _model("fast_40x56_res60x84")
    f = natural_nv12(1, 40, 56, seed=3).to(DEV)
    with torch.no_grad():
        want = M(xs[0].to(DEV), **kw)
        got = torch.compile(M)(xs[0].to(DEV), **kw)
        assert torch.equal(got, want)
        want = Mf(f, in_layout="nv12", out_layout="nv12", res_out=(60, 84))          # Resize, then tu::rgb_to_nv12
        got = torch.compile(Mf)(f, in_layout="nv12", out_layout="nv12", res_out=(60, 84))
        assert got.shape == (1, 90, 84) and torch.equal(got, want)
