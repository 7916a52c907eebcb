"""GPU: P010 video frames at both ends of the forward (tu_p010_to_rgb / tu_rgb_to_p010, csrc/resample.cu).

Every comparison is bitwise.  The conversion kernels equal the fp32 oracle of tests/test_p010_host.py; a forward with a P010 side
equals the composition of that oracle with the fp32 image path: P010 in = the TU_F32-input forward of oracle_p010_to_rgb(x), P010
out = oracle_rgb_to_p010 of the fp32 output."""
import ctypes as C

import pytest
import torch

from oracle.weights import synth_frames
from tests.golden.cases import CASES, FULLSIZE
from tests.test_gpu_models import build
from tests.test_nv12_host import oracle_nv12_to_rgb, oracle_rgb_to_nv12
from tests.test_p010_host import (COLOURS10, chroma_lattice, flat_chroma_frames10, oracle_p010_to_rgb, oracle_rgb_to_p010,
                                  words_to_codes)

pytestmark = pytest.mark.gpu

F32, F16, U8, U16 = torch.float32, torch.float16, torch.uint8, torch.uint16
DEV = torch.device("cuda:0")


def _lib():
    from transformerupscaler_b200 import _lib
    return _lib, _lib.load()


def p010_code(yuv):
    from transformerupscaler_b200 import _lib, engine
    return _lib.TU_U16 | _lib.TU_LAYOUT_P010 | engine.yuv_code(yuv)


def k_p010_to_rgb(f, yuv):
    _l, lib = _lib()
    B, R, W = f.shape
    H = R * 2 // 3
    out = torch.empty(B, 3, H, W, dtype=F32, device=f.device)
    _l.check(lib.tu_p010_to_rgb(f.data_ptr(), p010_code(yuv), out.data_ptr(), B, H, W, torch.cuda.current_stream().cuda_stream))
    return out


def k_rgb_to_p010(x, yuv):
    _l, lib = _lib()
    B, _, H, W = x.shape
    out = torch.empty(B, 3 * H // 2, W, dtype=U16, device=x.device)
    _l.check(lib.tu_rgb_to_p010(x.data_ptr(), out.data_ptr(), p010_code(yuv), B, H, W, torch.cuda.current_stream().cuda_stream))
    return out


def random_p010(B, H, W, seed):
    """random 16-bit words: every 10-bit code, illegal ones included, with random low 6 bits"""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 65536, (B, 3 * H // 2, W), generator=g, dtype=torch.int32).to(U16)


def natural_p010(B, H, W, seed, yuv="bt709"):
    """P010 frames of smooth synthetic content (what a decoder hands out), made with the oracle"""
    return oracle_rgb_to_p010(synth_frames(B, H, W, seed=seed), yuv)


def natural_nv12(B, H, W, seed, yuv="bt709"):
    return oracle_rgb_to_nv12(synth_frames(B, H, W, seed=seed).half(), yuv)


def same_words(a, b):
    return a.dtype == U16 and b.dtype == U16 and a.shape == b.shape and torch.equal(a.cpu(), b.cpu())


SIZES = [(H, W) for H in (2, 720) for W in (2, 6, 10, 1280)]


# ---------------------------------------------------------------------------------------------------------------------------------
# the conversion kernels
@pytest.mark.parametrize("yuv", COLOURS10)
@pytest.mark.parametrize("hw", SIZES)
def test_p010_to_rgb_kernel_matches_oracle(yuv, hw):
    H, W = hw
    f = random_p010(3, H, W, seed=H * 7 + W)
    got = k_p010_to_rgb(f.to(DEV), yuv).cpu()
    assert torch.equal(got, oracle_p010_to_rgb(f, yuv))


@pytest.mark.parametrize("yuv", COLOURS10)
def test_p010_to_rgb_kernel_flat_chroma_lattice(yuv):
    f = flat_chroma_frames10()                                            # every Y code, the (U, V) lattice
    assert f.shape[0] == len(chroma_lattice())
    got = k_p010_to_rgb(f.to(DEV), yuv).cpu()
    assert torch.equal(got, oracle_p010_to_rgb(f, yuv))
    # low bits are ignored
    g = torch.Generator().manual_seed(1)
    dirty = (f.to(torch.int32) | torch.randint(0, 64, f.shape, generator=g, dtype=torch.int32)).to(U16)
    assert torch.equal(k_p010_to_rgb(dirty.to(DEV), yuv).cpu(), got)


@pytest.mark.parametrize("yuv", COLOURS10)
@pytest.mark.parametrize("hw", SIZES)
def test_rgb_to_p010_kernel_matches_oracle(yuv, hw):
    H, W = hw
    g = torch.Generator().manual_seed(H * 11 + W)
    x = torch.rand(3, 3, H, W, generator=g) * 1.6 - 0.3                   # values outside [0, 1] too
    got = k_rgb_to_p010(x.to(DEV), yuv).cpu()
    assert same_words(got, oracle_rgb_to_p010(x, yuv))
    assert int((got.to(torch.int32) & 63).max()) == 0


@pytest.mark.parametrize("yuv", COLOURS10)
def test_rgb_to_p010_kernel_round_trip_of_lattice(yuv):
    """the flat lattice frames back through the kernel: the result is the oracle's, bit for bit"""
    f = flat_chroma_frames10()
    rgb = oracle_p010_to_rgb(f, yuv)
    assert same_words(k_rgb_to_p010(rgb.to(DEV), yuv), oracle_rgb_to_p010(rgb, yuv))


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
@pytest.mark.parametrize("yuv", ["bt709", "bt2020_full"])
def test_forward_p010_input_is_the_fp32_forward_of_the_converted_frame(name, path, yuv):
    c = CASES[name]
    B, _, H, W = c["shape"]
    M = _model(name)
    bf16 = path == "bf16"
    f = natural_p010(B, H, W, seed=c["xseed"], yuv=yuv).to(DEV)
    rgb = oracle_p010_to_rgb(f, yuv).to(DEV)
    with torch.no_grad():
        for clamp in (False, True):
            for D in (F32, F16, U8):
                got = _run(M, f, c["kw"], bf16, D, clamp, in_layout="p010", yuv=yuv)
                want = _run(M, rgb, c["kw"], bf16, D, clamp)
                assert got.dtype == D and torch.equal(got, want), (clamp, D)


OUT_CASES = ["window_72x104_r1p5", "window_64x80_x2", "residual_720p_1080p", "fast_40x56_x2", "fast_40x56_x3", "fast_40x56_x4",
             "fast_24x32_x6", "fast_40x56_res60x84"]


@pytest.mark.parametrize("name", OUT_CASES)
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forward_p010_output_is_the_converted_fp32_output(name, path):
    c = CASES[name]
    B, _, H, W = c["shape"]
    M = _model(name)
    bf16 = path == "bf16"
    x = synth_frames(B, H, W, seed=c["xseed"]).to(DEV)
    with torch.no_grad():
        for yuv in ("bt709", "bt601_full", "bt2020"):
            for clamp in (False, True):
                got = _run(M, x, c["kw"], bf16, U16, clamp, out_layout="p010", yuv=yuv)
                want = oracle_rgb_to_p010(_run(M, x, c["kw"], bf16, F32, clamp), yuv)
                assert same_words(got, want), (yuv, clamp)


@pytest.mark.parametrize("name", ["window_72x104_r1p5", "fast_36x52_x2_reflect", "fast_40x56_res60x84", "residual_720p_1080p"])
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forward_mixed_sides(name, path):
    """P010 -> P010, P010 -> NV12, NV12 -> P010, uint8 CHW -> P010, P010 -> HWC BGR through the model's forward"""
    c = CASES[name]
    B, _, H, W = c["shape"]
    M = _model(name)
    M.engine_precision = path
    try:
        bf16 = path == "bf16"
        kw = c["kw"]
        with torch.no_grad():
            f = natural_p010(B, H, W, seed=c["xseed"] + 1, yuv="bt2020").to(DEV)
            rgb = oracle_p010_to_rgb(f, "bt2020").to(DEV)
            got = M(f, in_layout="p010", out_layout="p010", yuv="bt2020", **kw)
            assert same_words(got, oracle_rgb_to_p010(_run(M, rgb, kw, bf16, F32), "bt2020"))
            bgr = M(f, in_layout="p010", out_layout="hwc_bgr", yuv="bt2020", **kw)
            assert bgr.dtype == U8 and torch.equal(bgr, _run(M, rgb, kw, bf16, U8, out_layout="hwc_bgr"))
            planar = M(f, in_layout="p010", yuv="bt2020", **kw)               # P010 in, uint8 CHW out
            assert planar.dtype == U8 and torch.equal(planar, _run(M, rgb, kw, bf16, U8))

            f = natural_p010(B, H, W, seed=c["xseed"] + 2, yuv="bt601").to(DEV)
            rgb = oracle_p010_to_rgb(f, "bt601").to(DEV)
            got = M(f, in_layout="p010", out_layout="nv12", yuv="bt601", **kw)
            assert got.dtype == U8 and torch.equal(got.cpu(), oracle_rgb_to_nv12(_run(M, rgb, kw, bf16, F16), "bt601"))

            n = natural_nv12(B, H, W, seed=c["xseed"] + 3, yuv="bt709_full").to(DEV)
            rgb16 = oracle_nv12_to_rgb(n, "bt709_full").half().to(DEV)
            got = M(n, in_layout="nv12", out_layout="p010", yuv="bt709_full", **kw)
            assert same_words(got, oracle_rgb_to_p010(_run(M, rgb16, kw, bf16, F32), "bt709_full"))

            xu = (synth_frames(B, H, W, seed=c["xseed"]) * 255).round().to(U8).to(DEV)
            got = M(xu, out_layout="p010", **kw)
            assert same_words(got, oracle_rgb_to_p010(_run(M, xu, kw, bf16, F32)))
    finally:
        M.engine_precision = None


@pytest.mark.parametrize("name", ["window_720p_1080p_b8", "residual_720p_4k"])
def test_fullsize_p010_to_p010_bf16(name):
    """the row-schedule bicubic kernel on fp32 frames at the BASELINE sizes"""
    c = FULLSIZE[name]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    f = natural_p010(B, H, W, seed=c["xseed"], yuv="bt2020").to(DEV)
    with torch.no_grad():
        got = _run(M, f, c["kw"], True, U16, in_layout="p010", out_layout="p010", yuv="bt2020").cpu()
        mid = _run(M, oracle_p010_to_rgb(f, "bt2020").to(DEV), c["kw"], True, F32)
    want = oracle_rgb_to_p010(mid, "bt2020")
    del mid
    torch.cuda.empty_cache()
    oh, ow = c["kw"]["res_out"]
    assert got.shape == (B, 3 * oh // 2, ow) and same_words(got, want)


# ---------------------------------------------------------------------------------------------------------------------------------
# rejections
def test_p010_rejections():
    from transformerupscaler_b200 import _lib as L
    lib = L.load()
    c = CASES["window_131x189_odd"]
    M = _model("window_131x189_odd")
    M72 = _model("window_72x104_r1p5")
    f = natural_p010(1, 72, 104, seed=1).to(DEV)
    with torch.no_grad():
        with pytest.raises(ValueError):                                   # (1, 196, 189): not a (B, 3H/2, W) buffer, odd W
            M(torch.zeros(1, 196, 189, dtype=U16, device=DEV), in_layout="p010", **c["kw"])
        with pytest.raises(ValueError):                                   # 3H/2 rows, but an odd W
            M(torch.zeros(1, 195, 189, dtype=U16, device=DEV), in_layout="p010", **c["kw"])
        with pytest.raises(ValueError):                                   # (B, 3, H, W) is not a P010 buffer
            M72(torch.zeros(1, 3, 72, 104, dtype=U16, device=DEV), in_layout="p010", res_out=(108, 156))
        with pytest.raises(ValueError):                                   # P010 frames are uint16
            M72(torch.zeros(1, 108, 104, dtype=U8, device=DEV), in_layout="p010", res_out=(108, 156))
        with pytest.raises(ValueError):                                   # odd output sizes
            M72(f, in_layout="p010", out_layout="p010", res_out=(108, 157))
        with pytest.raises(ValueError):
            M72(f, in_layout="p010", out_layout="p010", res_out=(109, 156))
        with pytest.raises(ValueError):                                   # P010 output of a float input
            M72(torch.zeros(1, 3, 72, 104, device=DEV), out_layout="p010", res_out=(108, 156))
        with pytest.raises(ValueError):                                   # BT.2020 with an NV12 side
            M72(f, in_layout="p010", out_layout="nv12", yuv="bt2020", res_out=(108, 156))
        with pytest.raises(ValueError):                                   # BT.2020 without a P010 side
            M72(torch.zeros(1, 3, 72, 104, dtype=U8, device=DEV), res_out=(108, 156), yuv="bt2020_full")
        with pytest.raises(ValueError):
            M72(torch.zeros(1, 108, 104, dtype=U8, device=DEV), in_layout="nv12", out_layout="hwc", yuv="bt2020")
        # a uint16 tensor without in_layout='p010' is read as float32, as before
        x16 = torch.randint(0, 2, (1, 3, 72, 104), dtype=torch.int32).to(U16).to(DEV)
        y = M72(x16, res_out=(108, 156))
        assert y.dtype == F32 and torch.equal(y, M72(x16.float(), res_out=(108, 156)))
    # the C ABI
    h = M72._packed(True, DEV)
    from transformerupscaler_b200 import engine
    pw = engine._REGISTRY[h]
    w = C.byref(pw.struct)
    out = torch.empty(1, 162, 156, dtype=U16, device=DEV)
    p010 = L.TU_U16 | L.TU_LAYOUT_P010
    st = torch.cuda.current_stream().cuda_stream
    need = lib.tu_forward_workspace_bytes_io(w, 1, 72, 104, 108, 156, 0, L.TU_BF16, p010, p010)
    old = lib.tu_forward_workspace_bytes_for(w, 1, 72, 104, 108, 156, 0, L.TU_BF16)
    assert need > old > 0
    ws = torch.empty(need, dtype=U8, device=DEV)

    def fwd(i, o, cdt=L.TU_BF16, nbytes=need):
        return lib.tu_forward(w, f.data_ptr(), i, out.data_ptr(), o, 1, 72, 104, 108, 156, 0, cdt, 1, ws.data_ptr(), nbytes, st)
    assert fwd(L.TU_U16, p010) == L.TU_ERR_ARG                                        # bare TU_U16
    assert fwd(p010, L.TU_U16) == L.TU_ERR_ARG
    assert fwd(p010, p010, cdt=L.TU_U16) == L.TU_ERR_ARG                              # never a compute dtype
    assert fwd(p010 | L.TU_YUV_BT2020 | L.TU_YUV_BT601, p010) == L.TU_ERR_ARG
    assert fwd(L.TU_U8 | L.TU_LAYOUT_P010, p010) == L.TU_ERR_ARG
    assert fwd(p010, L.TU_U8 | L.TU_LAYOUT_NV12 | L.TU_YUV_BT2020) == L.TU_ERR_ARG     # BT.2020 on the NV12 side
    assert fwd(p010, p010, nbytes=old) == L.TU_ERR_WORKSPACE                          # sized by the old query
    assert fwd(p010, p010) == 0
    torch.cuda.synchronize()
    with torch.no_grad():
        assert same_words(out, _run(M72, f, dict(res_out=(108, 156)), True, U16, in_layout="p010", out_layout="p010"))
    # BT.2020 through the NV12 ops
    rgb = torch.zeros(1, 3, 4, 4, dtype=F16, device=DEV)
    nv = torch.zeros(1, 6, 4, dtype=U8, device=DEV)
    nv12 = L.TU_U8 | L.TU_LAYOUT_NV12
    assert lib.tu_rgb_to_nv12(rgb.data_ptr(), nv.data_ptr(), nv12 | L.TU_YUV_BT2020, 1, 4, 4, st) == L.TU_ERR_ARG
    assert lib.tu_nv12_to_rgb(nv.data_ptr(), nv12 | L.TU_YUV_BT2020, rgb.data_ptr(), 1, 4, 4, st) == L.TU_ERR_ARG


# ---------------------------------------------------------------------------------------------------------------------------------
# wrappers
def test_p010_graphed_model_frame_pipeline_and_compile():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M = _model("window_72x104_r1p5")
    kw = dict(res_out=(108, 156), in_layout="p010", out_layout="p010", yuv="bt2020_full")
    xs = [natural_p010(2, 72, 104, seed=600 + i, yuv="bt2020_full") for i in range(5)]
    with torch.no_grad():
        eager = [M(x.to(DEV), **kw).clone() for x in xs]
    assert eager[0].shape == (2, 162, 156) and eager[0].dtype == U16
    G = GraphedModel(M)
    for x, e in zip(xs, eager):
        assert same_words(G(x.to(DEV), **kw), e)
    hin = [x.pin_memory() for x in xs]
    hout = [torch.zeros((2, 162, 156), dtype=U16).pin_memory() for _ in xs]
    assert all(t.is_pinned() and t.dtype == U16 for t in hin + hout)
    pipe = FramePipeline(M, depth=3, device=DEV, compute_streams=2, **kw)
    for a, b in zip(hin, hout):
        pipe.submit(a, b)
    pipe.drain()
    for b, e in zip(hout, eager):
        assert same_words(b, e)
    # torch.compile traces tu::forward through its fake kernel (P010 output shape) and returns the eager result
    Mf = _model("fast_40x56_res60x84")
    f = natural_p010(1, 40, 56, seed=3).to(DEV)
    with torch.no_grad():
        want = M(xs[0].to(DEV), **kw)
        got = torch.compile(M)(xs[0].to(DEV), **kw)
        assert same_words(got, want)
        want = Mf(f, in_layout="p010", out_layout="p010", res_out=(60, 84))          # Resize, then tu::rgb_to_p010
        got = torch.compile(Mf)(f, in_layout="p010", out_layout="p010", res_out=(60, 84))
        assert got.shape == (1, 90, 84) and same_words(got, want)
        assert torch.equal(words_to_codes(want) << 6, want.cpu().to(torch.int32))     # low bits zero
