"""GPU: float16 models and frames (fp16 image I/O on the bf16 tensor-core path).

The property everything here checks: for any module and input, the fp16 output equals, bit for bit, y.half(), where y is the fp32
output the same compute path returns for x.float() with fp32 parameters of the same values -- with and without the clamp.  fp16 ->
fp32 is exact and round-to-nearest commutes with the clamp to [0, 1], so no new tolerance is needed."""
import copy
import os

import numpy as np
import pytest
import torch

from oracle.weights import synth_state_dict, synth_frames
from tests.golden.cases import CASES, FULLSIZE, sample_fullsize
from tests.test_gpu_models import GOLD, TOL_BF16, bf16_pre_clamp_err, build, engine_pre_clamp, psnr

pytestmark = pytest.mark.gpu

F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16


@pytest.fixture(autouse=True)
def helpers_know_f16(monkeypatch):
    """tests/gpu_helpers.py maps torch dtypes to the library's codes; add fp16 for the calls of this module"""
    from tests import gpu_helpers as G
    from transformerupscaler_b200 import _lib
    _lib.load()
    monkeypatch.setitem(G.DT, F16, _lib.TU_F16)
    return G


def _pair(name):
    """(M16, M32, x16, kw): the case's module in fp16, the same values in an fp32 module, an fp16 input"""
    c = CASES[name]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"], c.get("gain", 1.0))
    M16 = copy.deepcopy(M).half()
    M32 = copy.deepcopy(M16).float()
    x16 = synth_frames(B, H, W, seed=c["xseed"]).half().cuda()
    return M16, M32, x16, c["kw"]


# ---------------------------------------------------------------------------------------------------------------------------------
# whole model
@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_fp16_module_is_the_rounded_fp32_result(name, path):
    M16, M32, x16, kw = _pair(name)
    M32.engine_precision = path
    if path == "fp32":
        M16.engine_precision = "fp32"
    with torch.no_grad():
        y16 = M16(x16, **kw)
        y32 = M32(x16.float(), **kw)
    assert y16.dtype == F16 and y32.dtype == F32
    assert torch.equal(y16, y32.half())
    bf16 = path == "bf16"
    pre16 = engine_pre_clamp(M16, x16, kw, bf16, out_dtype=F16)
    pre32 = engine_pre_clamp(M32, x16.float(), kw, bf16)
    assert pre16.dtype == F16
    assert torch.equal(pre16, pre32.half())


@pytest.mark.parametrize("name", list(CASES))
def test_fp16_module_within_bf16_bars_of_reference(name):
    c = CASES[name]
    M16, _, x16, kw = _pair(name)
    g = np.load(os.path.join(GOLD, name + ".npz"))
    st = c.get("stride", 1)
    with torch.no_grad():
        out = M16(x16, **kw)
    o = out.float().cpu()[..., ::st, ::st]
    ref = torch.from_numpy(np.clip(g["pre"], 0, 1))
    assert (o - ref).abs().max().item() < TOL_BF16
    assert psnr(o, ref) > 50.0
    pre = engine_pre_clamp(M16, x16, kw, True, out_dtype=F16).float().cpu().numpy()[..., ::st, ::st]
    assert bf16_pre_clamp_err(pre, g["pre"]) < TOL_BF16


def test_fp16_window_720p_1080p_b8_fullsize():
    name = "window_720p_1080p_b8"
    c = FULLSIZE[name]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    M16 = M.half()
    x16 = synth_frames(B, H, W, seed=c["xseed"]).half().cuda()
    g = np.load(os.path.join(GOLD, name + ".npz"))
    pre = engine_pre_clamp(M16, x16, c["kw"], True, out_dtype=F16)
    lat, crops = sample_fullsize(pre.float().cpu().numpy(), c)
    del pre
    with torch.no_grad():
        out = M16(x16, **c["kw"])
    assert out.dtype == F16
    olat, ocrops = sample_fullsize(out.float().cpu().numpy(), c)
    del out
    torch.cuda.empty_cache()
    err = max([bf16_pre_clamp_err(lat, g["pre"])] + [bf16_pre_clamp_err(cr, g[f"crop{i}"]) for i, cr in enumerate(crops)])
    assert err < TOL_BF16, err
    ref = np.clip(g["pre"], 0, 1)
    errc = max([np.abs(olat - ref).max()] + [np.abs(cr - np.clip(g[f"crop{i}"], 0, 1)).max() for i, cr in enumerate(ocrops)])
    assert errc < TOL_BF16, errc
    assert psnr(torch.from_numpy(olat), torch.from_numpy(ref)) > 50.0


@pytest.mark.parametrize("name", ["natural_window_96x176_r1p5", "natural_fast_96x176_x2"])
def test_fp16_natural_image_psnr_delta(name):
    from tests.golden.cases import NATURAL
    c = NATURAL[name]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    M, _ = build(c["model"], c["wseed"])
    hr = torch.from_numpy(g["hr_u8"]).float() / 255.0
    ref = torch.from_numpy(g["ref"].astype(np.float32))
    x16 = (torch.from_numpy(g["lr_u8"]).unsqueeze(0).float() / 255.0).half().cuda()
    with torch.no_grad():
        o = M.half()(x16, **c["kw"])[0].float().cpu()
    assert (o - ref).abs().max().item() < TOL_BF16
    assert abs(psnr(o, hr) - psnr(ref, hr)) <= 0.05, f"{name}: PSNR delta {psnr(o, hr) - psnr(ref, hr):+.4f} dB"


@pytest.mark.parametrize("name", ["window_72x104_r1p5", "window_131x189_odd", "fast_36x52_x2_reflect", "fast_40x56_res60x84",
                                  "residual_720p_1080p"])
def test_fp16_input_to_fp32_and_bf16_modules_is_unchanged(name):
    """fp16 frames now reach the library as they are; fp32 and bf16 modules return bitwise what they return for x.float(), in their
    own dtype (W = 52: the fp16 frame is widened before the fused conv1+conv2 kernel, like the fp32 frame takes it)"""
    _, M32, x16, kw = _pair(name)
    Mb = copy.deepcopy(M32).bfloat16()
    with torch.no_grad():
        for M, ac in ((M32, None), (M32, BF16), (Mb, None)):
            with torch.autocast("cuda", dtype=ac or BF16, enabled=ac is not None):
                a = M(x16, **kw)
                b = M(x16.float(), **kw)
            assert a.dtype == b.dtype and torch.equal(a, b), (ac, a.dtype)


# ---------------------------------------------------------------------------------------------------------------------------------
# dtype rules
@pytest.mark.parametrize("name", ["window_72x104_r1p5", "fast_40x56_x2", "residual_720p_1080p"])
def test_fp16_module_dtype_rules(name):
    """fp16 out without autocast and under autocast(float16); under autocast(bfloat16) Window / Residual still return fp16 (their
    reference output follows the parameters) and FastTransformer returns the autocast dtype, as it does for every module dtype"""
    M16, M32, x16, kw = _pair(name)
    fast = CASES[name]["model"] == "FastTransformer"
    with torch.no_grad():
        y = M16(x16, **kw)
        with torch.autocast("cuda", dtype=F16):
            ya = M16(x16, **kw)
        with torch.autocast("cuda", dtype=BF16):
            yb = M16(x16, **kw)
    assert y.dtype == F16 and ya.dtype == F16 and torch.equal(ya, y)
    if fast:
        assert yb.dtype == BF16 and torch.equal(yb, y.to(BF16))
    else:
        assert yb.dtype == F16 and torch.equal(yb, y)
    # uint8 frames into an fp16 module: uint8 frames out, the bf16 path's bytes
    c = CASES[name]
    B, _, H, W = c["shape"]
    xu = torch.randint(0, 256, (B, 3, H, W), generator=torch.Generator().manual_seed(5), dtype=torch.uint8).cuda()
    M32.engine_precision = "bf16"
    with torch.no_grad():
        yu = M16(xu, **kw)
        wu = M32(xu, **kw)
    assert yu.dtype == torch.uint8 and torch.equal(yu, wu)


def test_fp16_graphed_model_and_frame_pipeline():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M16, _, _, _ = _pair("window_72x104_r1p5")
    kw = dict(res_out=(108, 156))
    xs = [synth_frames(2, 72, 104, seed=500 + i).half() for i in range(5)]
    with torch.no_grad():
        eager = [M16(x.cuda(), **kw).clone() for x in xs]
    G = GraphedModel(M16)
    for x, e in zip(xs, eager):
        assert torch.equal(G(x.cuda(), **kw), e)
    hin = [x.pin_memory() for x in xs]
    hout = [torch.zeros((2, 3, 108, 156), dtype=F16).pin_memory() for _ in xs]
    pipe = FramePipeline(M16, depth=3, device=torch.device("cuda:0"), compute_streams=2, **kw)
    for a, b in zip(hin, hout):
        pipe.submit(a, b)
    pipe.drain()
    for b, e in zip(hout, eager):
        assert torch.equal(b, e.cpu())


# ---------------------------------------------------------------------------------------------------------------------------------
# single ops, bitwise against the fp32-I/O call on the same values
def _stem_weights(dev):
    sd = synth_state_dict("WindowTransformer", 0)
    w = sd["conv1.weight"].permute(2, 3, 1, 0).reshape(27, 64).contiguous().to(dev)
    w64 = torch.zeros(64, 64)
    w64[:, :27] = sd["conv1.weight"].permute(0, 2, 3, 1).reshape(64, 27)
    return sd, w, w64.to(dev, BF16), sd["conv1.bias"].to(dev)


@pytest.mark.parametrize("dt", [F32, BF16])
@pytest.mark.parametrize("shape", [(2, 37, 56), (1, 5, 300), (2, 19, 52), (1, 8, 1280)])
def test_stem_conv_fp16_input(helpers_know_f16, dt, shape):
    G = helpers_know_f16
    dev = torch.device("cuda:0")
    _, w, w64, b = _stem_weights(dev)
    x16 = synth_frames(*shape, seed=1).half().to(dev)
    for wt in ((None, w64) if dt == BF16 else (None,)):          # CUDA-core stem, tensor-core stem
        assert torch.equal(G.stem_conv(x16, w, b, dt, w64=wt), G.stem_conv(x16.float(), w, b, dt, w64=wt))


@pytest.mark.parametrize("shape", [(2, 19, 48), (1, 5, 304), (1, 70, 136), (3, 33, 256), (1, 8, 1280)])
def test_conv12_fused_fp16_input(helpers_know_f16, shape):
    G = helpers_know_f16
    dev = torch.device("cuda:0")
    sd = synth_state_dict("WindowTransformer", 2)
    w1, b1, w2, b2 = sd["conv1.weight"], sd["conv1.bias"], sd["conv2.weight"], sd["conv2.bias"]
    w64 = torch.zeros(64, 64)
    w64[:, :27] = w1.permute(0, 2, 3, 1).reshape(64, 27)
    w2p = w2.permute(2, 3, 0, 1).reshape(9, 64, 64).contiguous().to(dev, BF16)
    x16 = synth_frames(*shape, seed=21).half().to(dev)
    args = (w64.to(dev, BF16), b1.to(dev), w2p, b2.to(dev))
    assert torch.equal(G.conv12_fused(x16, *args), G.conv12_fused(x16.float(), *args))


BICUBIC_GEOMS = [((720, 1280), (360, 640), (1080, 1920)),      # x1.5, residual x3 (row schedule 0)
                 ((24, 48), (12, 24), (48, 96)), ((24, 48), (12, 24), (72, 144)), ((24, 48), (12, 24), (96, 192)),
                 ((8, 48), (4, 24), (48, 288)),                # x2 / x3 / x4 / x6, residual at twice the factor
                 ((45, 37), (20, 16), (200, 111)), ((72, 104), (36, 52), (108, 157))]     # no schedule; odd width


@pytest.mark.parametrize("geom", BICUBIC_GEOMS)
def test_bicubic_fp16_io(helpers_know_f16, geom):
    from transformerupscaler_b200 import _lib
    lib = _lib.load()
    G = helpers_know_f16
    dev = torch.device("cuda:0")
    (H, W), (rH, rW), (oH, oW) = geom
    x16 = synth_frames(2, H, W, seed=3).half().to(dev)
    rs = np.random.RandomState(11)
    res = torch.from_numpy(rs.uniform(-0.3, 0.3, (2, 3, rH, rW)).astype(np.float32)).to(dev)
    for clamp in (True, False):
        for variant in (2, 1, 0):              # row-schedule kernel where one applies, pair kernel, one-column kernel
            lib.tu_debug_set(b"bicubic_pair", variant)
            try:
                want = G.bicubic_add_clamp(x16.float(), res, oH, oW, F32, clamp)
                for out_dt in (F16, F32, BF16):
                    got = G.bicubic_add_clamp(x16, res, oH, oW, out_dt, clamp)
                    assert torch.equal(got, want.to(out_dt)), (clamp, variant, out_dt)
                for in_dt in (F32, BF16):
                    xi = x16.to(in_dt)
                    got = G.bicubic_add_clamp(xi, res, oH, oW, F16, clamp)
                    assert torch.equal(got, G.bicubic_add_clamp(xi, res, oH, oW, F32, clamp).half()), (clamp, variant, in_dt)
            finally:
                lib.tu_debug_set(b"bicubic_pair", 2)


def test_bicubic_fp16_input_runs_the_row_schedule_kernel(helpers_know_f16):
    G = helpers_know_f16
    dev = torch.device("cuda:0")
    x16 = synth_frames(2, 720, 1280, seed=3).half().to(dev)
    res = torch.zeros(2, 3, 360, 640, device=dev)
    G.bicubic_add_clamp(x16, res, 1080, 1920, F16, True)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        G.bicubic_add_clamp(x16, res, 1080, 1920, F16, True)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "bicubic" in e.name]
    assert any("bicubic_add_clamp_r32_kernel<__half, __half" in n for n in names), names


@pytest.mark.parametrize("r", [2, 3, 6])
def test_subpixel_and_final_conv_fp16_output(helpers_know_f16, r):
    G = helpers_know_f16
    dev = torch.device("cuda:0")
    rs = np.random.RandomState(18)
    B, H, W = 2, 11, 70
    x = torch.from_numpy(rs.uniform(-1, 1, (B, 3, H, W)).astype(np.float32)).to(dev)
    w = torch.from_numpy(rs.uniform(-0.2, 0.2, (3 * r * r, 3, 3, 3)).astype(np.float32))
    b = torch.from_numpy(rs.uniform(-0.1, 0.1, 3 * r * r).astype(np.float32)).to(dev)
    w2 = torch.from_numpy(rs.uniform(-0.2, 0.2, (3, 3, 3, 3)).astype(np.float32))
    b2 = torch.from_numpy(rs.uniform(-0.1, 0.1, 3).astype(np.float32))
    add = torch.from_numpy(rs.uniform(-0.5, 1.5, (B, 3, H * r, W * r)).astype(np.float32)).to(dev)
    wp = w.permute(2, 3, 1, 0).reshape(27, 3 * r * r).contiguous().to(dev)
    fin = torch.cat([w2.permute(2, 3, 1, 0).reshape(-1), b2])
    w2p, b2d = w2.permute(2, 3, 1, 0).reshape(27, 3).contiguous().to(dev), b2.to(dev)
    mid = G.conv3_ps(x, wp, b, r)
    for clamp in (False, True):
        got = G.subpixel_conv_add(x, wp, b, r, fin, add, F16, clamp)
        assert torch.equal(got, G.subpixel_conv_add(x, wp, b, r, fin, add, F32, clamp).half())
        got = G.final_conv_add(mid, w2p, b2d, add, F16, clamp)
        assert torch.equal(got, G.final_conv_add(mid, w2p, b2d, add, F32, clamp).half())


@pytest.mark.parametrize("geom", [((80, 112), (60, 84)), ((144, 192), (100, 150)), ((50, 70), (50, 35))])
def test_resize_aa_fp16_io(helpers_know_f16, geom):
    from transformerupscaler_b200 import engine
    G = helpers_know_f16
    (H, W), (oH, oW) = geom
    x16 = (synth_frames(2, H, W, seed=5) * 1.4 - 0.2).half().cuda()
    for clamp in (False, True):
        want = engine.tu_resize_aa(x16.float(), oH, oW, clamp)
        assert torch.equal(engine.tu_resize_aa(x16, oH, oW, clamp), want.half())                      # fp16 -> fp16 (same dtype)
        assert torch.equal(G.resize_aa(x16, oH, oW, clamp), want.half())                              # tu_resize_bilinear_aa
        assert torch.equal(engine.tu_resize_aa(x16, oH, oW, clamp, engine._code(F32)), want)          # fp16 -> fp32
        assert torch.equal(engine.tu_resize_aa(x16.float(), oH, oW, clamp, engine._code(F16)), want.half())
        xb = x16.to(BF16)
        assert torch.equal(engine.tu_resize_aa(xb, oH, oW, clamp, engine._code(F16)),
                           engine.tu_resize_aa(xb, oH, oW, clamp, engine._code(F32)).half())
