"""GPU: single ops of libtu_b200 (through the C ABI) vs the CPU oracle's restatement of the same op."""
import numpy as np
import pytest
import torch

from oracle import upscaler_oracle as orc
from oracle.weights import synth_state_dict, synth_frames
from tests import bf16_reference

pytestmark = pytest.mark.gpu

F32, BF16 = torch.float32, torch.bfloat16
# fp32 ops: exact-FFMA kernels vs fp32 CPU, differing only in summation order
TOL32 = 2e-5
# bf16 transformer block vs tests/bf16_reference.py: (max, mean) of |d| / max(1, |ref|)
TOL_BLOCK16 = (5e-3, 4e-4)     # measured on a B200: at most 1.9e-3, 1.6e-4 (ResidualTransformer)


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from transformerupscaler_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def _maxerr(a, b):
    return (a.detach().float().cpu() - b.detach().float().cpu()).abs().max().item()


def _tol(dtype, scale=1.0):
    return TOL32 * max(scale, 1.0) if dtype == F32 else 2e-2 * max(scale, 1.0)


@pytest.mark.parametrize("in_dt,dt", [(F32, F32), (F32, BF16), (BF16, BF16)])
def test_stem_conv(dev, in_dt, dt):
    from tests import gpu_helpers as G
    from transformerupscaler_b200.packing import PackedWeights
    sd = synth_state_dict("WindowTransformer", 0)
    x = synth_frames(2, 37, 53, seed=1).to(in_dt)
    ref = orc.conv3x3_nhwc(x.float().permute(0, 2, 3, 1).contiguous(), sd["conv1.weight"], sd["conv1.bias"], relu=True)
    w = sd["conv1.weight"].permute(2, 3, 1, 0).reshape(27, 64).contiguous().to(dev)
    out = G.stem_conv(x.to(dev), w, sd["conv1.bias"].to(dev), dt)
    assert _maxerr(out, ref) < _tol(dt, ref.abs().max().item())
    if dt == BF16:      # tensor-core stem: bf16 operands (image and filter rounded to bf16), fp32 accumulate
        w64 = torch.zeros(64, 64)
        w64[:, :27] = sd["conv1.weight"].permute(0, 2, 3, 1).reshape(64, 27)
        ref16 = orc.conv3x3_nhwc(x.to(BF16).float().permute(0, 2, 3, 1).contiguous(), sd["conv1.weight"].to(BF16).float(),
                                 sd["conv1.bias"], relu=True)
        for shape_x in (x, synth_frames(1, 5, 300, seed=2).to(in_dt)):
            if shape_x is not x:
                ref16 = orc.conv3x3_nhwc(shape_x.to(BF16).float().permute(0, 2, 3, 1).contiguous(),
                                         sd["conv1.weight"].to(BF16).float(), sd["conv1.bias"], relu=True)
            out16 = G.stem_conv(shape_x.to(dev), w, sd["conv1.bias"].to(dev), dt, w64=w64.to(dev, BF16))
            assert _maxerr(out16, ref16) < 1e-2


@pytest.mark.parametrize("in_dt", [F32, BF16, torch.uint8])
@pytest.mark.parametrize("shape", [(2, 19, 48), (1, 5, 304), (1, 1, 16), (1, 70, 136), (3, 33, 256)])
def test_conv12_fused(dev, in_dt, shape):
    """conv1 fused into conv2 (one kernel, conv1's output stays on chip) vs the two convolutions of the oracle on bf16-rounded
    operands (W:244-245, F:251-252, R:128-129)"""
    from tests import gpu_helpers as G
    sd = synth_state_dict("WindowTransformer", 2)
    B, H, W = shape
    if (W * torch.empty(0, dtype=in_dt).element_size()) % 16:
        pytest.skip("raw rows arrive by TMA: the image row pitch must be a multiple of 16 bytes (the forward then runs the two kernels)")
    x = synth_frames(B, H, W, seed=21)
    if in_dt == torch.uint8:
        xin = (x * 255).round().clamp(0, 255).to(torch.uint8)
        xf = xin.float() * (1.0 / 255.0)
    else:
        xin = x.to(in_dt)
        xf = xin.float()
    w1, b1, w2, b2 = sd["conv1.weight"], sd["conv1.bias"], sd["conv2.weight"], sd["conv2.bias"]
    # what the kernel computes: bf16 operands, fp32 accumulation, conv1's output rounded to bf16
    f1 = orc.conv3x3_nhwc(xf.to(BF16).float().permute(0, 2, 3, 1).contiguous(), w1.to(BF16).float(), b1, relu=True).to(BF16).float()
    ref = orc.conv3x3_nhwc(f1, w2.to(BF16).float(), b2, relu=True)
    w64 = torch.zeros(64, 64)
    w64[:, :27] = w1.permute(0, 2, 3, 1).reshape(64, 27)
    w2p = w2.permute(2, 3, 0, 1).reshape(9, 64, 64).contiguous()
    out = G.conv12_fused(xin.to(dev), w64.to(dev, BF16), b1.to(dev), w2p.to(dev, BF16), b2.to(dev))
    assert out.shape == ref.shape
    assert _maxerr(out, ref) < 2e-2 * max(ref.abs().max().item(), 1.0)
    # and against the two-kernel path of the engine (same operands; only summation order and 1-ulp bf16 flips differ)
    wst = w1.permute(2, 3, 1, 0).reshape(27, 64).contiguous().to(dev)
    two = G.conv3x3_c64(G.stem_conv(xin.to(dev), wst, b1.to(dev), BF16, w64=w64.to(dev, BF16)) if in_dt != torch.uint8 else
                        G.stem_conv(xf.to(dev), wst, b1.to(dev), BF16, w64=w64.to(dev, BF16)), w2p.to(dev, BF16), b2.to(dev), relu=1)
    assert _maxerr(out, two) < 2e-2 * max(ref.abs().max().item(), 1.0)


@pytest.mark.parametrize("dt", [F32, BF16])
@pytest.mark.parametrize("stride,relu,shape", [(1, 1, (2, 19, 45)), (2, 0, (1, 33, 41)), (2, 0, (1, 32, 48)), (1, 0, (1, 8, 130))])
def test_conv3x3_c64(dev, dt, stride, relu, shape):
    from tests import gpu_helpers as G
    rs = np.random.RandomState(5)
    B, H, W = shape
    x = torch.from_numpy(rs.uniform(-1, 1, (B, H, W, 64)).astype(np.float32)).to(dt)
    w = torch.from_numpy(rs.uniform(-0.05, 0.05, (64, 64, 3, 3)).astype(np.float32)).to(dt)
    b = torch.from_numpy(rs.uniform(-0.1, 0.1, 64).astype(np.float32))
    ref = orc.conv3x3_nhwc(x.float(), w.float(), b, stride=stride, relu=bool(relu))
    wp = w.float().permute(2, 3, 0, 1).reshape(9, 64, 64).contiguous().to(dev, dt)
    out = G.conv3x3_c64(x.to(dev), wp, b.to(dev), stride=stride, relu=relu)
    assert out.shape == ref.shape
    assert _maxerr(out, ref) < _tol(dt, ref.abs().max().item())


@pytest.mark.parametrize("dt", [F32, BF16])
@pytest.mark.parametrize("r", [2, 3, 6])
def test_conv3x3_pixelshuffle(dev, dt, r):
    from tests import gpu_helpers as G
    rs = np.random.RandomState(6)
    B, H, W = 1, 13, 21
    x = torch.from_numpy(rs.uniform(-1, 1, (B, H, W, 64)).astype(np.float32)).to(dt)
    w = torch.from_numpy(rs.uniform(-0.05, 0.05, (64 * r * r, 64, 3, 3)).astype(np.float32)).to(dt)
    b = torch.from_numpy(rs.uniform(-0.1, 0.1, 64 * r * r).astype(np.float32))
    ref = orc.pixel_shuffle_nhwc(orc.conv3x3_nhwc(x.float(), w.float(), b), r)
    wp = w.float().reshape(64, r * r, 64, 3, 3).permute(1, 3, 4, 0, 2).reshape(r * r, 9, 64, 64).contiguous().to(dev, dt)
    bp = b.reshape(64, r * r).t().reshape(-1).contiguous().to(dev)
    out = G.conv3x3_c64(x.to(dev), wp, bp, nchunk=r * r, ps_r=r)
    assert out.shape == ref.shape
    assert _maxerr(out, ref) < _tol(dt, ref.abs().max().item())


@pytest.mark.parametrize("dt", [F32, BF16])
@pytest.mark.parametrize("bias,relu", [(True, 0), (False, 1)])
def test_conv64to3(dev, dt, bias, relu):
    from tests import gpu_helpers as G
    rs = np.random.RandomState(7)
    x = torch.from_numpy(rs.uniform(-1, 1, (2, 17, 150, 64)).astype(np.float32)).to(dt)
    w = torch.from_numpy(rs.uniform(-0.05, 0.05, (3, 64, 3, 3)).astype(np.float32))
    b = torch.from_numpy(rs.uniform(-0.1, 0.1, 3).astype(np.float32)) if bias else None
    ref = orc.conv3x3_nhwc(x.float(), w, b, relu=bool(relu)).permute(0, 3, 1, 2)
    wp = w.permute(2, 3, 1, 0).reshape(9, 64, 3).contiguous().to(dev)
    out = G.conv64to3(x.to(dev), wp, None if b is None else b.to(dev), relu=relu)
    assert _maxerr(out, ref) < TOL32 * 4
    if dt == BF16:      # tensor-core head: bf16 weights (3 of 16 output channels real)
        w16 = torch.zeros(3, 4, 4, 64)                       # (ky, kx, co, ci) -> rows n = kx*4 + co
        w16[:, :3, :3] = w.permute(2, 3, 0, 1)
        w16 = w16.reshape(3, 16, 64)
        ref16 = orc.conv3x3_nhwc(x.float(), w.to(BF16).float(), b, relu=bool(relu)).permute(0, 3, 1, 2)
        out16 = G.conv64to3(x.to(dev), wp, None if b is None else b.to(dev), relu=relu, w16=w16.to(dev, BF16))
        assert _maxerr(out16, ref16) < 1e-3


@pytest.mark.parametrize("bias,relu", [(True, 0), (False, 1)])
@pytest.mark.parametrize("shape", [(2, 17, 152), (1, 1, 4), (1, 70, 640), (3, 9, 260)])
def test_conv64to3_stream(dev, bias, relu, shape):
    """64->3 heads (decoder_conv2 / up1_conv) on the streaming tensor-core kernel vs the oracle conv with bf16-rounded weights"""
    from tests import gpu_helpers as G
    rs = np.random.RandomState(17)
    B, H, W = shape
    x = torch.from_numpy(rs.uniform(-1, 1, (B, H, W, 64)).astype(np.float32)).to(BF16)
    w = torch.from_numpy(rs.uniform(-0.05, 0.05, (3, 64, 3, 3)).astype(np.float32))
    b = torch.from_numpy(rs.uniform(-0.1, 0.1, 3).astype(np.float32)) if bias else None
    ref16 = orc.conv3x3_nhwc(x.float(), w.to(BF16).float(), b, relu=bool(relu)).permute(0, 3, 1, 2)
    out = G.conv64to3_stream(x.to(dev), w, b, relu=relu)
    assert out.shape == ref16.shape
    assert _maxerr(out, ref16) < 1e-3


@pytest.mark.parametrize("shape", [(2, 17, 152), (1, 1, 4), (1, 2, 128), (1, 70, 640), (3, 9, 260), (1, 131, 256), (2, 64, 384), (1, 3, 129)])
def test_dec12_fused(dev, shape):
    """decoder_conv1 + ReLU + decoder_conv2 in one kernel (the 64-channel map stays on chip) vs the two convolutions of the
    oracle on bf16-rounded operands, decoder_conv1's output rounded to bf16 (W:297-298, F:312-313, R:156-157); shapes cover
    one / several 128-pixel strips (seam pixels), partial strips, single rows and more rows than one work item holds"""
    from tests import gpu_helpers as G
    rs = np.random.RandomState(23)
    B, H, W = shape
    x = torch.from_numpy(rs.uniform(-1, 1, (B, H, W, 64)).astype(np.float32)).to(BF16)
    w1 = torch.from_numpy(rs.uniform(-0.05, 0.05, (64, 64, 3, 3)).astype(np.float32)).to(BF16)
    b1 = torch.from_numpy(rs.uniform(-0.1, 0.1, 64).astype(np.float32))
    w2 = torch.from_numpy(rs.uniform(-0.05, 0.05, (3, 64, 3, 3)).astype(np.float32)).to(BF16)
    b2 = torch.from_numpy(rs.uniform(-0.1, 0.1, 3).astype(np.float32))
    mid = orc.conv3x3_nhwc(x.float(), w1.float(), b1, relu=True).to(BF16).float()
    ref = orc.conv3x3_nhwc(mid, w2.float(), b2).permute(0, 3, 1, 2)
    w1p = w1.float().permute(2, 3, 0, 1).reshape(9, 64, 64).contiguous().to(dev, BF16)
    w16 = torch.zeros(3, 4, 4, 64)                       # (ky, kx, co, ci) -> rows n = kx*4 + co
    w16[:, :3, :3] = w2.float().permute(2, 3, 0, 1)
    w16 = w16.reshape(3, 16, 64).to(dev, BF16)
    out = G.dec12_fused(x.to(dev), w1p, b1.to(dev), w16, b2.to(dev))
    assert out.shape == ref.shape
    assert not torch.isnan(out).any()
    assert _maxerr(out, ref) < 3e-3          # 1-ulp bf16 flips of the intermediate map (summation order differs from the oracle's)
    out2 = G.dec12_fused(x.to(dev), w1p, b1.to(dev), w16, b2.to(dev))
    assert torch.equal(out, out2)            # the seam atomics add two terms onto zero: order independent


@pytest.mark.parametrize("r", [2, 3, 6])
def test_conv3_ps_and_final(dev, r):
    from tests import gpu_helpers as G
    rs = np.random.RandomState(8)
    B, H, W = 2, 11, 70
    x = torch.from_numpy(rs.uniform(-1, 1, (B, 3, H, W)).astype(np.float32))
    w = torch.from_numpy(rs.uniform(-0.2, 0.2, (3 * r * r, 3, 3, 3)).astype(np.float32))
    b = torch.from_numpy(rs.uniform(-0.1, 0.1, 3 * r * r).astype(np.float32))
    ref = orc.pixel_shuffle_nhwc(orc.conv3x3_nhwc(x.permute(0, 2, 3, 1).contiguous(), w, b), r)
    wp = w.permute(2, 3, 1, 0).reshape(27, 3 * r * r).contiguous().to(dev)
    out = G.conv3_ps(x.to(dev), wp, b.to(dev), r)
    assert _maxerr(out, ref.permute(0, 3, 1, 2)) < TOL32
    # final 3->3 conv + addend + clamp
    w2 = torch.from_numpy(rs.uniform(-0.2, 0.2, (3, 3, 3, 3)).astype(np.float32))
    b2 = torch.from_numpy(rs.uniform(-0.1, 0.1, 3).astype(np.float32))
    add = torch.from_numpy(rs.uniform(0, 1, tuple(out.shape)).astype(np.float32))
    ref2 = (orc.conv3x3_nhwc(ref, w2, b2).permute(0, 3, 1, 2) + add).clamp(0, 1)
    out2 = G.final_conv_add(out, w2.permute(2, 3, 1, 0).reshape(27, 3).contiguous().to(dev), b2.to(dev), add.to(dev), F32, True)
    assert _maxerr(out2, ref2) < TOL32


@pytest.mark.parametrize("r", [2, 3, 6])
@pytest.mark.parametrize("shape", [(1, 13, 20), (2, 40, 300), (1, 3, 132), (1, 1, 4)])
def test_upfold_conv(dev, r, shape):
    """folded up1 stage + PixelShuffle + up1_conv + ReLU (tensor cores) vs the op chain of the oracle,
    FastTransformer/utils.py:43-98, 13-40; model.py:264-265"""
    from tests import gpu_helpers as G
    rs = np.random.RandomState(30 + r)
    B, H, W = shape
    x = torch.from_numpy(rs.uniform(-1, 1, (B, H, W, 64)).astype(np.float32)).to(BF16)
    w1 = torch.from_numpy(rs.uniform(-0.05, 0.05, (64 * r * r, 64, 3, 3)).astype(np.float32))
    b1 = torch.from_numpy(rs.uniform(-0.1, 0.1, 64 * r * r).astype(np.float32))
    w2 = torch.from_numpy(rs.uniform(-0.1, 0.1, (3, 64, 3, 3)).astype(np.float32))
    out, Wf, bf = G.upfold_conv(x.to(dev), w1, b1, w2, r)
    # (a) the reference op chain in fp32 on the same bf16 input: differs by the bf16 rounding of the folded filter only
    ref = orc.conv3x3_nhwc(orc.pixel_shuffle_nhwc(orc.conv3x3_nhwc(x.float(), w1, b1), r), w2, None, relu=True).permute(0, 3, 1, 2)
    assert out.shape == ref.shape
    assert _maxerr(out, ref) < 2e-2
    # (b) the same 5x5 convolution with the bf16-rounded folded filter, fp64 accumulation: tight
    Wi = Wf[1, 1].to(BF16).double()                                   # (o, ci, dy, dx)
    xp = torch.zeros(B, H + 4, W + 4, 64, dtype=torch.float64)
    xp[:, 2:H + 2, 2:W + 2] = x.double()
    acc = torch.zeros(B, H, W, 3 * r * r, dtype=torch.float64)
    for dy in range(5):
        for dx in range(5):
            acc += xp[:, dy:dy + H, dx:dx + W].reshape(-1, 64).matmul(Wi[:, :, dy, dx].t()).reshape(B, H, W, -1)
    acc = (acc + bf[1, 1]).clamp(min=0).reshape(B, H, W, 3, r, r).permute(0, 3, 1, 4, 2, 5).reshape(B, 3, H * r, W * r)
    inner = (out.double().cpu() - acc)[:, :, 1:-1, 1:-1]
    assert inner.abs().max().item() < 2e-4 if inner.numel() else True
    # (c) the border ring is computed with the fp32 border filters: close to the exact chain
    ring = (out.cpu() - ref).clone()
    ring[:, :, 1:-1, 1:-1] = 0
    assert ring.abs().max().item() < 2e-4


@pytest.mark.parametrize("r", [2, 3, 6])
@pytest.mark.parametrize("shape", [(2, 11, 70), (1, 31, 29), (1, 1, 1), (1, 40, 61)])
def test_subpixel_conv_add_fused(dev, r, shape):
    """fused tail (sub-pixel conv + PixelShuffle + 3->3 conv + sum + clamp) vs the op-by-op restatement, FastTransformer/model.py:316-327"""
    from tests import gpu_helpers as G
    rs = np.random.RandomState(18)
    B, H, W = shape
    x = torch.from_numpy(rs.uniform(-1, 1, (B, 3, H, W)).astype(np.float32))
    w = torch.from_numpy(rs.uniform(-0.2, 0.2, (3 * r * r, 3, 3, 3)).astype(np.float32))
    b = torch.from_numpy(rs.uniform(-0.1, 0.1, 3 * r * r).astype(np.float32))
    w2 = torch.from_numpy(rs.uniform(-0.2, 0.2, (3, 3, 3, 3)).astype(np.float32))
    b2 = torch.from_numpy(rs.uniform(-0.1, 0.1, 3).astype(np.float32))
    add = torch.from_numpy(rs.uniform(0, 1, (B, 3, H * r, W * r)).astype(np.float32))
    mid = orc.pixel_shuffle_nhwc(orc.conv3x3_nhwc(x.permute(0, 2, 3, 1).contiguous(), w, b), r)
    pre = orc.conv3x3_nhwc(mid, w2, b2).permute(0, 3, 1, 2) + add
    wp = w.permute(2, 3, 1, 0).reshape(27, 3 * r * r).contiguous().to(dev)
    fin = torch.cat([w2.permute(2, 3, 1, 0).reshape(-1), b2])
    for clamp in (False, True):
        out = G.subpixel_conv_add(x.to(dev), wp, b.to(dev), r, fin, add.to(dev), F32, clamp)
        assert _maxerr(out, pre.clamp(0, 1) if clamp else pre) < TOL32
    out16 = G.subpixel_conv_add(x.to(dev), wp, b.to(dev), r, fin, add.to(dev), BF16, True)
    assert _maxerr(out16, pre.clamp(0, 1)) < 4e-3


@pytest.mark.parametrize("dt", [F32, BF16])
@pytest.mark.parametrize("model,Hf,Wf", [("WindowTransformer", 36, 52), ("FastTransformer", 36, 52), ("FastTransformer", 64, 80)])
def test_patch_embed_unembed(dev, dt, model, Hf, Wf):
    from tests import gpu_helpers as G
    rs = np.random.RandomState(9)
    sd = synth_state_dict(model, 3)
    dim = sd["patch_embed.weight"].shape[0]
    fast = model == "FastTransformer"
    B = 2
    feat = torch.from_numpy(rs.uniform(-1, 1, (B, Hf, Wf, 64)).astype(np.float32)).to(dt)
    Ht, Wt = ((Hf + 7) // 8, (Wf + 7) // 8) if fast else (Hf // 8, Wf // 8)
    fpad = orc.reflect_pad_nhwc(feat.float(), Ht * 8 - Hf, Wt * 8 - Wf) if fast else feat.float()
    we = sd["patch_embed.weight"].to(dt).float()
    tok_ref = orc.patch_embed_nhwc(fpad, we, sd["patch_embed.bias"])            # (B,Ht,Wt,dim)
    wp = we.permute(0, 2, 3, 1).reshape(dim, 4096).contiguous().to(dev, dt)
    tok = G.patch_embed(feat.to(dev), wp, sd["patch_embed.bias"].to(dev), None, Ht, Wt, dim, True, fast)
    nWy, nWx = (Ht + 7) // 8, (Wt + 7) // 8
    grid = tok.reshape(B, nWy, nWx, 8, 8, dim).permute(0, 1, 3, 2, 4, 5).reshape(B, nWy * 8, nWx * 8, dim)
    scale = tok_ref.abs().max().item()
    assert _maxerr(grid[:, :Ht, :Wt], tok_ref) < _tol(dt, scale)
    if nWy * 8 > Ht:
        assert grid[:, Ht:].abs().max().item() == 0          # zero pad tokens (no bias)
    if nWx * 8 > Wt:
        assert grid[:, :, Wt:].abs().max().item() == 0
    # unembed + crop + skip
    wu = sd["patch_unembed.weight"].to(dt).float()
    Hc, Wc = (Hf, Wf) if fast else (min(Hf, 8 * Ht), min(Wf, 8 * Wt))
    ref = orc.patch_unembed_nhwc(grid[:, :Ht, :Wt].cpu().contiguous(), wu, sd["patch_unembed.bias"])[:, :Hc, :Wc] + feat.float()[:, :Hc, :Wc]
    wup = wu.permute(2, 3, 1, 0).reshape(4096, dim).contiguous().to(dev, dt)
    out = G.patch_unembed(tok, wup, sd["patch_unembed.bias"].to(dev), feat.to(dev), B, Ht, Wt, Hc, Wc, dim, True)
    assert _maxerr(out, ref) < _tol(dt, ref.abs().max().item())


@pytest.mark.parametrize("model,B,Hf,Wf", [("WindowTransformer", 2, 64, 80), ("WindowTransformer", 3, 40, 136), ("FastTransformer", 2, 64, 80),
                                            ("FastTransformer", 1, 24, 264), ("WindowTransformer", 5, 360, 640)])
def test_patch_embed_variants(dev, model, B, Hf, Wf):
    """patch embed on the tensor cores: the general persistent GEMM kernel, one tile per CTA with two CTAs per SM, and the same with the
    filter stages multicast inside clusters of two CTAs accumulate the same k-blocks in the same order: bitwise identical tokens, and
    equal to the oracle's patch_embed on bf16-rounded operands (W:251-254; F:268-270)"""
    from tests import gpu_helpers as G
    from transformerupscaler_b200 import _lib
    lib = _lib.load()
    rs = np.random.RandomState(19)
    sd = synth_state_dict(model, 3)
    dim = sd["patch_embed.weight"].shape[0]
    feat = torch.from_numpy(rs.uniform(-1, 1, (B, Hf, Wf, 64)).astype(np.float32)).to(BF16)
    Ht, Wt = Hf // 8, Wf // 8
    we = sd["patch_embed.weight"].to(BF16).float()
    wp = we.permute(0, 2, 3, 1).reshape(dim, 4096).contiguous().to(dev, BF16)
    outs = []
    try:
        for variant in (0, 1 + 4, 2 + 4, 1 + 4 + 8):      # bit mask: 1 two CTAs per SM, 2 cluster multicast, 4 also at dim 192, 8 L2 prefetch
            lib.tu_debug_set(b"embed_pair", variant)
            outs.append(G.patch_embed(feat.to(dev), wp, sd["patch_embed.bias"].to(dev), None, Ht, Wt, dim, True, False).clone())
    finally:
        lib.tu_debug_set(b"embed_pair", 1)
    assert all(torch.equal(outs[0], o) for o in outs[1:])
    if Hf * Wf <= 64 * 264:
        tok_ref = orc.patch_embed_nhwc(feat.float()[:, :Ht * 8, :Wt * 8], we, sd["patch_embed.bias"])
        nWy, nWx = (Ht + 7) // 8, (Wt + 7) // 8
        grid = outs[1].reshape(B, nWy, nWx, 8, 8, dim).permute(0, 1, 3, 2, 4, 5).reshape(B, nWy * 8, nWx * 8, dim)
        assert _maxerr(grid[:, :Ht, :Wt], tok_ref) < _tol(BF16, tok_ref.abs().max().item())


@pytest.mark.parametrize("dt", [F32, BF16])
@pytest.mark.parametrize("model", ["WindowTransformer", "FastTransformer", "ResidualTransformer"])
def test_transformer_block(dev, dt, model):
    from tests import gpu_helpers as G
    from transformerupscaler_b200.packing import PackedWeights
    rs = np.random.RandomState(10)
    sd = synth_state_dict(model, 4)
    pw = PackedWeights(model, sd, dt, dev)
    dim, heads = pw.dim, pw.heads
    if model == "ResidualTransformer":
        B, S = 2, 300
        x = torch.from_numpy(rs.standard_normal((B, S, dim)).astype(np.float32))
        sdq = {k: (v.to(dt).float() if v.dim() == 2 else v) for k, v in sd.items()}
        ref = orc.mha_block(x, sdq, "transformer_blocks.1.", heads, F32)
        ref16 = bf16_reference.mha_block(x, sd, "transformer_blocks.1.", heads)
        out = G.transformer_block(x.reshape(B * S, dim).to(dev).clone(), pw.blocks[1], dim, heads, False, S, dt)
        out = out.reshape(B, S, dim)
    else:
        nW = 5
        x = torch.from_numpy(rs.standard_normal((nW, 64, dim)).astype(np.float32))
        sdq = {k: (v.to(dt).float() if (v.dim() == 2 and "table" not in k) else v) for k, v in sd.items()}
        ref = orc.window_block(x, sdq, "window_blocks.1.", heads, F32)
        # window_attn_mma_kernel sums the softmax row over the fp32 probabilities, before they are rounded for P V
        ref16 = bf16_reference.window_block(x, sd, "window_blocks.1.", heads, rowsum_rounded=False)
        out = G.transformer_block(x.reshape(nW * 64, dim).to(dev).clone(), pw.blocks[1], dim, heads, True, 0, dt)
        out = out.reshape(nW, 64, dim)
    if dt == F32:
        assert _maxerr(out, ref) < 5e-5
    else:       # the same bf16 stores (LN out, qkv, probabilities, attn out, MLP hidden) as the reference
        d = (out.cpu().double() - ref16).abs() / ref16.abs().clamp(min=1.0)
        assert d.max().item() < TOL_BLOCK16[0] and d.mean().item() < TOL_BLOCK16[1]


@pytest.mark.parametrize("dt", [F32, BF16])
@pytest.mark.parametrize("dim,heads", [(128, 8), (192, 12)])
def test_window_attention(dev, dt, dim, heads):
    """softmax(q k^T + bias) v per window and head vs a direct restatement (WindowTransformer/model.py:104-127)."""
    from tests import gpu_helpers as G
    rs = np.random.RandomState(12)
    nW = 7
    qkv = torch.from_numpy(rs.standard_normal((nW * 64, 3 * dim)).astype(np.float32)).to(dt)
    bias = torch.from_numpy((0.5 * rs.standard_normal((heads, 64, 64))).astype(np.float32))
    q, k, v = qkv.float().reshape(nW, 64, 3, heads, 16).permute(2, 0, 3, 1, 4)      # (nW, h, 64, 16) each
    att = torch.softmax(q @ k.transpose(-1, -2) + bias[None], dim=-1) @ v            # q is taken as already scaled
    ref = att.permute(0, 2, 1, 3).reshape(nW * 64, dim)
    out = G.window_attention(qkv.to(dev), bias.to(dev), dim, heads)
    assert _maxerr(out, ref) < (2e-5 if dt == F32 else 3e-2)


@pytest.mark.parametrize("in_dt,out_dt", [(F32, F32), (BF16, BF16), (F32, BF16)])
@pytest.mark.parametrize("geom", [((72, 104), (36, 52), (108, 156)), ((64, 80), (32, 40), (128, 160)), ((45, 37), (20, 16), (200, 111))])
def test_bicubic_add_clamp(dev, in_dt, out_dt, geom):
    from tests import gpu_helpers as G
    (H, W), (rH, rW), (oH, oW) = geom
    x = synth_frames(2, H, W, seed=3).to(in_dt)
    rs = np.random.RandomState(11)
    res = torch.from_numpy(rs.uniform(-0.3, 0.3, (2, 3, rH, rW)).astype(np.float32))
    ref = orc.bicubic_nchw(x.float(), (oH, oW)) + orc.bicubic_nchw(res, (oH, oW))
    out = G.bicubic_add_clamp(x.to(dev), res.to(dev), oH, oW, out_dt, False)
    tol = 2e-6 if out_dt == F32 else 8e-3        # bf16 store: half-ulp of values up to ~1.3
    assert _maxerr(out, ref) < tol
    outc = G.bicubic_add_clamp(x.to(dev), res.to(dev), oH, oW, out_dt, True)
    assert _maxerr(outc, ref.clamp(0, 1)) < tol
    # x only (residual absent)
    out1 = G.bicubic_add_clamp(x.to(dev), None, oH, oW, out_dt, False)
    assert _maxerr(out1, orc.bicubic_nchw(x.float(), (oH, oW))) < tol


@pytest.mark.parametrize("in_dt,out_dt", [(BF16, BF16), (torch.uint8, torch.uint8), (BF16, F32), (torch.uint8, BF16), (BF16, torch.uint8)])
@pytest.mark.parametrize("geom", [((720, 1280), (360, 640), (1080, 1920)), ((72, 104), (36, 52), (108, 156)), ((48, 64), (24, 40), (72, 250)),
                                  ((24, 304), (12, 152), (36, 456)),
                                  # x 3:1, residual 6:1 (ResidualTransformer 720p -> 4K, R:125,160): the second row schedule
                                  ((720, 1280), (360, 640), (2160, 3840)), ((24, 48), (12, 24), (72, 144)), ((16, 64), (8, 40), (48, 200)),
                                  # the other integer scales of inference.py (x n:1, residual 2n:1): 2, 4, 6
                                  ((720, 1280), (360, 640), (1440, 2560)), ((24, 48), (12, 24), (48, 96)), ((48, 64), (24, 40), (96, 250)),
                                  ((360, 640), (180, 320), (1440, 2560)), ((8, 48), (4, 24), (32, 192)), ((16, 32), (8, 24), (64, 150)),
                                  ((96, 128), (48, 64), (576, 768)), ((8, 48), (4, 24), (48, 288))])
def test_bicubic_fixed_row_pattern_kernel(dev, in_dt, out_dt, geom):
    """The unrolled periodic-row-schedule kernels (outH = 3/2 H = 3 rH: 720p -> 1080p, tile and streaming forms; outH = n H = 2n rH for
    n = 2, 3, 4, 6: inference.py's scales, 720p -> 4K at n = 3) against the pair kernel they replace (bitwise: same sums in
    the same order, zero-weight taps are exact no-ops) and against the oracle.  W:224-305 (241, 301, 304-305)."""
    from tests import gpu_helpers as G
    from transformerupscaler_b200 import _lib
    lib = _lib.load()
    (H, W), (rH, rW), (oH, oW) = geom
    B = 2
    x = synth_frames(B, H, W, seed=3)
    if in_dt == torch.uint8:
        x = (x * 255).round().clamp(0, 255).to(torch.uint8)
    else:
        x = x.to(in_dt)
    rs = np.random.RandomState(11)
    res = torch.from_numpy(rs.uniform(-0.3, 0.3, (B, 3, rH, rW)).astype(np.float32))
    outs = {}
    try:
        for variant in (3, 2, 1):     # streaming form, tile form, pair kernel
            lib.tu_debug_set(b"bicubic_pair", variant)
            outs[variant] = G.bicubic_add_clamp(x.to(dev), res.to(dev), oH, oW, out_dt, True).cpu()
        lib.tu_debug_set(b"bicubic_pair", 2)
        for tile in (1, 2):           # rows per CTA: the smaller / the larger tile (the default picks by grid size)
            lib.tu_debug_set(b"bicubic_tile", tile)
            outs[10 + tile] = G.bicubic_add_clamp(x.to(dev), res.to(dev), oH, oW, out_dt, True).cpu()
    finally:
        lib.tu_debug_set(b"bicubic_pair", 2)
        lib.tu_debug_set(b"bicubic_tile", 0)
    for variant in (3, 2, 11, 12):
        assert torch.equal(outs[variant], outs[1]), variant
    if H <= 128:
        xf = x.float() / 255 if in_dt == torch.uint8 else x.float()
        ref = (orc.bicubic_nchw(xf, (oH, oW)) + orc.bicubic_nchw(res, (oH, oW))).clamp(0, 1)
        got = outs[2].float() / 255 if out_dt == torch.uint8 else outs[2].float()
        tol = 2e-6 if out_dt == F32 else (1.01 / 255 if out_dt == torch.uint8 else 8e-3)     # uint8: truncation of v * 255
        assert _maxerr(got, ref) < tol


@pytest.mark.parametrize("in_dt", [BF16, torch.uint8])
@pytest.mark.parametrize("bgr", [False, True])
@pytest.mark.parametrize("geom", [((720, 1280), (360, 640), (1080, 1920)), ((24, 304), (12, 152), (36, 456)), ((24, 48), (12, 24), (72, 144)),
                                  ((48, 64), (24, 40), (96, 250))])
def test_bicubic_row_schedule_kernel_interleaved_frames(dev, in_dt, bgr, geom):
    """uint8 HWC RGB / BGR frames out of the unrolled row-schedule kernel (app_overlay.py:382-386 fused into the last kernel): bitwise the
    pair kernel's frames, and the planar result with the channels moved / reversed."""
    from tests import gpu_helpers as G
    from transformerupscaler_b200 import _lib
    lib = _lib.load()
    (H, W), (rH, rW), (oH, oW) = geom
    x = synth_frames(2, H, W, seed=5)
    x = (x * 255).round().clamp(0, 255).to(torch.uint8) if in_dt == torch.uint8 else x.to(in_dt)
    rs = np.random.RandomState(12)
    res = torch.from_numpy(rs.uniform(-0.3, 0.3, (2, 3, rH, rW)).astype(np.float32))
    layout = _lib.TU_LAYOUT_HWC_BGR if bgr else _lib.TU_LAYOUT_HWC
    outs = {}
    try:
        for variant in (2, 1):
            lib.tu_debug_set(b"bicubic_pair", variant)
            outs[variant] = G.bicubic_add_clamp(x.to(dev), res.to(dev), oH, oW, torch.uint8, True, layout).cpu()
        lib.tu_debug_set(b"bicubic_pair", 2)
        lib.tu_debug_set(b"bicubic_tile", 2)
        outs[12] = G.bicubic_add_clamp(x.to(dev), res.to(dev), oH, oW, torch.uint8, True, layout).cpu()
    finally:
        lib.tu_debug_set(b"bicubic_pair", 2)
        lib.tu_debug_set(b"bicubic_tile", 0)
    assert torch.equal(outs[2], outs[1]) and torch.equal(outs[12], outs[1])
    planar = G.bicubic_add_clamp(x.to(dev), res.to(dev), oH, oW, torch.uint8, True).cpu()
    want = planar.permute(0, 2, 3, 1)
    assert torch.equal(outs[2], want.flip(-1) if bgr else want)


@pytest.mark.parametrize("geom", [((80, 112), (60, 84)), ((144, 192), (100, 150)), ((50, 70), (50, 35))])
def test_resize_aa(dev, geom):
    from tests import gpu_helpers as G
    (H, W), (oH, oW) = geom
    x = synth_frames(2, H, W, seed=5)
    ref = orc.aa_bilinear_resize_nchw(x, (oH, oW))
    out = G.resize_aa(x.to(dev), oH, oW, False)
    assert _maxerr(out, ref) < 5e-6      # fp32, different summation order / weight normalisation order


@pytest.mark.parametrize("shape", [(2, 36, 52), (1, 33, 47), (3, 720, 1280)])
@pytest.mark.parametrize("bgr", [False, True])
def test_frames_to_planar(shape, bgr):
    from transformerupscaler_b200 import _lib
    lib = _lib.load()
    B, H, W = shape
    g = torch.Generator().manual_seed(3)
    x = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).cuda()
    out = torch.empty(B, 3, H, W, dtype=torch.uint8, device="cuda")
    _lib.check(lib.tu_frames_to_planar(x.data_ptr(), _lib.TU_LAYOUT_HWC_BGR if bgr else _lib.TU_LAYOUT_HWC, out.data_ptr(), B, H, W,
                                       torch.cuda.current_stream().cuda_stream))
    want = (x[..., [2, 1, 0]] if bgr else x).permute(0, 3, 1, 2)
    assert torch.equal(out, want)


@pytest.mark.parametrize("B,S", [(2, 3600), (3, 328), (1, 128), (1, 1032), (5, 256)])
def test_global_attention_tcgen05_block(dev, B, S):
    """ResidualTransformer's TransformerBlock (R:22-50) with the tcgen05 flash attention (S tile in TMEM, P through shared memory, K / V^T
    by TMA, key range split evenly over the SMs with merged partials) vs the oracle's nn.MultiheadAttention restatement and vs the
    mma.sync kernel it replaces; token counts with partial query / key tiles and inactive second query tiles included."""
    from tests import gpu_helpers as G
    from transformerupscaler_b200 import _lib
    from transformerupscaler_b200.packing import PackedWeights
    lib = _lib.load()
    rs = np.random.RandomState(20 + S)
    sd = synth_state_dict("ResidualTransformer", 6)
    pw = PackedWeights("ResidualTransformer", sd, BF16, dev)
    dim, heads = pw.dim, pw.heads
    x = torch.from_numpy((1.5 * rs.standard_normal((B, S, dim))).astype(np.float32))
    sdq = {k: (v.to(BF16).float() if v.dim() == 2 else v) for k, v in sd.items()}
    ref = orc.mha_block(x, sdq, "transformer_blocks.2.", heads, F32)
    try:
        lib.tu_debug_set(b"global_attn_tc", 1)            # opt-in: the forward defaults to the (measured faster) mma.sync kernel
        n0 = lib.tu_launch_count()
        new = G.transformer_block(x.reshape(B * S, dim).to(dev).clone(), pw.blocks[2], dim, heads, False, S, BF16, full_workspace=True)
        torch.cuda.synchronize()
        n_new = lib.tu_launch_count() - n0
        # run-to-run: the partials are merged in a fixed order, no atomics
        again = G.transformer_block(x.reshape(B * S, dim).to(dev).clone(), pw.blocks[2], dim, heads, False, S, BF16, full_workspace=True)
        torch.cuda.synchronize()
    finally:
        lib.tu_debug_set(b"global_attn_tc", 0)
    n1 = lib.tu_launch_count()
    old = G.transformer_block(x.reshape(B * S, dim).to(dev).clone(), pw.blocks[2], dim, heads, False, S, BF16, full_workspace=True)
    torch.cuda.synchronize()
    n_old = lib.tu_launch_count() - n1
    assert n_new == n_old + 2, (n_new, n_old)            # V^T + attention + merge instead of one kernel: the tcgen05 path really ran
    assert _maxerr(new.reshape(B, S, dim), ref) < 6e-2
    assert _maxerr(new, old) < 3e-2
    assert torch.equal(again, new)


@pytest.mark.parametrize("B,S", [(2, 3600), (1, 3600), (3, 328), (1, 130), (5, 256), (2, 1032)])
def test_global_attention_balanced_launch(dev, B, S):
    """ResidualTransformer's attention (R:31,44: nn.MultiheadAttention, head_dim 16) with the BALANCED launches of the mma.sync kernel
    (units of (query tile, key tile) cut into equal contiguous ranges per resident CTA, partial (m, l, o) of split query tiles merged by a
    second kernel: debug key ga_shape 4 = 64-query tiles, 5 = 128-query tiles) against the plain launch (one CTA per query tile) and a
    float64 softmax(q k^T) v of the same bf16 inputs; ragged token counts split tiles in every possible place."""
    from transformerupscaler_b200 import _lib
    lib = _lib.load()
    heads, dim = 8, 128
    g = torch.Generator().manual_seed(100 + S)
    qkv = torch.randn(B * S, 3 * dim, generator=g).bfloat16()
    qkv[:, :dim] *= 0.25
    q, k, v = (qkv[:, i * dim:(i + 1) * dim].double().reshape(B, S, heads, 16).permute(0, 2, 1, 3) for i in range(3))
    ref = (torch.softmax(q @ k.transpose(-1, -2), dim=-1) @ v).permute(0, 2, 1, 3).reshape(B * S, dim)
    d_qkv = qkv.to(dev)
    nws = lib.tu_global_attention_workspace_bytes(B, S, heads)
    assert nws > 0
    ws = torch.empty(nws, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    outs = {}
    try:
        for shape in (0, 4, 5, -1):
            lib.tu_debug_set(b"ga_shape", shape)
            out = torch.full((B * S, dim), float("nan"), dtype=torch.bfloat16, device=dev)
            _lib.check(lib.tu_global_attention(d_qkv.data_ptr(), out.data_ptr(), B, S, heads, ws.data_ptr(), nws, st))
            again = torch.empty_like(out)
            _lib.check(lib.tu_global_attention(d_qkv.data_ptr(), again.data_ptr(), B, S, heads, ws.data_ptr(), nws, st))
            torch.cuda.synchronize()
            assert torch.equal(out, again), shape                      # partials are merged in a fixed order
            outs[shape] = out.float().cpu()
    finally:
        lib.tu_debug_set(b"ga_shape", -1)
    for shape, out in outs.items():
        assert torch.isfinite(out).all(), shape
        assert (out.double() - ref).abs().max().item() < 2e-2, shape   # bf16 probabilities and outputs
        assert (out - outs[0]).abs().max().item() < 8e-3, shape        # same arithmetic per key tile, different merge points
