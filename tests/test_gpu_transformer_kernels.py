"""GPU: the fused transformer kernels -- the window stacks (tc/window_stack_tcgen05.cu, dim 128; tc/window_stack192_tcgen05.cu,
dim 192) and the two kernels of a ResidualTransformer layer (tc/residual_block_tcgen05.cu) -- against tests/bf16_reference.py,
the oracle's blocks in float64 with the kernels' bf16 stores.

The error of a value is |out - ref| / max(1, |ref - offset|), offset being the shared offset of the token row (0 except in the
"offset" regime): a LayerNorm that loses the spread of a row under its mean shows up however large that mean is.  Bounds are per
quantity and input regime (max, mean), set from errors measured on a B200 (TOL).  What they
must absorb is what the reference leaves out on purpose: fp32 summation order, the fitted tanh GELU, ex2 / rcp / tanh .approx and
the fp32 LayerNorm statistics.  A single block is also run alone (the stack kernel with a one-block weight set): there the errors
do not pile up through the stack, which is what lets a wrong index or coefficient of one block stand out
(tests/test_bf16_reference_host.py::test_planted_bugs_exceed_the_gpu_bounds).
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import upscaler_oracle as orc
from oracle.weights import synth_state_dict
from tests import bf16_reference as br

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16
QKV_KEY = {"WindowTransformer": "attn.qkv.weight", "FastTransformer": "attn.qkv.weight", "ResidualTransformer": "attn.in_proj_weight"}

# Bounds on (max, mean) of the relative error, per kernel output and input regime: the errors measured on a B200 (1000 W) with the
# Chan-combined LayerNorm statistics, times 2.5-4.  "block" = one block run alone through the stack kernel.  The peaked-softmax
# and large-GELU regimes amplify every bf16 rounding flip of the logits / hidden units, and through a whole stack that compounds
# (the reference itself moves by 0.14 max when it runs in fp32 instead of fp64 with peaked softmax): their stack bounds are loose,
# their one-block bounds are not.  At an offset of 1000 the fp32 residual stream and the fp32 row mean are worth 6e-5 a value.
TOL = {
    "block128": {"default": (4e-3, 2e-4), "table30": (4e-3, 2e-4), "peaked": (3e-2, 3e-4), "fc1x4": (1.5e-2, 4e-4),
                 "offset": (8e-3, 1e-3)},
    "block192": {"default": (4e-3, 2e-4), "table30": (4e-3, 2e-4), "peaked": (2.5e-2, 4e-4), "fc1x4": (1.5e-2, 5e-4),
                 "offset": (1e-2, 1.2e-3)},
    "stack128": {"default": (2.5e-2, 3e-3), "table30": (2e-2, 3e-3), "peaked": (1.0, 8e-2), "fc1x4": (0.1, 1.2e-2),
                 "offset": (4e-2, 6e-3)},
    "stack192": {"default": (1.5e-2, 2.5e-3), "table30": (1.5e-2, 2.5e-3), "peaked": (0.8, 6e-2), "fc1x4": (0.1, 1e-2),
                 "offset": (4e-2, 6e-3)},
    "resid_pre": {"default": (2e-2, 1.5e-6), "offset": (2e-2, 1e-4)},
    "resid_post": {"default": (4e-3, 3e-4), "offset": (1e-2, 6e-4)},
}
REGIMES = ["default", "table30", "peaked", "fc1x4", "offset"]
OFFSETS = (0.0, 10.0, 100.0, 1000.0)       # mean / std of the offset rows; then constant rows, and rows whose variance is LayerNorm's eps


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from transformerupscaler_b200 import _lib
    _lib.load()
    return torch.device("cuda:0")


def regime_sd(model, regime, seed=5):
    """synth_state_dict with one kind of tensor scaled: the relative-position tables to trained magnitude, the qkv weights for a peaked
    softmax, or fc1 so that the GELU's inputs pass |x| = 8 (the clamp of the kernels' fitted GELU)"""
    sd = synth_state_dict(model, seed)
    key, gain = {"table30": ("attn.relative_position_bias_table", 30.0), "peaked": (QKV_KEY[model], 3.5),
                 "fc1x4": ("mlp.0.weight", 4.0)}.get(regime, (None, 1.0))
    return {k: (v * gain if key and k.endswith(key) else v) for k, v in sd.items()}


def regime_tokens(M, dim, regime, seed):
    """(M, dim) fp32 tokens and the per-row offset the error is measured from"""
    rs = np.random.RandomState(seed)
    x = rs.standard_normal((M, dim))
    off = np.zeros(M)
    if regime == "offset":
        n = len(OFFSETS)
        kind = np.arange(M) % (n + 2)
        sign = np.where(rs.uniform(size=M) < 0.5, -1.0, 1.0)
        off = np.where(kind < n, np.array(OFFSETS + (0.0, 0.0))[kind] * sign, 3.0 * rs.standard_normal(M))
        spread = np.where(kind < n, 1.0, np.where(kind == n, 0.0, 10 ** -2.5))
        x = off[:, None] + spread[:, None] * x
    return torch.from_numpy(x.astype(np.float32)), torch.from_numpy(off)


def rel_err(out, ref, off):
    ref = ref.double().reshape(out.shape[0], -1)
    d = (out.detach().cpu().double().reshape(ref.shape) - ref).abs() / (ref - off.double()[:, None]).abs().clamp(min=1.0)
    return d.max().item(), d.mean().item()


def check(quantity, regime, out, ref, off):
    emax, emean = rel_err(out, ref, off)
    tmax, tmean = TOL[quantity][regime]
    assert emax < tmax and emean < tmean, (quantity, regime, emax, emean)


def one_block(sd, b, prefix="window_blocks."):
    """the state dict with block b as its only block"""
    out = {k: v for k, v in sd.items() if not k.startswith(prefix)}
    out.update({prefix + "0." + k[len(f"{prefix}{b}."):]: v for k, v in sd.items() if k.startswith(f"{prefix}{b}.")})
    return out


def block0_logits_and_preacts(x, sd, heads, prefix="window_blocks.0."):
    """largest |attention logit| and |fc1 pre-activation| of the first block (float64, exact): the range a regime actually reaches"""
    f = torch.float64
    h = orc.layer_norm(x.double(), sd[prefix + "norm1.weight"].double(), sd[prefix + "norm1.bias"].double())
    nW, N, D = h.shape
    qkv = orc.linear(h, sd[prefix + "attn.qkv.weight"].to(f), sd[prefix + "attn.qkv.bias"].to(f)).reshape(nW, N, 3, heads, 16)
    q, k = qkv[:, :, 0].transpose(1, 2) * 0.25, qkv[:, :, 1].transpose(1, 2)
    s = q @ k.transpose(-1, -2) + orc.dense_rel_bias(sd[prefix + "attn.relative_position_bias_table"].to(f))[None]
    h2 = orc.layer_norm(x.double(), sd[prefix + "norm2.weight"].double(), sd[prefix + "norm2.bias"].double())
    a = orc.linear(h2, sd[prefix + "mlp.0.weight"].to(f), sd[prefix + "mlp.0.bias"].to(f))
    return s.abs().max().item(), a.abs().max().item()


@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("model", ["WindowTransformer", "FastTransformer"])
def test_window_stack_vs_bf16_reference(dev, model, regime):
    """tu_window_stack (all blocks, then every block alone) vs the bf16-store reference (W:272-273, F:288-289)"""
    from tests import gpu_helpers as G
    from transformerupscaler_b200.packing import PackedWeights
    sd = regime_sd(model, regime)
    pw = PackedWeights(model, sd, BF16, dev)
    dim, heads, nb = pw.dim, pw.heads, pw.n_blocks
    nW = 6
    x, off = regime_tokens(nW * 64, dim, regime, seed=21)
    if regime in ("peaked", "fc1x4"):
        logit, pre = block0_logits_and_preacts(x.reshape(nW, 64, dim), sd, heads)
        assert logit >= 20 if regime == "peaked" else pre > 8, (logit, pre)
    out = G.window_stack(x.to(dev).clone(), pw)
    ref = br.window_stack(x.reshape(nW, 64, dim), sd, heads, nb)
    check(f"stack{dim}", regime, out, ref, off)
    for b in range(nb):
        sd1 = one_block(sd, b)
        out = G.window_stack(x.to(dev).clone(), PackedWeights(model, sd1, BF16, dev))
        ref = br.window_block(x.reshape(nW, 64, dim), sd1, "window_blocks.0.", heads)
        check(f"block{dim}", regime, out, ref, off)


@pytest.mark.parametrize("model", ["WindowTransformer", "FastTransformer"])
def test_window_stack_schedule_invariance(dev, model):
    """A 128-token tile's output does not depend on how many tiles share the launch (fewer tiles than SMs, as many, one more, two
    rounds), on the order the CTAs walk them (snake bit 2) or on when the relative-position bias is fetched (stack_var bit 0), and
    two runs are identical: bitwise."""
    from tests import gpu_helpers as G
    from transformerupscaler_b200 import _lib
    from transformerupscaler_b200.packing import PackedWeights
    lib = _lib.load()
    pw = PackedWeights(model, synth_state_dict(model, 5), BF16, dev)
    dim, T = pw.dim, 297
    x = torch.from_numpy(np.random.RandomState(23).standard_normal((T * 128, dim)).astype(np.float32)).to(dev)
    alone = torch.cat([G.window_stack(x[t * 128:(t + 1) * 128].clone(), pw) for t in range(T)])
    for n in (1, 2, 147, 148, 149, 297):
        out = G.window_stack(x[:n * 128].clone(), pw)
        assert torch.equal(out, alone[:n * 128]), n
    base = G.window_stack(x.clone(), pw)
    assert torch.equal(G.window_stack(x.clone(), pw), base)
    try:
        for key, val in ((b"snake", 4), (b"stack_var", 1)):
            lib.tu_debug_set(key, val)
            assert torch.equal(G.window_stack(x.clone(), pw), base), key
            lib.tu_debug_set(key, 0)
    finally:
        lib.tu_debug_set(b"snake", 0)
        lib.tu_debug_set(b"stack_var", 0)


@pytest.mark.parametrize("regime", ["default", "offset"])
@pytest.mark.parametrize("M", [1, 128, 130, 328, 3600, 7200])
def test_residual_block_kernels_vs_bf16_reference(dev, M, regime):
    """tu_resid_pre (LN1 + in_proj -> bf16 q | k | v) and tu_resid_post (out_proj, LN2, MLP, both residual adds) of one
    ResidualTransformer layer (R:22-50) vs the bf16-store reference, with partial last tiles; the 128 rows after M must stay
    untouched in the token stream and in qkv"""
    from tests import gpu_helpers as G
    from transformerupscaler_b200 import _lib
    from transformerupscaler_b200.packing import PackedWeights
    lib = _lib.load()
    sd = synth_state_dict("ResidualTransformer", 6)
    pw = PackedWeights("ResidualTransformer", sd, BF16, dev)
    x, off = regime_tokens(M, 128, regime, seed=M)
    att = torch.from_numpy(np.random.RandomState(M + 1).standard_normal((M, 128)).astype(np.float32) * 0.5).to(BF16)
    nan = float("nan")
    tok = torch.full((M + 128, 128), nan, device=dev)
    tok[:M] = x.to(dev)
    qkv = torch.full((M + 128, 384), nan, dtype=BF16, device=dev)
    atts = torch.full((M + 128, 128), nan, dtype=BF16, device=dev)
    atts[:M] = att.to(dev)
    for layer in (0, pw.n_blocks - 1):
        pre = f"transformer_blocks.{layer}."
        G.chk(lib.tu_resid_pre(G.p(tok), G.p(qkv), C.byref(pw.struct), layer, M, G.stream()))
        torch.cuda.synchronize()
        assert torch.equal(tok[:M].cpu(), x) and tok[M:].isnan().all().item()
        assert qkv[M:].isnan().all().item()
        check("resid_pre", regime, qkv[:M], br.resid_pre(x, sd, pre), torch.zeros(M))
        t2 = tok.clone()
        G.chk(lib.tu_resid_post(G.p(t2), G.p(atts), C.byref(pw.struct), layer, M, G.stream()))
        torch.cuda.synchronize()
        assert t2[M:].isnan().all().item()
        check("resid_post", regime, t2[:M], br.resid_post(x, att.double(), sd, pre), off)
