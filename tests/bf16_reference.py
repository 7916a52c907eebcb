"""TEST INFRASTRUCTURE ONLY -- the transformer blocks of the bf16 tensor-core kernels, restated in float64 with each kernel's bf16
stores (round to nearest even) inserted where the kernel makes them.

Built on :mod:`oracle.upscaler_oracle` (``layer_norm``, ``linear``, ``gelu_erf``, ``dense_rel_bias``): with ``rounding=False`` every
function here is the oracle's block in float64.  With ``rounding=True`` the 2-D weights are rounded to bf16 (the kernels' weight
operands; LayerNorm parameters, biases and the relative-position tables stay fp32) and the activations are rounded where the
kernels store bf16:

  tc/window_stack_tcgen05.cu (dim 128)                 tc/window_stack192_tcgen05.cu (dim 192)
    LN1 / LN2 output        layernorm_to_a32 :182          layernorm_to_a32 :217
    qkv + bias (q x 0.25)   :426-429                       :476-479 (one head pair at a time)
    probabilities           :494-497 (the row sum is the   :536-539 (same)
                            ones-column MMA :506 over the
                            rounded probabilities)
    attention output x 1/l  :515-516                       :557-558
    GELU output             :547-551 (TMEM)                :590-595 (even chunks TMEM, odd chunks shared memory: both bf16)
  tc/residual_block_tcgen05.cu (ResidualTransformer, dim 128)
    pre:  LN1 output :118, in_proj + bias (q x 0.25) -> bf16 qkv rows :279-282
    post: attention output arrives as bf16; LN2 output :118, GELU output :336-339
The residual stream (TMEM in the fused kernels, the fp32 token buffer elsewhere) is not rounded here: it stays float64.  The kernels
keep it in fp32 with the proj / fc2 biases folded into offset vectors; that, the summation order of the fp32 accumulators, the fitted
tanh GELU, ex2 / rcp / tanh ``.approx`` and the LayerNorm statistics are NOT emulated: the test tolerances absorb them, so that a
reordering of the kernel's arithmetic passes and a wrong index, coefficient or statistic does not.

The per-block bf16 path (transformer_simt.cu::transformer_block_impl: layernorm_kernel, tc_linear, window_attn_mma_kernel,
global_attn_mma_kernel) stores bf16 at the same points, with one difference: window_attn_mma_kernel takes the softmax row sum over
the fp32 probabilities before they are rounded (transformer_simt.cu:156-157), where the fused stack sums the rounded ones.
``rowsum_rounded=False`` selects that.  global_attn_mma_kernel sums the rounded probabilities (ones-column MMA, :360) relative to a
running maximum; the emulation takes them relative to the row maximum.
"""
from __future__ import annotations

import torch

from oracle import upscaler_oracle as orc

F64 = torch.float64


def bf16(t: torch.Tensor) -> torch.Tensor:
    """round to the nearest bf16 (ties to even), kept in t's dtype"""
    return t.to(torch.bfloat16).to(t.dtype)


def _ident(t: torch.Tensor) -> torch.Tensor:
    return t


def _w(sd, name: str, r) -> torch.Tensor:
    return r(sd[name].detach().to("cpu", F64))


def _v(sd, name: str) -> torch.Tensor:
    return sd[name].detach().to("cpu", F64)


def _attention(q, k, v, bias, r, rowsum_rounded: bool) -> torch.Tensor:
    """softmax(q k^T + bias) v over the last two axes; q already scaled; probabilities relative to the row maximum"""
    s = q.matmul(k.transpose(-2, -1))
    if bias is not None:
        s = s + bias
    e = torch.exp(s - s.amax(-1, keepdim=True))
    p = r(e)
    l = (p if rowsum_rounded else e).sum(-1, keepdim=True)
    return r(p.matmul(v) / l)


def _mlp(x, sd, pre: str, r, eps: float, gelu) -> torch.Tensor:
    h = r(orc.layer_norm(x, _v(sd, pre + "norm2.weight"), _v(sd, pre + "norm2.bias"), eps))
    h = r(gelu(orc.linear(h, _w(sd, pre + "mlp.0.weight", r), _v(sd, pre + "mlp.0.bias"))))
    return x + orc.linear(h, _w(sd, pre + "mlp.2.weight", r), _v(sd, pre + "mlp.2.bias"))


def window_block(x: torch.Tensor, sd, pre: str, heads: int, rounding: bool = True, rowsum_rounded: bool = True,
                 eps: float = 1e-5, gelu=orc.gelu_erf) -> torch.Tensor:
    """One WindowTransformerBlock on (nWin, 64, dim) tokens, float64 (orc.window_block with the kernels' bf16 stores)."""
    r = bf16 if rounding else _ident
    x = x.to(F64)
    nW, N, D = x.shape
    hd = D // heads
    h = r(orc.layer_norm(x, _v(sd, pre + "norm1.weight"), _v(sd, pre + "norm1.bias"), eps))
    qkv = orc.linear(h, _w(sd, pre + "attn.qkv.weight", r), _v(sd, pre + "attn.qkv.bias"))
    qkv = r(qkv.reshape(nW, N, 3, heads, hd).permute(2, 0, 3, 1, 4))
    q, k, v = qkv[0] * hd ** -0.5, qkv[1], qkv[2]          # hd = 16: the scale is a power of two, exact after rounding
    bias = orc.dense_rel_bias(_v(sd, pre + "attn.relative_position_bias_table"))[None]
    o = _attention(q, k, v, bias, r, rowsum_rounded).transpose(1, 2).reshape(nW, N, D)
    x = x + orc.linear(o, _w(sd, pre + "attn.proj.weight", r), _v(sd, pre + "attn.proj.bias"))
    return _mlp(x, sd, pre, r, eps, gelu)


def window_stack(x: torch.Tensor, sd, heads: int, n_blocks: int, rounding: bool = True, prefix: str = "window_blocks.",
                 **kw) -> torch.Tensor:
    """all blocks of the fused window stack on (nWin, 64, dim) tokens"""
    x = x.to(F64)
    for b in range(n_blocks):
        x = window_block(x, sd, f"{prefix}{b}.", heads, rounding, **kw)
    return x


def resid_pre(x: torch.Tensor, sd, pre: str, rounding: bool = True, eps: float = 1e-5) -> torch.Tensor:
    """ResidualTransformer layer, first kernel: (M, 128) tokens -> (M, 384) q | k | v with q scaled by head_dim^-0.5 (bf16 values)"""
    r = bf16 if rounding else _ident
    D = x.shape[-1]
    h = r(orc.layer_norm(x.to(F64), _v(sd, pre + "norm1.weight"), _v(sd, pre + "norm1.bias"), eps))
    qkv = orc.linear(h, _w(sd, pre + "attn.in_proj_weight", r), _v(sd, pre + "attn.in_proj_bias"))
    qkv[..., :D] *= 0.25
    return r(qkv)


def resid_post(x: torch.Tensor, att: torch.Tensor, sd, pre: str, rounding: bool = True, eps: float = 1e-5,
               gelu=orc.gelu_erf) -> torch.Tensor:
    """ResidualTransformer layer, second kernel: x + out_proj(att), then the MLP half of the block; att (M, 128) as the kernel reads it"""
    r = bf16 if rounding else _ident
    x = x.to(F64) + orc.linear(att.to(F64), _w(sd, pre + "attn.out_proj.weight", r), _v(sd, pre + "attn.out_proj.bias"))
    return _mlp(x, sd, pre, r, eps, gelu)


def global_attention(qkv: torch.Tensor, heads: int, rounding: bool = True) -> torch.Tensor:
    """(B, S, 3 dim) q | k | v with q pre-scaled -> (B, S, dim) attention output (nn.MultiheadAttention's core)"""
    r = bf16 if rounding else _ident
    B, S, D3 = qkv.shape
    D = D3 // 3
    q, k, v = [t.reshape(B, S, heads, D // heads).transpose(1, 2) for t in qkv.to(F64).split(D, dim=-1)]
    return _attention(q, k, v, None, r, True).transpose(1, 2).reshape(B, S, D)


def mha_block(x: torch.Tensor, sd, pre: str, heads: int, rounding: bool = True, eps: float = 1e-5, gelu=orc.gelu_erf) -> torch.Tensor:
    """ResidualTransformer TransformerBlock on (B, S, dim) tokens, float64 (orc.mha_block with the kernels' bf16 stores)"""
    qkv = resid_pre(x, sd, pre, rounding, eps)
    att = global_attention(qkv, heads, rounding)
    return resid_post(x, att, sd, pre, rounding, eps, gelu)
