"""CPU: tests/bf16_reference.py, the reference the fused transformer kernels are tested against (tests/test_gpu_transformer_kernels.py).

With its bf16 stores switched off it must be the oracle's block; with them on, each planted bug below must move its output by at least
five times the GPU test's bound for that output, so that a kernel with the bug could not pass.

Not in the table: GELU in its tanh form instead of the erf form.  It moves one block by 1.3e-4 mean, one ResidualTransformer MLP half
(tu_resid_post) by the same, and the kernels' own GELU -- a fitted polynomial under tanh.approx, whose 2^-11 relative error is the
larger part -- already sits 1e-4 mean from the erf form there (measured on a B200): the two are not separable at the bf16 outputs.
"""
import numpy as np
import pytest
import torch

from oracle import upscaler_oracle as orc
from oracle.weights import synth_state_dict
from tests import bf16_reference as br
from tests.test_gpu_transformer_kernels import TOL, regime_sd, regime_tokens, rel_err

F64 = torch.float64
WINDOW_MODELS = ["WindowTransformer", "FastTransformer"]


def _heads(sd):
    return sd["window_blocks.0.attn.relative_position_bias_table"].shape[1]


@pytest.mark.parametrize("model", WINDOW_MODELS)
def test_rounding_off_is_the_oracle_window_block(model):
    sd = synth_state_dict(model, 5)
    heads = _heads(sd)
    x = torch.from_numpy(np.random.RandomState(3).standard_normal((3, 64, 16 * heads)))
    for b in (0, 1):
        pre = f"window_blocks.{b}."
        want = orc.window_block(x, sd, pre, heads, F64)
        for rowsum_rounded in (True, False):
            got = br.window_block(x, sd, pre, heads, rounding=False, rowsum_rounded=rowsum_rounded)
            assert (got - want).abs().max().item() < 1e-12
        assert (br.window_block(x, sd, pre, heads) - want).abs().max().item() > 1e-4      # the stores do round


def test_rounding_off_is_the_oracle_mha_block():
    sd = synth_state_dict("ResidualTransformer", 6)
    x = torch.from_numpy(np.random.RandomState(4).standard_normal((2, 150, 128)))
    pre = "transformer_blocks.1."
    want = orc.mha_block(x, sd, pre, 8, F64)
    assert (br.mha_block(x, sd, pre, 8, rounding=False) - want).abs().max().item() < 1e-12
    qkv = br.resid_pre(x, sd, pre)
    assert torch.equal(qkv, br.bf16(qkv))                      # the pre kernel's output is bf16
    assert (br.mha_block(x, sd, pre, 8) - want).abs().max().item() > 1e-4


def _swap_qk_heads(sd, pre, dim, h):
    """q and k rows of head h exchanged with those of head h + 1"""
    k = pre + "attn.qkv.weight"
    w, src = sd[k].clone(), sd[k]
    for base in (0, dim):
        a, b = base + 16 * h, base + 16 * (h + 1)
        w[a:a + 16], w[b:b + 16] = src[b:b + 16], src[a:a + 16]
    return {**sd, k: w}


def _transpose_table(sd, pre, h):
    """head h's relative-position bias transposed: the table read at the negated offset"""
    k = pre + "attn.relative_position_bias_table"
    t = sd[k].clone()
    t[:, h] = sd[k].flip(0)[:, h]
    return {**sd, k: t}


def _tanh_gelu(z):
    return torch.nn.functional.gelu(z, approximate="tanh")


# bug -> (regime whose weights make it visible, how it is planted into block `pre` of a state dict (`nxt`: the prefix of the block
# after it in the model) / into the reference's arguments)
BUGS = {
    "transposed rel-pos bias, head 3": ("table30", lambda sd, pre, nxt, dim: (_transpose_table(sd, pre, 3), {})),
    "block b+1's bias table in block b": ("table30", lambda sd, pre, nxt, dim: (
        {**sd, pre + "attn.relative_position_bias_table": sd[nxt + "attn.relative_position_bias_table"]}, {})),
    "LayerNorm eps 1e-6": ("offset", lambda sd, pre, nxt, dim: (sd, {"eps": 1e-6})),
    "LN1 gamma shifted by one channel": ("default", lambda sd, pre, nxt, dim: (
        {**sd, pre + "norm1.weight": torch.roll(sd[pre + "norm1.weight"], 1)}, {})),
    "q/k of head 3 swapped with head 4": ("default", lambda sd, pre, nxt, dim: (_swap_qk_heads(sd, pre, dim, 3), {})),
}


@pytest.mark.parametrize("bug", list(BUGS))
@pytest.mark.parametrize("model", WINDOW_MODELS)
def test_planted_bugs_exceed_the_gpu_bounds(model, bug, capsys):
    """one block (block 0) as the GPU test runs it alone through the stack kernel: the bug moves the reference's output by >= 5x the
    bound on the max or on the mean error.  Also reported: how far the bug moves the whole stack, against the old bound of the
    stack test (absolute max 0.15, mean 1.5e-2 against the oracle with bf16 weights), which let most of them through."""
    regime, plant = BUGS[bug]
    sd = regime_sd(model, regime)
    heads, dim = _heads(sd), 16 * _heads(sd)
    nb = orc._n_blocks(sd, "window_blocks.")
    x, off = regime_tokens(6 * 64, dim, regime, seed=21)
    x = x.reshape(6, 64, dim)
    good = br.window_block(x, sd, "window_blocks.0.", heads)
    bad_sd, kw = plant(sd, "window_blocks.0.", "window_blocks.1.", dim)
    bad = br.window_block(x, bad_sd, "window_blocks.0.", heads, **kw)
    smax, smean = rel_err(bad.reshape(-1, dim), good, off)
    tmax, tmean = TOL[f"block{dim}"][regime]
    # the same bug in every block of the whole stack, against the old bound
    bad_all, kw_all = sd, {}
    for b in range(nb - 1 if "b+1" in bug else nb):
        bad_all, kw_all = plant(bad_all, f"window_blocks.{b}.", f"window_blocks.{b + 1}.", dim)
    stack_good = br.window_stack(x, sd, heads, nb)
    d = (br.window_stack(x, bad_all, heads, nb, **kw_all) - stack_good).abs()
    old_caught = d.max().item() > 0.15 or d.mean().item() > 1.5e-2
    with capsys.disabled():
        print(f"\n{model} {bug} [{regime}]: one block max {smax:.2e} ({smax / tmax:.1f}x bound) mean {smean:.2e} "
              f"({smean / tmean:.1f}x bound); whole stack max {d.max().item():.2e} mean {d.mean().item():.2e}: "
              f"{'caught' if old_caught else 'passed'} by the old stack bound")
    assert smax >= 5 * tmax or smean >= 5 * tmean, (smax, smean, tmax, tmean)

