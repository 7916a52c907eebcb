"""CPU: the oracle restatement vs golden vectors produced by the unmodified reference modules."""
import os

import numpy as np
import pytest
import torch

from oracle import upscaler_oracle as orc
from oracle.weights import synth_state_dict, synth_frames
from tests.golden.cases import CASES, FULLSIZE, sample_fullsize

GOLD = os.path.join(os.path.dirname(__file__), "golden")
# fp32 oracle vs fp32 reference: both are fp32 evaluations of the same graph with different
# summation orders; the bicubic tap arithmetic is restated bit-for-bit.  Tolerance in the test:
TOL_FP32 = 2e-5


def load_case(name):
    c = CASES[name]
    B, _, H, W = c["shape"]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    return c, synth_state_dict(c["model"], c["wseed"], c.get("gain", 1.0)), synth_frames(B, H, W, seed=c["xseed"]), g


@pytest.mark.parametrize("name", [n for n in CASES if CASES[n]["shape"][2] < 400])
def test_oracle_matches_reference_golden(name):
    c, sd, x, g = load_case(name)
    pre = orc.forward(c["model"], sd, x, pre_clamp=True, **c["kw"]).numpy()
    assert tuple(g["shape"]) == pre.shape
    st = c.get("stride", 1)
    err = np.abs(pre[..., ::st, ::st] - g["pre"]).max()
    assert err < TOL_FP32, f"{name}: max-abs {err}"
    out = orc.forward(c["model"], sd, x, **c["kw"]).numpy()
    assert out.min() >= 0.0 and out.max() <= 1.0


def test_oracle_residual_720p_golden():
    c, sd, x, g = load_case("residual_720p_1080p")
    pre = orc.forward(c["model"], sd, x, pre_clamp=True, **c["kw"]).numpy()
    err = np.abs(pre[..., ::8, ::8] - g["pre"]).max()
    assert err < 1e-4, f"max-abs {err}"      # 8 global-attention blocks over 3600 tokens in fp32


def test_oracle_error_behaviour():
    sd = synth_state_dict("FastTransformer", 0)
    with pytest.raises(ValueError, match="was not built"):
        orc.fast_forward(sd, torch.rand(1, 3, 16, 16), upscale_factor=5)
    sdr = synth_state_dict("ResidualTransformer", 0)
    with pytest.raises(RuntimeError, match="must match"):
        orc.residual_forward(sdr, torch.rand(1, 3, 64, 64))


@pytest.mark.parametrize("name", ["natural_window_96x176_r1p5", "natural_fast_96x176_x2"])
def test_oracle_matches_reference_on_natural_image(name):
    """LR/HR pair cut from one of the reference's training images (tests/golden/make_natural.py); the stored reference
    output is fp16, hence the looser bound"""
    from tests.golden.cases import NATURAL
    c = NATURAL[name]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    x = torch.from_numpy(g["lr_u8"]).float().div(255.0).unsqueeze(0)
    out = orc.forward(c["model"], synth_state_dict(c["model"], c["wseed"]), x, **c["kw"])[0].numpy()
    ref = g["ref"].astype(np.float32)
    assert out.shape == ref.shape == g["hr_u8"].shape
    assert np.abs(out - ref).max() < 6e-4          # fp16 storage of values in [0, 1]: half-ulp 2.4e-4


def _ragged_cases():
    from tests.test_gpu_models import _ragged_cases as rc
    return rc()


@pytest.mark.parametrize("model,shape,kw,seed", _ragged_cases())
def test_oracle_matches_live_reference_on_ragged_shapes(model, shape, kw, seed):
    """the same seeded sweep of awkward shapes the GPU suite runs, here the oracle against the reference: always against the stored
    sweep (tests/golden/ragged_<k>.npz, tests/golden/make_ragged.py: the oracle arithmetic that matched the reference on every case
    of the sweep to TOL_FP32, on a coprime-stride lattice plus the corners), and against the UNMODIFIED reference modules executed
    live whenever a copy of the reference's models/ is in baseline/_ref (python baseline/fetch_ref.py <reference checkout>)"""
    import sys
    from tests.golden.cases import ragged_sample
    B, H, W = shape
    sd = synth_state_dict(model, seed)
    x = synth_frames(B, H, W, seed=seed + 100)
    k = _ragged_cases().index((model, shape, kw, seed))
    g = np.load(os.path.join(GOLD, f"ragged_{k:02d}.npz"))
    assert (str(g["model"]), int(g["seed"]), str(g["kw"])) == (model, seed, repr(sorted(kw.items())))
    pre = orc.forward(model, sd, x, pre_clamp=True, **kw).numpy()
    assert tuple(g["shape"]) == pre.shape
    st, lat, crops = ragged_sample(pre)
    assert st == int(g["stride"])
    err = max([np.abs(lat - g["pre"]).max()] + [np.abs(cr - g[f"crop{i}"]).max() for i, cr in enumerate(crops)])
    assert err < TOL_FP32, (model, shape, kw, err)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref_dir = os.path.join(root, "baseline", "_ref", "models")
    if not os.path.isdir(os.path.join(ref_dir, model)):
        return
    if root not in sys.path:
        sys.path.insert(0, root)
    from baseline.refload import reference_model_class
    M = reference_model_class(ref_dir, model)().eval()
    M.load_state_dict(sd, strict=True)
    with torch.no_grad():
        ref = M(x, **kw)
    out = orc.forward(model, sd, x, **kw)
    assert tuple(out.shape) == tuple(ref.shape)
    assert (out - ref).abs().max().item() < TOL_FP32, (model, shape, kw)


_FULL_DEFAULT = ("window_720p_1080p_b8", "fast_720p_x2", "residual_720p_4k", "fast_720p_res1080p")


@pytest.mark.parametrize("name", list(FULLSIZE))
def test_oracle_matches_reference_at_baseline_sizes(name):
    """BASELINE.json's configurations at their real sizes (first stored frame): the oracle against the unmodified reference's
    pre-clamp output on the stride-13 lattice and the corner crops.  The x3 / x4 / x6 / 1080p cases take 15-60 s and up to 20 GB
    each on CPU and run with TU_FULLSIZE_ORACLE=1 (they passed in the build container when the fixtures were made)."""
    if name not in _FULL_DEFAULT and not os.environ.get("TU_FULLSIZE_ORACLE"):
        pytest.skip("set TU_FULLSIZE_ORACLE=1 to run the large oracle cases")
    c = dict(FULLSIZE[name])
    B, _, H, W = c["shape"]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    sd = synth_state_dict(c["model"], c["wseed"])
    x = synth_frames(B, H, W, seed=c["xseed"])[:1]
    pre = orc.forward(c["model"], sd, x, pre_clamp=True, **c["kw"]).numpy()
    c["frames"] = (0,)
    lat, crops = sample_fullsize(pre, c)
    err = max([np.abs(lat - g["pre"][:1]).max()] + [np.abs(cr - g[f"crop{i}"][:1]).max() for i, cr in enumerate(crops)])
    assert err < TOL_FP32, f"{name}: max-abs {err}"
