"""CPU: fp16 image I/O (TU_F16) at the C ABI and the host-side facts it rests on: the dtype code, fp16 rejected as a compute dtype,
the fp16 clamp-and-store identity of the row-schedule bicubic kernel (transformerupscaler_b200/csrc/resample.cu, clamp_store_pair<f16>)
and the packing of an fp16 state dict."""
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from transformerupscaler_b200 import _lib
    return _lib.load()


def test_f16_code_in_header_and_binding():
    from transformerupscaler_b200 import _lib, engine
    src = open(os.path.join(ROOT, "include", "tu_b200.h")).read()
    assert re.search(r"#define\s+TU_F16\s+3\b", src)
    assert _lib.TU_F16 == 3
    assert engine._DT[torch.float16] == _lib.TU_F16 and engine._TORCH_DT[_lib.TU_F16] == torch.float16


def test_f16_is_not_a_compute_dtype(lib):
    from transformerupscaler_b200 import _lib
    for model in (0, 1, 2):
        assert lib.tu_forward_workspace_bytes(model, 1, 720, 1280, 1080, 1920, 2, _lib.TU_F16) == 0
        assert "compute dtype" in _lib.last_error()
    w = _lib.TuModelWeights()
    w.model, w.dim, w.heads, w.n_blocks = 0, 128, 8, 8
    import ctypes as C
    assert lib.tu_forward_workspace_bytes_for(C.byref(w), 1, 72, 104, 108, 156, 0, _lib.TU_F16) == 0
    assert lib.tu_forward_workspace_bytes_for(C.byref(w), 1, 72, 104, 108, 156, 0, _lib.TU_BF16) > 0


def _dense_f16_neighbourhood():
    """every finite fp16 value, the fp32 midpoints between neighbouring fp16 values and the fp32 values one ulp either side of
    them (the round-to-nearest-even ties and near-ties), +-0, fp16 subnormals, values around 1 and fp32 extremes"""
    h = np.arange(0, 1 << 16, dtype=np.uint32).astype(np.uint16).view(np.float16)
    h = np.sort(h[np.isfinite(h)].astype(np.float32))
    mid = ((h[:-1].astype(np.float64) + h[1:].astype(np.float64)) / 2).astype(np.float32)
    extra = np.array([0.0, -0.0, 1.0, 1.0 - 2**-12, 1.0 + 2**-11, 1.0 + 2**-12, 1.0 - 2**-11, 2**-24, 2**-25, -2**-25, 2**-14,
                      65504.0, 65520.0, 3.0e38, -3.0e38, 2**-140, -2**-140], dtype=np.float32)
    v = np.concatenate([h, mid, np.nextafter(mid, np.float32(np.inf)), np.nextafter(mid, np.float32(-np.inf)), extra])
    return torch.from_numpy(v)


def test_f16_relu_then_min_equals_clamp_then_round():
    """cvt.rn.relu.f16x2.f32 + min.f16x2 with 1.0 == round-to-fp16(clamp(v, 0, 1)): rounding is monotonic and 0, 1 are fp16 values"""
    v = _dense_f16_neighbourhood()
    want = v.clamp(0, 1).to(torch.float16)
    relu_rounded = torch.where(v > 0, v, torch.zeros_like(v)).to(torch.float16)          # relu: negatives (and -0) become +0
    got = torch.minimum(relu_rounded, torch.tensor(1.0, dtype=torch.float16))
    nz = want.float() != 0
    assert torch.equal(got.view(torch.int16)[nz], want.view(torch.int16)[nz])              # bit patterns, not values
    assert torch.equal(got.float()[~nz], want.float()[~nz])                                # zeros: +0 here, torch.clamp keeps -0


def test_f16_widening_is_exact_and_rounding_once_commutes_with_clamp():
    """the two facts the fp16 I/O path stands on: fp16 -> fp32 never rounds, and round(clamp(v)) == clamp(round(v))"""
    v = _dense_f16_neighbourhood()
    h = v[torch.isfinite(v.to(torch.float16))].to(torch.float16)
    assert torch.equal(h.float().to(torch.float16).view(torch.int16), h.view(torch.int16))
    a = v.clamp(0, 1).to(torch.float16)
    b = v.to(torch.float16).clamp(0, 1)
    assert torch.equal(a.float(), b.float())


@pytest.mark.parametrize("model", ["WindowTransformer", "FastTransformer", "ResidualTransformer"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_fp16_state_dict_packs_to_the_bytes_of_its_fp32_upcast(model, dtype):
    """PackedWeights (bf16 slabs, fp64 folds, fragment-ordered bias, pos_embed) and the host arrays CPackedWeights hands to
    tu_pack_weights: an fp16 state dict gives the bytes its fp32 upcast gives"""
    from oracle.weights import synth_state_dict
    from transformerupscaler_b200.packing import PackedWeights
    sd16 = {k: (v.half() if v.is_floating_point() else v) for k, v in synth_state_dict(model, 3).items()}
    sd32 = {k: (v.float() if v.is_floating_point() else v) for k, v in sd16.items()}
    a = PackedWeights(model, sd16, dtype, torch.device("cpu"))
    b = PackedWeights(model, sd32, dtype, torch.device("cpu"))
    assert len(a.keep) == len(b.keep)
    for x, y in zip(a.keep, b.keep):
        assert x.dtype == y.dtype and x.shape == y.shape
        assert torch.equal(x.reshape(-1).view(torch.uint8), y.reshape(-1).view(torch.uint8))
    # CPackedWeights' host side: every tensor becomes an fp32 (int64 index) host array before tu_pack_weights sees it
    for k in sd16:
        h16 = sd16[k].detach().to("cpu", torch.int64 if sd16[k].dtype == torch.int64 else torch.float32)
        assert torch.equal(h16, sd32[k].to(h16.dtype))
