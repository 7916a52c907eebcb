"""GPU: the reference's own entry points, UNMODIFIED (baseline/_ref/speed_test.py and inference.py, verbatim copies made by
baseline/fetch_ref.py), executed against this repository's drop-in `models/` package: importlib.import_module("models.<M>.model")
resolves to the engine (a regular package wins over the reference's namespace directories), the checkpoint is a state_dict with the
reference's keys, and the call patterns are the scripts' own -- speed_test.py:60-67 (`model(lr_img, res_out=(2160, 3840))` over
its 200-item dataset of ten LR/HR scale pairs) and inference.py:117-123 (`torch.autocast(float16)` + `upscale_factor=`)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from PIL import Image

from oracle.weights import synth_state_dict

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")


def _env(extra=()):
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, REF, *extra, env.get("PYTHONPATH", "")])
    return env


def _need(script):
    # the reference's sources are not part of this repository: without a copy in baseline/_ref there is nothing to run
    if not os.path.exists(os.path.join(REF, script)):
        pytest.skip(f"needs the reference's {script} in baseline/_ref (python baseline/fetch_ref.py <reference checkout>)")


def _png(path, h, w, seed):
    rs = np.random.RandomState(seed)
    yy, xx = np.meshgrid(np.linspace(0, 1, h), np.linspace(0, 1, w), indexing="ij")
    img = np.stack([0.5 + 0.4 * np.sin(6.28 * (rs.uniform(1, 4) * xx + rs.uniform(1, 4) * yy)) for _ in range(3)], -1)
    Image.fromarray((img * 255).astype(np.uint8)).save(path)


@pytest.mark.parametrize("model,shape,kw,autocast_fp16", [
    ("WindowTransformer", (90, 160), dict(res_out=(2160, 3840)), False),      # speed_test.py:60-67
    ("FastTransformer", (120, 200), dict(upscale_factor=3), True),             # inference.py:117-123
    ("FastTransformer", (120, 200), dict(upscale_factor=4), True),
    ("WindowTransformer", (120, 200), dict(upscale_factor=2), True)])
def test_reference_call_patterns_run_on_the_drop_in_models(tmp_path, model, shape, kw, autocast_fp16):
    """The scripts' call patterns without the scripts (the two tests below run the reference's own files when they are present):
    the class found through importlib.import_module("models.<M>.model"), a checkpoint saved as a state_dict with the reference's
    keys and loaded with torch.load(map_location=device), then model(lr, res_out=(2160, 3840)) under no_grad, or
    model(x, upscale_factor=s) under torch.autocast(float16); the result against the CPU oracle."""
    import importlib
    from oracle import upscaler_oracle as orc
    from oracle.weights import synth_frames
    ckpt = tmp_path / "model_epoch_1.pth"
    torch.save(synth_state_dict(model, 5), str(ckpt))
    cls = importlib.import_module(f"models.{model}.model").TransformerModel
    assert cls.__module__.startswith("transformerupscaler_b200.")
    M = cls().to("cuda")
    M.load_state_dict(torch.load(str(ckpt), map_location="cuda"))
    M.eval()
    x = synth_frames(1, *shape, seed=6)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16, enabled=autocast_fp16):
        y = M(x.cuda(), **kw)
    ref = orc.forward(model, synth_state_dict(model, 5), x, **kw)
    assert tuple(y.shape) == tuple(ref.shape)
    # under autocast the reference's FastTransformer ends in convs (low-precision output); the other two end in fp32 ops
    assert y.dtype == (torch.float16 if autocast_fp16 and model == "FastTransformer" else torch.float32)
    assert (y.float().cpu() - ref).abs().max().item() < (2e-2 if autocast_fp16 else 1e-4)


def test_reference_speed_test_script_runs_on_the_drop_in_models(tmp_path):
    _need("speed_test.py")
    data = tmp_path / "data"
    ckpt = tmp_path / "ckpt"
    data.mkdir(); ckpt.mkdir()
    for i in range(20):                       # the dataset's hard-coded len 200 = 20 images x 10 scale pairs (data_class.py:47-50)
        _png(str(data / f"image_{i}.png"), 90, 160, i)
    torch.save(synth_state_dict("WindowTransformer", 3), str(ckpt / "model_epoch_7.pth"))
    r = subprocess.run([sys.executable, os.path.join(REF, "speed_test.py"), "--model", "WindowTransformer", "--data_dir", str(data),
                        "--checkpoint_dir", str(ckpt)], cwd=str(tmp_path), env=_env(), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "Processing 200 images" in r.stdout and "Average inference time per image" in r.stdout
    assert "model_epoch_7.pth" in r.stdout


@pytest.mark.parametrize("model,scale", [("FastTransformer", 3), ("FastTransformer", 4), ("WindowTransformer", 2)])
def test_reference_inference_script_runs_on_the_drop_in_models(tmp_path, model, scale):
    _need("inference.py")
    ckpt = tmp_path / "ckpt"
    ckpt.mkdir()
    _png(str(tmp_path / "in.png"), 120, 200, 5)
    torch.save(synth_state_dict(model, 4), str(ckpt / "model_epoch_2.pth"))
    r = subprocess.run([sys.executable, os.path.join(REF, "inference.py"), "--image_path", str(tmp_path / "in.png"), "--model", model,
                        "--checkpoint_dir", str(ckpt), "--scale", str(scale), "--inp", str(tmp_path / "input.jpg"),
                        "--out", str(tmp_path / "model.jpg")], cwd=str(tmp_path),
                       env=_env([os.path.join(ROOT, "tests", "stubs")]), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "Running inference on device: cuda" in r.stdout and "Model Scores" in r.stdout
    out = Image.open(str(tmp_path / "model.jpg"))
    assert out.size == (200 * scale, 120 * scale)
    # the JPEG the script wrote is the engine's output: compare with a direct call of the drop-in class on the same tensor
    import importlib
    import torchvision.transforms as T
    M = importlib.import_module(f"models.{model}.model").TransformerModel().to("cuda")
    M.load_state_dict(torch.load(str(ckpt / "model_epoch_2.pth"), map_location="cuda"))
    M.eval()
    x = T.ToTensor()(Image.open(str(tmp_path / "in.png")).convert("RGB")).unsqueeze(0).cuda()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        y = M(x, upscale_factor=scale)
    # through the same JPEG encoder the script used (random-init weights give noisy images: the codec's loss is large, so the
    # comparison is between two encodings of what must be the same pixels)
    import io
    bio = io.BytesIO()
    T.ToPILImage()(y.squeeze(0).float().cpu()).save(bio, "JPEG")
    want = np.asarray(Image.open(io.BytesIO(bio.getvalue())).convert("RGB")).astype(np.float64)
    got = np.asarray(out.convert("RGB")).astype(np.float64)
    assert np.abs(got - want).mean() < 0.5
