"""CPU: host-side mirror of the reference interface — state_dict compatibility, precision selection, the shape logic
of the three forwards, error behaviour, and frame sharding over a 2-rank gloo group."""
import importlib
import os

import pytest
import torch

from oracle.weights import _spec, synth_state_dict

MODELS = ["WindowTransformer", "FastTransformer", "ResidualTransformer"]


def make(name):
    return importlib.import_module(f"transformerupscaler_b200.models.{name}.model").TransformerModel()


@pytest.mark.parametrize("name", MODELS)
def test_state_dict_keys_and_shapes_match_reference_spec(name):
    m = make(name)
    sd = m.state_dict()
    spec = {k: tuple(shape) for k, shape, _, _ in _spec(name)}
    assert set(sd) == set(spec)
    for k, v in sd.items():
        assert tuple(v.shape) == spec[k], k
    m.load_state_dict(synth_state_dict(name, 3), strict=True)
    # root-level drop-in alias used by importlib.import_module(f"models.{name}.model")
    alias = importlib.import_module(f"models.{name}.model").TransformerModel
    assert alias is type(m)


@pytest.mark.parametrize("name", MODELS)
def test_cpu_tensor_and_training_mode_are_rejected(name):
    m = make(name)
    with pytest.raises(RuntimeError, match="forward-only"):
        m(torch.rand(1, 3, 32, 32))
    m.eval()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(torch.rand(1, 3, 32, 32))


def test_fast_forward_shape_logic(monkeypatch):
    from transformerupscaler_b200 import engine
    calls = []

    def fake_forward(x, handle, oh, ow, scale, cbf, obf, clamp, in_layout=0):
        calls.append(("fwd", oh, ow, scale, clamp))
        return torch.zeros(x.shape[0], 3, oh, ow)

    def fake_resize(x, oh, ow, clamp, out_code=-1):
        calls.append(("resize", oh, ow, clamp))
        return torch.zeros(x.shape[0], 3, oh, ow)

    monkeypatch.setattr(engine, "tu_forward", fake_forward)
    monkeypatch.setattr(engine, "tu_resize_aa", fake_resize)
    x = torch.zeros(1, 3, 40, 56)
    # upscale_factor overrides res_out; no resize because the size already matches
    out = engine.run_forward(1, "FastTransformer", x, (1080, 1920), 3, True, False, torch.float32)
    assert tuple(out.shape) == (1, 3, 120, 168) and calls == [("fwd", 120, 168, 3, True)]
    # res_out path: factor = ceil(max ratio) = 2, then antialiased resize + clamp afterwards
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", x, (60, 84), None, True, False, torch.float32)
    assert tuple(out.shape) == (1, 3, 60, 84)
    assert calls == [("fwd", 80, 112, 2, False), ("resize", 60, 84, True)]
    # require_ratio=False (train.py:124) keeps the integer-factor size
    calls.clear()
    out = engine.run_forward(1, "FastTransformer", x, (60, 84), None, False, False, torch.float32)
    assert tuple(out.shape) == (1, 3, 80, 112)
    # the reference compares with (H_out, H_out): a square target equal to that skips the resize
    calls.clear()
    engine.run_forward(1, "FastTransformer", torch.zeros(1, 3, 40, 40), (80, 80), None, True, False, torch.float32)
    assert calls == [("fwd", 80, 80, 2, True)]
    with pytest.raises(ValueError, match="scale=5 was not built"):
        engine.run_forward(1, "FastTransformer", x, (200, 280), None, True, False, torch.float32)
    # Window / Residual: upscale_factor overrides res_out
    calls.clear()
    engine.run_forward(1, "WindowTransformer", x, (1080, 1920), 2, True, False, torch.float32)
    assert calls == [("fwd", 80, 112, 0, True)]


def test_frame_shard_partitions():
    from transformerupscaler_b200.sharding import frame_shard
    for total, world in [(64, 8), (64, 3), (5, 8), (8, 1)]:
        cover = []
        for r in range(world):
            a, b = frame_shard(total, r, world)
            cover += list(range(a, b))
        assert cover == list(range(total))
    assert frame_shard(64, 1, 2) == (32, 64)


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    from transformerupscaler_b200.sharding import frame_shard, gather_frames, max_over_ranks
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    total = 5
    frames = torch.arange(total, dtype=torch.float32).reshape(total, 1, 1, 1).expand(total, 3, 2, 2).contiguous()
    a, b = frame_shard(total, rank, world)
    local = frames[a:b] * 2.0                      # stand-in for "upscale my frames"
    full = gather_frames(local, total)
    ms = max_over_ranks(10.0 + rank)
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, torch.equal(full, frames * 2.0), ms))


def test_two_rank_gloo_sharding_and_timing():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    assert [r[1] for r in res] == [True, True]       # every rank reassembles the 1-GPU batch order
    assert [r[2] for r in res] == [11.0, 11.0]       # max over ranks


@pytest.mark.parametrize("r", [2, 3, 6])
def test_fold_up1_matches_the_op_chain(r):
    """packing.fold_up1: the folded 5x5 filter (with its border cases) reproduces conv -> PixelShuffle -> conv (fp64),
    FastTransformer/utils.py:43-98 + model.py:264-265"""
    import numpy as np
    from oracle import upscaler_oracle as orc
    from transformerupscaler_b200.packing import fold_up1, pack_fold_bank, FOLD_CFG
    rs = np.random.RandomState(40 + r)
    H, W = 5, 7
    x = torch.from_numpy(rs.uniform(-1, 1, (1, H, W, 64)))
    w1 = torch.from_numpy(rs.uniform(-0.1, 0.1, (64 * r * r, 64, 3, 3)))
    b1 = torch.from_numpy(rs.uniform(-0.1, 0.1, 64 * r * r))
    w2 = torch.from_numpy(rs.uniform(-0.1, 0.1, (3, 64, 3, 3)))
    ref = orc.conv3x3_nhwc(orc.pixel_shuffle_nhwc(orc.conv3x3_nhwc(x, w1, b1), r), w2, None)[0]      # (rH, rW, 3)
    Wf, bf = fold_up1(w1, b1, w2, r)
    xp = torch.zeros(H + 4, W + 4, 64, dtype=torch.float64)
    xp[2:H + 2, 2:W + 2] = x[0]
    oH, oW = H * r, W * r
    got = torch.zeros(oH, oW, 3, dtype=torch.float64)
    for Y in range(oH):
        for X in range(oW):
            vy = 0 if Y == 0 else 2 if Y == oH - 1 else 1
            vx = 0 if X == 0 else 2 if X == oW - 1 else 1
            y, i, xx, j = Y // r, Y % r, X // r, X % r
            patch = xp[y:y + 5, xx:xx + 5]                             # (dy, dx, ci)
            for c in range(3):
                o = (c * r + i) * r + j
                got[Y, X, c] = (Wf[vy, vx, o].permute(1, 2, 0) * patch).sum() + bf[vy, vx, o]
    assert (got - ref).abs().max().item() < 1e-12
    # tensor-core bank: row n of chunk ch <-> output ((c r + i) - ch RPC) r + j, block blk <-> dy = 4 - blk, kx <-> dx
    NO, rpc, nchunk = FOLD_CFG[r]
    bank, bias = pack_fold_bank(Wf, bf, r)
    assert bank.shape == (nchunk, 5, 5, NO, 64) and bias.shape == (nchunk * NO,)
    for o in (0, 3 * r * r - 1, r * r + 1):
        row, j = o // r, o % r
        ch, q = row // rpc, row % rpc
        assert torch.equal(bank[ch, 3, 1, q * r + j], Wf[1, 1, o, :, 3, 3])
        assert bias[ch * NO + q * r + j] == bf[1, 1, o]


# A stand-in for the reference's models/ tree, same layout: namespace directories (no __init__.py), model.py per model, and the
# relative import of FastTransformer/model.py (`from .utils import ...`).  Its forward runs on CPU, as the reference's does.
_STAND_IN_MODEL = """import torch
import torch.nn.functional as F
{extra}

class TransformerModel(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.conv1 = torch.nn.Conv2d(3, 3, 3, padding=1)

    def forward(self, x, res_out=(1080, 1920)):
        return F.interpolate(self.conv1(x), size=res_out, mode="bicubic", align_corners=False)
"""


def test_reference_loader_resolves_to_the_reference_not_to_the_drop_in_alias(tmp_path):
    """bench.py's reference arm / cpu_baseline must time the UNMODIFIED reference modules (a copy of the reference's models/ in
    baseline/_ref), although this repository ships a `models` package with the same module paths.  The reference's sources are
    not part of this repository, so the loader is pointed at a stand-in tree of the same layout."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    ref = str(tmp_path / "models")
    for name in MODELS:
        os.makedirs(os.path.join(ref, name))
        extra = "from .utils import default_conv  # noqa: F401" if name == "FastTransformer" else ""
        with open(os.path.join(ref, name, "model.py"), "w") as fh:
            fh.write(_STAND_IN_MODEL.format(extra=extra))
    with open(os.path.join(ref, "FastTransformer", "utils.py"), "w") as fh:
        fh.write("def default_conv(*args):\n    return None\n")
    if root not in sys.path:
        sys.path.insert(0, root)
    from baseline.refload import reference_model_class
    for name in ("WindowTransformer", "FastTransformer", "ResidualTransformer"):
        cls = reference_model_class(ref, name)
        assert os.path.abspath(sys.modules[cls.__module__].__file__).startswith(ref)
        m = cls().eval()
        assert isinstance(m, torch.nn.Module) and not cls.__module__.startswith("transformerupscaler_b200")
    # and the reference really runs on CPU (the drop-in alias raises without a CUDA device)
    m = reference_model_class(ref, "WindowTransformer")().eval()
    with torch.no_grad():
        y = m(torch.rand(1, 3, 64, 80), res_out=(96, 120))
    assert tuple(y.shape) == (1, 3, 96, 120)


def test_stack_split_enumeration(tmp_path):
    """The block-level work split of the window-stack kernels (csrc/tc/stack_split.cuh, plain C++ for the host): every
    (tile, block) unit exactly once, a tile cut at most once, its leading blocks the first segment of a CTA and the rest the last
    segment of the next one (tests/host/stack_split_check.cpp states the rules)."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "stack_split_check")
    subprocess.run([gxx, "-std=c++17", "-O1", "-o", exe, os.path.join(root, "tests", "host", "stack_split_check.cpp")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


def test_frag_rel_bias_is_the_mma_fragment_order():
    """packing.frag_rel_bias: [h][rg][n][lane][half][e] = dense[h][rg*16 + half*8 + lane//4][n*8 + (lane%4)*2 + e]
    (what window_stack{,192}_tcgen05.cu fetch with one 16-byte load per lane; pack_weights.cu::frag_rel is the same loop)."""
    from transformerupscaler_b200.packing import frag_rel_bias
    g = torch.Generator().manual_seed(5)
    dense = torch.randn(3, 64, 64, generator=g)
    f = frag_rel_bias(dense).reshape(3, 4, 8, 32, 2, 2)
    for h, rg, n, lane, half, e in [(0, 0, 0, 0, 0, 0), (2, 3, 7, 31, 1, 1), (1, 2, 5, 13, 0, 1), (1, 1, 3, 22, 1, 0)]:
        assert f[h, rg, n, lane, half, e] == dense[h, rg * 16 + half * 8 + lane // 4, n * 8 + (lane % 4) * 2 + e]
    assert torch.equal(torch.sort(f.reshape(3, -1), dim=1).values, torch.sort(dense.reshape(3, -1), dim=1).values)
