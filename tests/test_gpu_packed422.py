"""GPU: packed 4:2:2 frames (yuyv422, uyvy422, y210), dense and as per-frame surfaces.  Every comparison is bitwise: the kernels against
the oracle of tests/test_packed422_host.py (y210 words with random low 6 bits on read), both directions against the nv16 / p210 ops on
the same samples, surfaces against the dense path, and whole forwards against the nv16 / p210 forward of the same samples.  Surfaces
are strided (H, W, 2) views into sentinel-filled pools (pitched rows, a guard row above each frame, shuffled frame slots); every byte
outside the 2W samples of each frame row must keep its sentinel."""
import gc

import pytest
import torch

from tests.golden.cases import CASES, FULLSIZE
from tests.test_gpu_models import build
from tests.test_gpu_p010 import _model, natural_nv12, natural_p010
from tests.test_gpu_yuv_planes import Surfaces
from tests.test_gpu_yuvp import SENTINEL, engine_fwd, eq, st
from tests.test_packed422_host import PACKED, code, colours, from_semi, oracle_packed_to_rgb, oracle_rgb_to_packed, random_packed, to_semi
from tests.test_yuv422_host import code as code_422
from transformerupscaler_b200.synth import synth_frames

pytestmark = pytest.mark.gpu

F32, F16, U8, U16 = torch.float32, torch.float16, torch.uint8, torch.uint16
DEV = torch.device("cuda:0")
PLANES_PER_LAUNCH = 64               # kPlanesPerLaunch of csrc/resample.cu


def _l():
    from transformerupscaler_b200 import _lib
    return _lib, _lib.load()


def is16(fmt):
    return PACKED[fmt][0] == U16


def rgb_dtype(fmt):
    return F32 if is16(fmt) else F16


class Pool:
    """B packed frames of H x W as (H, W, 2) views into a sentinel-filled byte pool: a row pitch of the row rounded up to 256 bytes plus
    an odd multiple of the macropixel (4 / 8 bytes), a guard row above each frame, shuffled frame slots.  pitched=False: rows of exactly
    2W samples"""

    def __init__(self, fmt, B, H, W, seed, pitched=True):
        self.fmt, self.dt = fmt, PACKED[fmt][0]
        es = 2 if self.dt == U16 else 1
        row, mp = 2 * W * es, 4 * es
        pitch = (-(-row // 256) * 256 + mp * (2 * (seed % 3) + 1)) if pitched else row
        self.perm = torch.randperm(B, generator=torch.Generator().manual_seed(seed)).tolist()
        self.idx = torch.tensor(self.perm, device=DEV)
        self.pool = torch.full((B, H + 2, pitch), SENTINEL, dtype=U8, device=DEV)
        self.rows, self.cols = slice(1, 1 + H), slice(0, row)
        self.frames = [self.pool[s, self.rows, self.cols].view(self.dt).unflatten(1, (W, 2)) for s in self.perm]

    def write(self, dense):
        B, H, W, _ = dense.shape
        self.pool[self.idx, self.rows, self.cols] = dense.to(DEV).contiguous().view(B, H, -1).view(U8)

    def read(self):
        p = self.pool[self.idx, self.rows, self.cols].view(self.dt)
        return p.unflatten(2, (p.shape[2] // 2, 2))

    def untouched(self):
        c = self.pool.clone()
        c[self.idx, self.rows, self.cols] = SENTINEL
        return bool((c == SENTINEL).all())

    def descriptors(self):
        from transformerupscaler_b200 import engine
        return engine._descriptors(engine._flat(self.frames), code(self.fmt))


def k_to_rgb(fmt, yuv, f=None, S=None, B=None, H=None, W=None):
    L, lib = _l()
    if f is not None:
        B, H, W = f.shape[:3]
    out = torch.empty(B, 3, H, W, dtype=rgb_dtype(fmt), device=DEV)
    L.check(lib.tu_packed422_to_rgb(f.data_ptr() if f is not None else None, S.descriptors() if S is not None else None, code(fmt, yuv),
                                    out.data_ptr(), B, H, W, st()))
    return out


def k_from_rgb(fmt, yuv, x, S=None):
    L, lib = _l()
    B, _, H, W = x.shape
    out = None if S is not None else torch.empty(B, H, W, 2, dtype=PACKED[fmt][0], device=DEV)
    L.check(lib.tu_rgb_to_packed422(x.data_ptr(), out.data_ptr() if out is not None else None, S.descriptors() if S is not None else None,
                                    code(fmt, yuv), B, H, W, st()))
    return out


def k_semi_to_rgb(fmt, yuv, f):
    """the nv16 / p210 op on the same samples (f: packed frames)"""
    L, lib = _l()
    B, H, W = f.shape[:3]
    semi = to_semi(f, fmt).contiguous()
    out = torch.empty(B, 3, H, W, dtype=rgb_dtype(fmt), device=DEV)
    L.check(lib.tu_yuv422sp_to_rgb(semi.data_ptr(), None, code_422(PACKED[fmt][1], yuv), out.data_ptr(), B, H, W, st()))
    return out


def k_rgb_to_semi(fmt, yuv, x):
    L, lib = _l()
    B, _, H, W = x.shape
    out = torch.empty(B, 2 * H, W, dtype=PACKED[fmt][0], device=DEV)
    L.check(lib.tu_rgb_to_yuv422sp(x.data_ptr(), out.data_ptr(), None, code_422(PACKED[fmt][1], yuv), B, H, W, st()))
    return out


def natural(fmt, B, H, W, seed, yuv="bt709"):
    rgb = synth_frames(B, H, W, seed=seed)
    return oracle_rgb_to_packed(rgb if is16(fmt) else rgb.half(), fmt, yuv)


SIZES = [(1, 2), (3, 6), (6, 10), (720, 1280), (1080, 1920)]


# ---------------------------------------------------------------------------------------------------------------------------------
# the conversion kernels
@pytest.mark.parametrize("fmt", list(PACKED))
@pytest.mark.parametrize("hw", SIZES)
def test_kernels_match_oracle_dense_and_surfaces(fmt, hw):
    H, W = hw
    B = 1 if H * W > 100000 else 3
    f = random_packed(fmt, B, H, W, seed=H * 31 + W)                    # y210: whole random words, low 6 bits included
    g = torch.Generator().manual_seed(H * 7 + W)
    x = (torch.rand(B, 3, H, W, generator=g) * 1.6 - 0.3).to(rgb_dtype(fmt))        # values outside [0, 1] too
    fd, xd = f.to(DEV), x.to(DEV)
    for i, yuv in enumerate(colours(fmt)):
        want = oracle_packed_to_rgb(f, fmt, yuv).to(rgb_dtype(fmt))
        got = k_to_rgb(fmt, yuv, fd)
        assert eq(got, want) and eq(got, k_semi_to_rgb(fmt, yuv, fd)), yuv
        S = Pool(fmt, B, H, W, seed=i, pitched=i % 2 == 0)
        S.write(fd)
        assert eq(k_to_rgb(fmt, yuv, S=S, B=B, H=H, W=W), want) and S.untouched(), yuv
        want = oracle_rgb_to_packed(x, fmt, yuv)
        got = k_from_rgb(fmt, yuv, xd)
        assert eq(got, want) and eq(to_semi(got, fmt), k_rgb_to_semi(fmt, yuv, xd)), yuv
        T = Pool(fmt, B, H, W, seed=i + 1, pitched=i % 2 == 1)
        k_from_rgb(fmt, yuv, xd, T)
        assert eq(T.read(), want) and T.untouched(), yuv


@pytest.mark.parametrize("fmt", list(PACKED))
@pytest.mark.parametrize("B", [PLANES_PER_LAUNCH + 1, 2 * PLANES_PER_LAUNCH + 2])
def test_batches_of_several_launches(fmt, B):
    H, W = 5, 10
    f = random_packed(fmt, B, H, W, seed=B).to(DEV)
    yuv = "bt2020" if is16(fmt) else "bt601_full"
    want = oracle_packed_to_rgb(f, fmt, yuv).to(rgb_dtype(fmt))
    assert eq(k_to_rgb(fmt, yuv, f), want)
    S = Pool(fmt, B, H, W, seed=4)
    S.write(f)
    assert eq(k_to_rgb(fmt, yuv, S=S, B=B, H=H, W=W), want)
    x = want.to(DEV)
    back = oracle_rgb_to_packed(x.cpu(), fmt, yuv)
    assert eq(k_from_rgb(fmt, yuv, x), back)
    T = Pool(fmt, B, H, W, seed=5, pitched=False)
    k_from_rgb(fmt, yuv, x, T)
    assert eq(T.read(), back) and T.untouched() and S.untouched()


# ---------------------------------------------------------------------------------------------------------------------------------
# whole forwards
FWD_CASES = ["window_72x104_r1p5", "fast_40x56_x2", "fast_40x56_res60x84", "residual_720p_1080p"]


@pytest.mark.parametrize("name", FWD_CASES)
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forwards(name, path):
    c = CASES[name]
    B, _, H, W = c["shape"]
    kw = c["kw"]
    M = _model(name)
    M.engine_precision = path
    bf16 = path == "bf16"
    s = c["xseed"]
    try:
        with torch.no_grad():
            # packed -> packed is the nv16 / p210 forward of the same samples; the forward is the fp16 / fp32 one of the converted frame
            for fmt, ofmt, yuv in (("yuyv422", "yuyv422", "bt601"), ("uyvy422", "uyvy422", "bt709_full"), ("yuyv422", "uyvy422", "bt709"),
                                   ("y210", "y210", "bt2020")):
                f = natural(fmt, B, H, W, seed=s, yuv=yuv).to(DEV)
                got = M(f, in_layout=fmt, out_layout=ofmt, yuv=yuv, **kw)
                sf, so = PACKED[fmt][1], PACKED[ofmt][1]
                want = M(to_semi(f, fmt).contiguous(), in_layout=sf, out_layout=so, yuv=yuv, **kw)
                assert got.dtype == PACKED[ofmt][0] and got.dim() == 4 and got.shape[3] == 2, fmt
                assert eq(got, from_semi(want, ofmt)), (fmt, ofmt)
                assert eq(got, engine_fwd(M, k_to_rgb(fmt, yuv, f), bf16, PACKED[ofmt][0], kw, out_layout=ofmt, yuv=yuv)), fmt
                assert eq(got, k_from_rgb(ofmt, yuv, engine_fwd(M, f, bf16, rgb_dtype(fmt), kw, in_layout=fmt, yuv=yuv))), fmt
            oh, ow = got.shape[1:3]
            # mixed sides: yuyv422 surfaces -> NV12; NV12 surfaces -> uyvy422 surfaces; BGRA -> y210; y210 -> P010
            f = natural("yuyv422", B, H, W, seed=s + 1).to(DEV)
            S = Pool("yuyv422", B, H, W, seed=s)
            S.write(f)
            assert eq(M(S.frames, in_layout="yuyv422", out_layout="nv12", **kw), M(f, in_layout="yuyv422", out_layout="nv12", **kw))
            assert S.untouched()
            nv = natural_nv12(B, H, W, seed=s + 2).to(DEV)
            N = Surfaces("nv12", B, H, W, split=True, seed=s)
            N.write(nv)
            O = Pool("uyvy422", B, oh, ow, seed=s + 1)
            assert M(N.planes, in_layout="nv12", out_layout="uyvy422", out=O.frames, **kw) is O.frames
            assert eq(O.read(), M(nv, in_layout="nv12", out_layout="uyvy422", **kw)) and O.untouched() and N.untouched()
            bgra = (torch.rand(B, H, W, 4, generator=torch.Generator().manual_seed(s)) * 255).to(U8).to(DEV)
            got = M(bgra, in_layout="bgra", out_layout="y210", **kw)
            assert got.dtype == U16 and eq(got, from_semi(M(bgra, in_layout="bgra", out_layout="p210", **kw), "y210"))
            assert int((got.view(torch.int16).to(torch.int32) & 0x3F).max()) == 0                 # low 6 bits zero
            y210 = natural("y210", B, H, W, seed=s + 3, yuv="bt2020").to(DEV)
            y210 = (y210.to(torch.int32) | torch.randint(0, 64, y210.shape, device=DEV, dtype=torch.int32)).to(U16)   # low bits ignored
            assert eq(M(y210, in_layout="y210", out_layout="p010", yuv="bt2020", **kw),
                      M(to_semi(y210, "y210").contiguous(), in_layout="p210", out_layout="p010", yuv="bt2020", **kw))
    finally:
        M.engine_precision = None


def test_fullsize_window_yuyv422_to_uyvy422_bf16():
    c = FULLSIZE["window_720p_1080p_b8"]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    f = natural("yuyv422", B, H, W, seed=c["xseed"]).to(DEV)
    with torch.no_grad():
        got = M(f, in_layout="yuyv422", out_layout="uyvy422", **c["kw"])
        assert got.shape == (B, 1080, 1920, 2)
        assert eq(got, from_semi(M(to_semi(f, "yuyv422").contiguous(), in_layout="nv16", out_layout="nv16", **c["kw"]), "uyvy422"))
        S = Pool("yuyv422", B, H, W, seed=1)
        S.write(f)
        O = Pool("uyvy422", B, 1080, 1920, seed=2)
        M(S.frames, in_layout="yuyv422", out_layout="uyvy422", out=O.frames, **c["kw"])
    assert eq(O.read(), got) and O.untouched() and S.untouched()


def test_fullsize_residual_y210_bf16():
    c = FULLSIZE["residual_720p_4k"]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    M.engine_precision = "bf16"
    f = natural("y210", B, H, W, seed=c["xseed"], yuv="bt2020").to(DEV)
    kw = dict(in_layout="y210", out_layout="y210", yuv="bt2020", **c["kw"])
    with torch.no_grad():
        want = M(f, **kw)
        assert want.shape == (B, 2160, 3840, 2)
        assert eq(want, from_semi(M(to_semi(f, "y210").contiguous(), in_layout="p210", out_layout="p210", yuv="bt2020", **c["kw"]), "y210"))
        S = Pool("y210", B, H, W, seed=3)
        S.write(f)
        O = Pool("y210", B, 2160, 3840, seed=4)
        M(S.frames, out=O.frames, **kw)
    assert eq(O.read(), want) and O.untouched()


# ---------------------------------------------------------------------------------------------------------------------------------
# wrappers
def test_captured_graph_replays_surfaces_after_the_lists_are_gone():
    M = _model("window_72x104_r1p5")
    kw = dict(res_out=(108, 156), in_layout="yuyv422", out_layout="y210")
    f1, f2 = natural("yuyv422", 2, 72, 104, seed=21).to(DEV), natural("yuyv422", 2, 72, 104, seed=22).to(DEV)
    S, O = Pool("yuyv422", 2, 72, 104, seed=3), Pool("y210", 2, 108, 156, seed=4)
    S.write(f1)
    frames_in, frames_out = list(S.frames), list(O.frames)
    with torch.no_grad():
        s = torch.cuda.Stream(DEV)
        s.wait_stream(torch.cuda.current_stream(DEV))
        with torch.cuda.stream(s):
            M(frames_in, out=frames_out, **kw)                           # packs the weights outside the capture
        torch.cuda.current_stream(DEV).wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            M(frames_in, out=frames_out, **kw)
    del frames_in, frames_out                                            # the descriptor lists (and their ctypes tables) are gone
    S.frames = O.frames = None
    gc.collect()
    S.write(f2)                                                          # new contents in the same surfaces
    O.write(torch.zeros(2, 108, 156, 2, dtype=U16))
    g.replay()
    torch.cuda.synchronize()
    with torch.no_grad():
        want = M(f2, **kw)
    assert eq(O.read(), want) and O.untouched()


def test_graphed_model_frame_pipeline_and_compile():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M = _model("window_72x104_r1p5")
    for fmt, ofmt, yuv in (("yuyv422", "yuyv422", "bt709"), ("uyvy422", "nv12", "bt601"), ("y210", "y210", "bt2020_full")):
        kw = dict(res_out=(108, 156), in_layout=fmt, out_layout=ofmt, yuv=yuv)
        xs = [natural(fmt, 2, 72, 104, seed=700 + i, yuv=yuv) for i in range(4)]
        with torch.no_grad():
            eager = [M(x.to(DEV), **kw).clone() for x in xs]
        G = GraphedModel(M)
        for x, e in zip(xs, eager):
            assert eq(G(x.to(DEV), **kw), e)
        hin = [x.pin_memory() for x in xs]                               # the webcam case: pinned (B, H, W, 2) host frames
        hout = [torch.zeros(eager[0].shape, dtype=eager[0].dtype).pin_memory() for _ in xs]
        pipe = FramePipeline(M, depth=3, device=DEV, compute_streams=2, **kw)
        for a, b in zip(hin, hout):
            pipe.submit(a, b)
        pipe.drain()
        for b, e in zip(hout, eager):
            assert eq(b, e)
        with pytest.raises(TypeError, match="frame planes"):
            pipe.submit([x.to(DEV)[0] for x in xs[:2]], hout[0])
        with torch.no_grad():
            assert eq(torch.compile(M)(xs[0].to(DEV), **kw), eager[0])
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(M)(list(Pool("y210", 1, 72, 104, seed=1).frames), in_layout="y210", res_out=(108, 156))
    # surfaces out under torch.compile
    f = natural("uyvy422", 1, 72, 104, seed=9).to(DEV)
    kw = dict(in_layout="uyvy422", out_layout="yuyv422", res_out=(108, 156))
    with torch.no_grad():
        want = M(f, **kw)
        O = Pool("yuyv422", 1, 108, 156, seed=1)
        torch.compile(M)(f, out=O.frames, **kw)
    assert eq(O.read(), want) and O.untouched()
    # the Resize path ends in tu::rgb_to_packed422 (compiled) and tu::rgb_to_packed422_planes (eager)
    Mf = _model("fast_40x56_res60x84")
    for fin, fout in (("yuyv422", "uyvy422"), ("y210", "y210"), ("nv12", "yuyv422")):
        f = (natural(fin, 1, 40, 56, seed=3) if fin != "nv12" else natural_nv12(1, 40, 56, seed=3)).to(DEV)
        kw = dict(in_layout=fin, out_layout=fout, res_out=(60, 84))
        with torch.no_grad():
            want = Mf(f, **kw)
            assert want.shape == (1, 60, 84, 2) and eq(torch.compile(Mf)(f, **kw), want)
            O = Pool(fout, 1, 60, 84, seed=1)
            Mf(f, out=O.frames, **kw)
        assert eq(O.read(), want) and O.untouched()
    p010 = natural_p010(1, 40, 56, seed=4).to(DEV)
    with torch.no_grad():
        assert eq(Mf(p010, in_layout="p010", out_layout="y210", res_out=(60, 84)),
                  from_semi(Mf(p010, in_layout="p010", out_layout="p210", res_out=(60, 84)), "y210"))
