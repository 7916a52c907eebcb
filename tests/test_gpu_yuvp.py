"""GPU: planar YUV frames (yuv420p, yuv444p, yuv444p16), dense and as per-frame surfaces (TuFramePlanes3: three planes with row
pitches).  Every comparison is bitwise: the kernels against the oracle of tests/test_yuvp_host.py, yuv420p against NV12 with its
chroma interleaved, 4:4:4 forwards against the fp16 / fp32 forward of the converted frame, the luma planes against NV12 / P010
outputs, and surfaces against the dense path.  Surfaces are strided views into sentinel-filled pools (a row pitch of the row rounded
up to 256 bytes plus an odd multiple of the alignment, a guard row above each plane, shuffled frame slots, 8-bit 4:4:4 planes at odd
addresses); every byte outside the valid samples of the planes' rows must keep its sentinel."""
import pytest
import torch

from tests.golden.cases import CASES, FULLSIZE
from tests.test_gpu_models import build
from tests.test_gpu_p010 import _model, natural_nv12
from tests.test_gpu_yuv_planes import Surfaces
from tests.test_p010_host import COLOURS10
from tests.test_yuvp_host import (COLOURS8, nv12_to_yuv420p, oracle_rgb_to_yuv420p, oracle_rgb_to_yuv444, oracle_yuv420p_to_rgb,
                                  oracle_yuv444_to_rgb, split420, yuv420p_to_nv12)
from transformerupscaler_b200.synth import synth_frames

pytestmark = pytest.mark.gpu

F32, F16, U8, U16 = torch.float32, torch.float16, torch.uint8, torch.uint16
DEV = torch.device("cuda:0")
SENTINEL = 0xA5
PLANES_PER_LAUNCH = 64               # kPlanesPerLaunch of csrc/resample.cu
FMTS = ("yuv420p", "yuv444p", "yuv444p16")


def _l():
    from transformerupscaler_b200 import _lib
    return _lib, _lib.load()


def code(fmt, yuv="bt709"):
    from transformerupscaler_b200 import _lib as L, engine
    return {"yuv420p": L.TU_U8 | L.TU_LAYOUT_YUV420P, "yuv444p": L.TU_U8 | L.TU_LAYOUT_YUV444P,
            "yuv444p16": L.TU_U16 | L.TU_LAYOUT_YUV444P}[fmt] | engine.yuv_code(yuv)


def st():
    return torch.cuda.current_stream().cuda_stream


def eq(a, b):
    """bitwise equality (uint16 compared as int16 words)"""
    if a.dtype == U16:
        a, b = a.view(torch.int16), b.view(torch.int16)
    return a.shape == b.shape and torch.equal(a.to(DEV), b.to(DEV))


def planes_of(fmt, f):
    """dense frames -> [Y, U, V] (B, h, w) planes"""
    return list(split420(f)) if fmt == "yuv420p" else [f[:, 0], f[:, 1], f[:, 2]]


def dense_of(fmt, planes):
    y, u, v = planes
    if fmt == "yuv420p":
        B, H, W = y.shape
        return torch.cat([y.reshape(B, -1), u.reshape(B, -1), v.reshape(B, -1)], 1).reshape(B, 3 * H // 2, W)
    return torch.stack([y, u, v], 1)


class Surfaces3:
    """B planar YUV frames of H x W in strided views of sentinel-filled byte pools, one pool per plane.  pitched=False: rows of exactly
    the row's bytes (a dense plane, as FFmpeg's linesize often is)"""

    def __init__(self, fmt, B, H, W, seed, pitched=True):
        self.fmt, self.B = fmt, B
        es = 2 if fmt == "yuv444p16" else 1
        ch, cw = (H // 2, W // 2) if fmt == "yuv420p" else (H, W)
        self.dims = [(H, W), (ch, cw), (ch, cw)]
        self.perm = torch.randperm(B, generator=torch.Generator().manual_seed(seed)).tolist()
        self.idx = torch.tensor(self.perm, device=DEV)
        self.regions = []
        for p, (h, w) in enumerate(self.dims):
            row = w * es
            # 8-bit 4:4:4 planes may start at any byte; the yuv420p luma and every 16-bit plane at even bytes
            off = (1 if (seed + p) % 2 else 3) if fmt == "yuv444p" and pitched else 0
            pitch = (-(-row // 256) * 256 + 2 * (2 * ((seed + p) % 3) + 1) + off) if pitched else row
            pool = torch.full((B, h + 2, pitch), SENTINEL, dtype=U8, device=DEV)
            self.regions.append((pool, slice(1, 1 + h), slice(off, off + row)))
        dt = U16 if es == 2 else U8
        self.planes = [tuple(pool[s, rows, cols].view(dt) for pool, rows, cols in self.regions) for s in self.perm]

    def write(self, dense):
        for (pool, rows, cols), plane in zip(self.regions, planes_of(self.fmt, dense.to(DEV))):
            pool[self.idx, rows, cols] = plane.contiguous().view(U8)

    def read(self):
        planes = [pool[self.idx, rows, cols] for pool, rows, cols in self.regions]
        if self.fmt == "yuv444p16":
            planes = [p.view(U16) for p in planes]
        return dense_of(self.fmt, planes)

    def untouched(self):
        ok = True
        for pool, rows, cols in self.regions:
            c = pool.clone()
            c[self.idx, rows, cols] = SENTINEL
            ok &= bool((c == SENTINEL).all())
        return ok

    def descriptors(self):
        from transformerupscaler_b200 import engine
        return engine._descriptors(engine._flat(self.planes), code(self.fmt))


def rgb_dtype(fmt):
    return F32 if fmt == "yuv444p16" else F16


def k_to_rgb(fmt, yuv, f=None, S=None, B=None, H=None, W=None):
    L, lib = _l()
    if f is not None:
        B = f.shape[0]
        H, W = (f.shape[1] * 2 // 3, f.shape[2]) if fmt == "yuv420p" else f.shape[2:]
    out = torch.empty(B, 3, H, W, dtype=rgb_dtype(fmt), device=DEV)
    L.check(lib.tu_yuvp_to_rgb(f.data_ptr() if f is not None else None, S.descriptors() if S is not None else None, code(fmt, yuv),
                               out.data_ptr(), B, H, W, st()))
    return out


def k_from_rgb(fmt, yuv, x, S=None):
    L, lib = _l()
    B, _, H, W = x.shape
    shape = (B, 3 * H // 2, W) if fmt == "yuv420p" else (B, 3, H, W)
    out = None if S is not None else torch.empty(shape, dtype=U16 if fmt == "yuv444p16" else U8, device=DEV)
    L.check(lib.tu_rgb_to_yuvp(x.data_ptr(), out.data_ptr() if out is not None else None, S.descriptors() if S is not None else None,
                               code(fmt, yuv), B, H, W, st()))
    return out


def random_frames(fmt, B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    shape = (B, 3 * H // 2, W) if fmt == "yuv420p" else (B, 3, H, W)
    hi = 65536 if fmt == "yuv444p16" else 256
    return torch.randint(0, hi, shape, generator=g, dtype=torch.int32).to(U16 if fmt == "yuv444p16" else U8)


def oracle_to_rgb(fmt, f, yuv):
    rgb = oracle_yuv420p_to_rgb(f, yuv) if fmt == "yuv420p" else oracle_yuv444_to_rgb(f, yuv)
    return rgb.to(rgb_dtype(fmt))


def oracle_from_rgb(fmt, x, yuv):
    return oracle_rgb_to_yuv420p(x.cpu(), yuv) if fmt == "yuv420p" else oracle_rgb_to_yuv444(x.cpu(), yuv, fmt == "yuv444p16")


def colours(fmt):
    return COLOURS10 if fmt == "yuv444p16" else COLOURS8


SIZES = {"yuv420p": [(2, 2), (2, 6), (6, 10), (4, 1280), (720, 1280)],                          # W/2 odd in the first three
         "yuv444p": [(1, 1), (2, 2), (3, 5), (7, 9), (2, 6), (5, 1283), (720, 1280)],
         "yuv444p16": [(1, 1), (2, 2), (3, 5), (7, 9), (2, 6), (5, 1283), (720, 1280)]}
CASES_K = [(fmt, hw) for fmt in FMTS for hw in SIZES[fmt]]


# ---------------------------------------------------------------------------------------------------------------------------------
# the conversion kernels
@pytest.mark.parametrize("fmt,hw", CASES_K)
def test_kernels_match_oracle_dense_and_surfaces(fmt, hw):
    H, W = hw
    f = random_frames(fmt, 3, H, W, seed=H * 31 + W)
    g = torch.Generator().manual_seed(H * 7 + W)
    x = (torch.rand(3, 3, H, W, generator=g) * 1.6 - 0.3).to(rgb_dtype(fmt))        # values outside [0, 1] too
    for i, yuv in enumerate(colours(fmt)):
        want = oracle_to_rgb(fmt, f, yuv)
        fd = f.to(DEV)
        assert eq(k_to_rgb(fmt, yuv, fd), want), yuv
        S = Surfaces3(fmt, 3, H, W, seed=i, pitched=i % 2 == 0)
        S.write(fd)
        assert eq(k_to_rgb(fmt, yuv, S=S, B=3, H=H, W=W), want) and S.untouched(), yuv
        want = oracle_from_rgb(fmt, x, yuv)
        xd = x.to(DEV)
        assert eq(k_from_rgb(fmt, yuv, xd), want), yuv
        T = Surfaces3(fmt, 3, H, W, seed=i + 1, pitched=i % 2 == 1)
        k_from_rgb(fmt, yuv, xd, T)
        assert eq(T.read(), want) and T.untouched(), yuv


@pytest.mark.parametrize("hw", SIZES["yuv420p"])
def test_yuv420p_kernels_are_the_nv12_kernels(hw):
    H, W = hw
    L, lib = _l()
    f = random_frames("yuv420p", 2, H, W, seed=H + W).to(DEV)
    x = (torch.rand(2, 3, H, W, generator=torch.Generator().manual_seed(W)) * 1.4 - 0.2).half().to(DEV)
    for yuv in COLOURS8:
        nv = yuv420p_to_nv12(f)
        rgb = torch.empty(2, 3, H, W, dtype=F16, device=DEV)
        L.check(lib.tu_nv12_to_rgb(nv.contiguous().data_ptr(), L.TU_U8 | L.TU_LAYOUT_NV12 | code("yuv420p", yuv) & 0xF000, rgb.data_ptr(),
                                   2, H, W, st()))
        assert eq(k_to_rgb("yuv420p", yuv, f), rgb)
        out = torch.empty(2, 3 * H // 2, W, dtype=U8, device=DEV)
        L.check(lib.tu_rgb_to_nv12(x.data_ptr(), out.data_ptr(), L.TU_U8 | L.TU_LAYOUT_NV12 | code("yuv420p", yuv) & 0xF000, 2, H, W, st()))
        assert eq(k_from_rgb("yuv420p", yuv, x), nv12_to_yuv420p(out))


@pytest.mark.parametrize("fmt", FMTS)
def test_batch_larger_than_one_launch(fmt):
    B, H, W = PLANES_PER_LAUNCH + 6, 6, 10
    f = random_frames(fmt, B, H, W, seed=99).to(DEV)
    yuv = "bt2020" if fmt == "yuv444p16" else "bt601_full"
    want = oracle_to_rgb(fmt, f, yuv)
    assert eq(k_to_rgb(fmt, yuv, f), want)
    S = Surfaces3(fmt, B, H, W, seed=4)
    S.write(f)
    assert eq(k_to_rgb(fmt, yuv, S=S, B=B, H=H, W=W), want)
    x = want.to(DEV)
    back = oracle_from_rgb(fmt, x, yuv)
    assert eq(k_from_rgb(fmt, yuv, x), back)
    T = Surfaces3(fmt, B, H, W, seed=5, pitched=False)
    k_from_rgb(fmt, yuv, x, T)
    assert eq(T.read(), back) and T.untouched() and S.untouched()


def test_yv12_by_swapped_pointers():
    """a YV12 frame (Y, then V, then U) is read and written through TuFramePlanes3 with u and v pointing at its U and V planes"""
    from transformerupscaler_b200 import _lib as L
    _, lib = _l()
    B, H, W = 3, 8, 12
    f = random_frames("yuv420p", B, H, W, seed=5).to(DEV)
    y, u, v = split420(f)
    yv12 = torch.cat([y.reshape(B, -1), v.reshape(B, -1), u.reshape(B, -1)], 1).contiguous()
    n, q = H * W, H * W // 4
    P = L.TuFramePlanes3
    fr = (P * B)(*[P(yv12[b].data_ptr(), yv12[b, n + q:].data_ptr(), yv12[b, n:].data_ptr(), W, W // 2, W // 2) for b in range(B)])
    rgb = torch.empty(B, 3, H, W, dtype=F16, device=DEV)
    L.check(lib.tu_yuvp_to_rgb(None, fr, code("yuv420p"), rgb.data_ptr(), B, H, W, st()))
    assert eq(rgb, k_to_rgb("yuv420p", "bt709", f))
    yv12.zero_()
    L.check(lib.tu_rgb_to_yuvp(rgb.data_ptr(), None, fr, code("yuv420p"), B, H, W, st()))
    y2 = yv12[:, :n].reshape(B, H, W)
    v2, u2 = yv12[:, n:n + q].reshape(B, H // 2, W // 2), yv12[:, n + q:].reshape(B, H // 2, W // 2)
    assert eq(torch.cat([y2.reshape(B, -1), u2.reshape(B, -1), v2.reshape(B, -1)], 1).reshape(B, 3 * H // 2, W),
              k_from_rgb("yuv420p", "bt709", rgb))


# ---------------------------------------------------------------------------------------------------------------------------------
# whole forwards
FWD_CASES = ["window_72x104_r1p5", "window_64x80_x2", "fast_40x56_x2", "fast_24x32_x6", "fast_40x56_res60x84", "residual_720p_1080p"]


def natural(fmt, B, H, W, seed, yuv="bt709"):
    rgb = synth_frames(B, H, W, seed=seed)
    if fmt == "yuv420p":
        return oracle_rgb_to_yuv420p(rgb.half(), yuv)
    return oracle_rgb_to_yuv444(rgb.half() if fmt == "yuv444p" else rgb, yuv, fmt == "yuv444p16")


def engine_fwd(M, x, bf16, out_dtype, kw, **lk):
    """the forward through engine.run_forward, which (unlike the model classes) takes an fp16 / fp32 image with a YUV out_layout"""
    from transformerupscaler_b200 import engine
    return engine.run_forward(M._packed(bf16, DEV), M.ENGINE_MODEL, x, kw.get("res_out", (1080, 1920)), kw.get("upscale_factor"),
                              kw.get("require_ratio", True), bf16, out_dtype, **lk)


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
            # yuv420p is NV12 with the chroma de-interleaved, in and out
            nv = natural_nv12(B, H, W, seed=s, yuv="bt601").to(DEV)
            f420 = nv12_to_yuv420p(nv)
            want = M(nv, in_layout="nv12", out_layout="nv12", yuv="bt601", **kw)
            got = M(f420, in_layout="yuv420p", out_layout="yuv420p", yuv="bt601", **kw)
            assert got.dtype == U8 and eq(got, nv12_to_yuv420p(want))
            oh, ow = want.shape[1] * 2 // 3, want.shape[2]
            # 4:4:4 in: the fp16 (8-bit) / fp32 (16-bit) forward of the converted frame; 4:4:4 out: that output converted
            f444 = natural("yuv444p", B, H, W, seed=s + 1).to(DEV)
            rgb16 = k_to_rgb("yuv444p", "bt709", f444)
            got = M(f444, in_layout="yuv444p", out_layout="yuv444p", **kw)
            assert got.shape == (B, 3, oh, ow) and got.dtype == U8
            assert eq(got, engine_fwd(M, rgb16, bf16, U8, kw, out_layout="yuv444p"))
            assert eq(got, k_from_rgb("yuv444p", "bt709", engine_fwd(M, f444, bf16, F16, kw, in_layout="yuv444p")))
            f16w = natural("yuv444p16", B, H, W, seed=s + 2, yuv="bt2020").to(DEV)
            rgb32 = k_to_rgb("yuv444p16", "bt2020", f16w)
            got = M(f16w, in_layout="yuv444p16", out_layout="yuv444p16", yuv="bt2020", **kw)
            assert got.shape == (B, 3, oh, ow) and got.dtype == U16
            assert eq(got, engine_fwd(M, rgb32, bf16, U16, kw, out_layout="yuv444p16", yuv="bt2020"))
            assert eq(got, k_from_rgb("yuv444p16", "bt2020", engine_fwd(M, f16w, bf16, F32, kw, in_layout="yuv444p16", yuv="bt2020")))
            # the luma planes of 4:4:4 outputs are those of the NV12 / P010 outputs of the same forward
            xu = (torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(s)) * 255).to(U8).to(DEV)
            assert eq(M(xu, out_layout="yuv444p", **kw)[:, 0], M(xu, out_layout="nv12", **kw)[:, :oh])
            assert eq(M(xu, out_layout="yuv444p16", **kw)[:, 0], M(xu, out_layout="p010", **kw)[:, :oh])
            # mixed sides
            assert eq(M(f420, in_layout="yuv420p", out_layout="p010", **kw), M(yuv420p_to_nv12(f420), in_layout="nv12", out_layout="p010", **kw))
            assert eq(M(f16w, in_layout="yuv444p16", out_layout="bgra", yuv="bt2020", **kw),
                      engine_fwd(M, rgb32, bf16, U8, kw, out_layout="bgra"))
            # surfaces: NV12 surfaces -> yuv444p surfaces, yuv444p16 surfaces -> yuv420p surfaces, against the dense results
            S = Surfaces("nv12", B, H, W, split=True, seed=s)
            S.write(nv)
            O = Surfaces3("yuv444p", B, oh, ow, seed=s)
            assert M(S.planes, in_layout="nv12", out_layout="yuv444p", yuv="bt601", out=O.planes, **kw) is O.planes
            assert eq(O.read(), M(nv, in_layout="nv12", out_layout="yuv444p", yuv="bt601", **kw)) and O.untouched() and S.untouched()
            P = Surfaces3("yuv444p16", B, H, W, seed=s + 1)
            P.write(f16w)
            O = Surfaces3("yuv420p", B, oh, ow, seed=s + 2)
            M(P.planes, in_layout="yuv444p16", out_layout="yuv420p", out=O.planes, **kw)
            assert eq(O.read(), M(f16w, in_layout="yuv444p16", out_layout="yuv420p", **kw)) and O.untouched() and P.untouched()
            Q = Surfaces3("yuv444p", B, H, W, seed=s + 3)
            Q.write(f444)
            assert eq(M(Q.planes, in_layout="yuv444p", out_layout="hwc", **kw), M(f444, in_layout="yuv444p", out_layout="hwc", **kw))
    finally:
        M.engine_precision = None


def test_forward_batch_larger_than_one_launch():
    M = _model("window_72x104_r1p5")
    B = PLANES_PER_LAUNCH + 6
    f = natural("yuv444p", B, 72, 104, seed=5).to(DEV)
    S = Surfaces3("yuv444p", B, 72, 104, seed=6)
    S.write(f)
    O = Surfaces3("yuv420p", B, 108, 156, seed=7)
    with torch.no_grad():
        M(S.planes, in_layout="yuv444p", out_layout="yuv420p", out=O.planes, res_out=(108, 156))
        want = M(f, in_layout="yuv444p", out_layout="yuv420p", res_out=(108, 156))
    assert eq(O.read(), want) and O.untouched() and S.untouched()


def test_fullsize_window_yuv420p_is_nv12_bf16():
    c = FULLSIZE["window_720p_1080p_b8"]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    nv = natural_nv12(B, H, W, seed=c["xseed"]).to(DEV)
    with torch.no_grad():
        want = nv12_to_yuv420p(M(nv, in_layout="nv12", out_layout="nv12", **c["kw"]))
        assert eq(M(nv12_to_yuv420p(nv), in_layout="yuv420p", out_layout="yuv420p", **c["kw"]), want)
        S = Surfaces3("yuv420p", B, H, W, seed=1)
        S.write(nv12_to_yuv420p(nv))
        O = Surfaces3("yuv420p", B, 1080, 1920, seed=2, pitched=False)
        M(S.planes, in_layout="yuv420p", out_layout="yuv420p", out=O.planes, **c["kw"])
    assert eq(O.read(), want) and O.untouched()


def test_fullsize_residual_yuv444p16_bf16():
    c = FULLSIZE["residual_720p_4k"]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    M.engine_precision = "bf16"
    f = natural("yuv444p16", B, H, W, seed=c["xseed"], yuv="bt2020").to(DEV)
    kw = dict(in_layout="yuv444p16", out_layout="yuv444p16", yuv="bt2020", **c["kw"])
    with torch.no_grad():
        want = M(f, **kw)
        assert eq(want, engine_fwd(M, k_to_rgb("yuv444p16", "bt2020", f), True, U16, c["kw"], out_layout="yuv444p16", yuv="bt2020"))
        S = Surfaces3("yuv444p16", B, H, W, seed=3)
        S.write(f)
        O = Surfaces3("yuv444p16", B, 2160, 3840, seed=4)
        M(S.planes, out=O.planes, **kw)
    assert eq(O.read(), want) and O.untouched()
    assert int((want.view(torch.int16).to(torch.int32) & 63).abs().max()) == 0          # low 6 bits zero


# ---------------------------------------------------------------------------------------------------------------------------------
# wrappers
def test_graphed_model_frame_pipeline_and_compile():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M = _model("window_72x104_r1p5")
    for fmt, ofmt, yuv, oshape in (("yuv420p", "yuv444p16", "bt709_full", (2, 3, 108, 156)),
                                   ("yuv444p16", "yuv420p", "bt601", (2, 162, 156))):
        kw = dict(res_out=(108, 156), in_layout=fmt, out_layout=ofmt, yuv=yuv)
        xs = [natural(fmt, 2, 72, 104, seed=700 + i, yuv=yuv) for i in range(4)]
        with torch.no_grad():
            eager = [M(x.to(DEV), **kw).clone() for x in xs]
        assert eager[0].shape == oshape
        G = GraphedModel(M)
        for x, e in zip(xs, eager):
            assert eq(G(x.to(DEV), **kw), e)
        hin = [x.pin_memory() for x in xs]
        hout = [torch.zeros(oshape, dtype=eager[0].dtype).pin_memory() for _ in xs]
        pipe = FramePipeline(M, depth=3, device=DEV, compute_streams=2, **kw)
        for a, b in zip(hin, hout):
            pipe.submit(a, b)
        pipe.drain()
        for b, e in zip(hout, eager):
            assert eq(b, e)
        with torch.no_grad():
            assert eq(torch.compile(M)(xs[0].to(DEV), **kw), eager[0])
    # surfaces out under torch.compile: tu::forward_planes declares the planes it writes
    f = natural("yuv420p", 1, 72, 104, seed=9).to(DEV)
    kw = dict(in_layout="yuv420p", out_layout="yuv444p", res_out=(108, 156))
    with torch.no_grad():
        want = M(f, **kw)
        O = Surfaces3("yuv444p", 1, 108, 156, seed=1)
        torch.compile(M)(f, out=O.planes, **kw)
    assert eq(O.read(), want) and O.untouched()
    # the Resize path ends in tu::rgb_to_yuvp (compiled) / tu::rgb_to_yuvp_planes (eager)
    Mf = _model("fast_40x56_res60x84")
    f = natural("yuv444p", 1, 40, 56, seed=3).to(DEV)
    kw = dict(in_layout="yuv444p", out_layout="yuv444p", res_out=(60, 84))
    with torch.no_grad():
        want = Mf(f, **kw)
        assert want.shape == (1, 3, 60, 84) and eq(torch.compile(Mf)(f, **kw), want)
        O = Surfaces3("yuv444p", 1, 60, 84, seed=1)
        Mf(f, out=O.planes, **kw)
    assert eq(O.read(), want) and O.untouched()
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(M)(O.planes, in_layout="yuv444p", res_out=(108, 156))
    pipe = FramePipeline(M, depth=2, device=DEV, in_layout="yuv444p", res_out=(108, 156))
    with pytest.raises(TypeError, match="frame planes"):
        pipe.submit(O.planes, torch.empty(1, 3, 108, 156, dtype=U8).pin_memory())


def test_uint16_with_other_layouts_is_float32():
    """a uint16 tensor that is not a P010 / yuv444p16 frame is an image like any other: read as float32"""
    M = _model("window_72x104_r1p5")
    x = (torch.rand(1, 3, 72, 104, generator=torch.Generator().manual_seed(1)) * 2).to(U16).to(DEV)
    with torch.no_grad():
        assert eq(M(x, res_out=(108, 156)), M(x.float(), res_out=(108, 156)))
