"""GPU: NV12 / P010 frames read from and written into per-frame decoder / encoder surfaces (TuFramePlanes: two planes with row
pitches, anywhere in device memory).

Every comparison is bitwise against the dense (B, 3H/2, W) path on the same frame contents.  Surfaces are strided views into
sentinel-filled pools the way decoders and encoders lay them out: a row pitch of W rounded up to 256 bytes plus an odd multiple of the
alignment, a guard row above each plane, the chroma plane in a separate allocation or at an aligned-height offset behind the luma,
and the frames of a batch at shuffled slots.  Every byte outside the W samples of the planes' rows must keep its sentinel."""
import gc

import pytest
import torch

from tests.golden.cases import CASES, FULLSIZE
from tests.test_gpu_models import build
from tests.test_gpu_p010 import _model, natural_nv12, natural_p010
from tests.test_nv12_host import COLOURS, flat_chroma_frames
from tests.test_p010_host import COLOURS10, flat_chroma_frames10

pytestmark = pytest.mark.gpu

F32, F16, U8, U16 = torch.float32, torch.float16, torch.uint8, torch.uint16
DEV = torch.device("cuda:0")
SENTINEL = 0xA5                      # every pool byte: 0xA5 in NV12 pools, the word 0xA5A5 in P010 pools
PLANES_PER_LAUNCH = 64               # kPlanesPerLaunch of csrc/resample.cu


class Surfaces:
    """B frame surfaces of H x W samples in strided views of sentinel-filled byte pools"""

    def __init__(self, fmt, B, H, W, split, seed):
        self.p010 = fmt == "p010"
        es, al = (2, 4) if self.p010 else (1, 2)
        self.B, self.H, self.row = B, H, W * es
        self.pitch = -(-self.row // 256) * 256 + al * (2 * (seed % 3) + 1)
        self.split = split
        self.Hal = -(-H // 16) * 16 + 16                                 # the chroma plane's row in a shared pool (1088 for 1072 ...)
        self.perm = torch.randperm(B, generator=torch.Generator().manual_seed(seed)).tolist()
        if split:
            self.pools = [torch.full((B, H + 2, self.pitch), SENTINEL, dtype=U8, device=DEV),
                          torch.full((B, H // 2 + 2, self.pitch), SENTINEL, dtype=U8, device=DEV)]
        else:
            self.pools = [torch.full((B, self.Hal + H // 2 + 1, self.pitch), SENTINEL, dtype=U8, device=DEV)]
        dt = U16 if self.p010 else U8
        self.planes = [(y.view(dt), c.view(dt)) for y, c in self._views(self.pools)]

    def _views(self, pools):
        """byte views (y, uv) of every frame in `pools`"""
        H, r = self.H, self.row
        yp, cp = (pools[0], pools[1]) if self.split else (pools[0], pools[0])
        c0 = 1 if self.split else self.Hal
        return [(yp[s, 1:1 + H, :r], cp[s, c0:c0 + H // 2, :r]) for s in self.perm]

    def _regions(self, pools):
        """(pool, frame slots, rows, columns) of the luma and the chroma planes, for batched indexing"""
        H, r, idx = self.H, self.row, torch.tensor(self.perm, device=DEV)
        if self.split:
            return [(pools[0], idx, slice(1, 1 + H), slice(0, r)), (pools[1], idx, slice(1, 1 + H // 2), slice(0, r))]
        return [(pools[0], idx, slice(1, 1 + H), slice(0, r)), (pools[0], idx, slice(self.Hal, self.Hal + H // 2), slice(0, r))]

    def write(self, dense):
        """copy dense frames (B, 3H/2, W) into the surfaces, in place"""
        d = dense.to(DEV).contiguous().view(U8)
        (yp, i, yr, yc), (cp, _, cr, cc) = self._regions(self.pools)
        yp[i, yr, yc] = d[:, :self.H]
        cp[i, cr, cc] = d[:, self.H:]

    def read(self):
        """the surfaces' frames as a dense (B, 3H/2, W) tensor"""
        (yp, i, yr, yc), (cp, _, cr, cc) = self._regions(self.pools)
        d = torch.cat([yp[i, yr, yc], cp[i, cr, cc]], 1)
        return d.view(U16) if self.p010 else d

    def untouched(self):
        """every byte outside the planes' rows still holds the sentinel"""
        clones = [p.clone() for p in self.pools]
        for p, i, rows, cols in self._regions(clones):
            p[i, rows, cols] = SENTINEL
        return all(bool((p == SENTINEL).all()) for p in clones)


def _l():
    from transformerupscaler_b200 import _lib
    return _lib, _lib.load()


def code(fmt, yuv):
    from transformerupscaler_b200 import _lib, engine
    base = _lib.TU_U16 | _lib.TU_LAYOUT_P010 if fmt == "p010" else _lib.TU_U8 | _lib.TU_LAYOUT_NV12
    return base | engine.yuv_code(yuv)


def st():
    return torch.cuda.current_stream().cuda_stream


def rgb_dtype(fmt):
    return F32 if fmt == "p010" else F16


CHUNK = 32768                        # frames per call of a dense op (its grid's y dimension holds at most 65535)


def dense_to_rgb(fmt, f, yuv):
    L, lib = _l()
    B, R, W = f.shape
    H = R * 2 // 3
    out = torch.empty(B, 3, H, W, dtype=rgb_dtype(fmt), device=DEV)
    op = lib.tu_p010_to_rgb if fmt == "p010" else lib.tu_nv12_to_rgb
    for b0 in range(0, B, CHUNK):
        n = min(CHUNK, B - b0)
        L.check(op(f[b0:].data_ptr(), code(fmt, yuv), out[b0:].data_ptr(), n, H, W, st()))
    return out


def planes_to_rgb(fmt, S, yuv):
    from transformerupscaler_b200 import engine
    L, lib = _l()
    W = S.planes[0][0].shape[1]
    out = torch.empty(S.B, 3, S.H, W, dtype=rgb_dtype(fmt), device=DEV)
    L.check(lib.tu_yuv420_planes_to_rgb(engine._descriptors(engine._flat(S.planes)), code(fmt, yuv), out.data_ptr(), S.B, S.H, W, st()))
    return out


def rgb_to_dense(fmt, x, yuv):
    L, lib = _l()
    B, _, H, W = x.shape
    out = torch.empty(B, 3 * H // 2, W, dtype=U16 if fmt == "p010" else U8, device=DEV)
    op = lib.tu_rgb_to_p010 if fmt == "p010" else lib.tu_rgb_to_nv12
    for b0 in range(0, B, CHUNK):
        n = min(CHUNK, B - b0)
        L.check(op(x[b0:].data_ptr(), out[b0:].data_ptr(), code(fmt, yuv), n, H, W, st()))
    return out


def rgb_to_planes(fmt, x, S, yuv):
    from transformerupscaler_b200 import engine
    L, lib = _l()
    B, _, H, W = x.shape
    L.check(lib.tu_rgb_to_yuv420_planes(x.data_ptr(), engine._descriptors(engine._flat(S.planes)), code(fmt, yuv), B, H, W, st()))


def random_frames(fmt, B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    hi = 65536 if fmt == "p010" else 256
    return torch.randint(0, hi, (B, 3 * H // 2, W), generator=g, dtype=torch.int32).to(U16 if fmt == "p010" else U8).to(DEV)


FMT_COLOURS = [("nv12", y) for y in COLOURS] + [("p010", y) for y in COLOURS10]
SIZES = [(2, 2), (2, 6), (2, 10), (4, 1280), (720, 10), (720, 1280)]     # edge sizes; W = 2 (mod 4)


# ---------------------------------------------------------------------------------------------------------------------------------
# the conversion ops
@pytest.mark.parametrize("fmt,yuv", FMT_COLOURS)
@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("split", [True, False])
def test_planes_to_rgb_equals_dense(fmt, yuv, hw, split):
    H, W = hw
    f = random_frames(fmt, 3, H, W, seed=H * 13 + W)
    S = Surfaces(fmt, 3, H, W, split, seed=H + W)
    S.write(f)
    assert torch.equal(planes_to_rgb(fmt, S, yuv), dense_to_rgb(fmt, f, yuv))
    assert S.untouched()


@pytest.mark.parametrize("fmt,yuv", FMT_COLOURS)
@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("split", [True, False])
def test_rgb_to_planes_equals_dense(fmt, yuv, hw, split):
    H, W = hw
    g = torch.Generator().manual_seed(H * 17 + W)
    x = (torch.rand(3, 3, H, W, generator=g) * 1.6 - 0.3).to(rgb_dtype(fmt)).to(DEV)     # values outside [0, 1] too
    S = Surfaces(fmt, 3, H, W, split, seed=H + 2 * W)
    rgb_to_planes(fmt, x, S, yuv)
    assert torch.equal(S.read(), rgb_to_dense(fmt, x, yuv))
    assert S.untouched()


@pytest.mark.parametrize("fmt,yuv", FMT_COLOURS)
def test_chroma_lattice_both_directions(fmt, yuv):
    """every (Y, U, V) lattice case of the dense kernels' tests, as surfaces: many more frames than one launch's table"""
    f = (flat_chroma_frames10() if fmt == "p010" else flat_chroma_frames()).to(DEV)
    B, R, W = f.shape
    H = R * 2 // 3
    S = Surfaces(fmt, B, H, W, split=fmt == "nv12", seed=7)
    S.write(f)
    rgb = dense_to_rgb(fmt, f, yuv)
    assert torch.equal(planes_to_rgb(fmt, S, yuv), rgb)
    T = Surfaces(fmt, B, H, W, split=fmt == "p010", seed=8)
    rgb_to_planes(fmt, rgb, T, yuv)
    assert torch.equal(T.read(), rgb_to_dense(fmt, rgb, yuv))
    assert S.untouched() and T.untouched()


@pytest.mark.parametrize("fmt", ["nv12", "p010"])
def test_split_launches(fmt):
    """B = K + 6 frames: two launches, the second with the RGB side offset to frame K"""
    B, H, W = PLANES_PER_LAUNCH + 6, 6, 10
    f = random_frames(fmt, B, H, W, seed=99)
    S = Surfaces(fmt, B, H, W, split=True, seed=4)
    S.write(f)
    yuv = "bt2020" if fmt == "p010" else "bt601"
    rgb = dense_to_rgb(fmt, f, yuv)
    assert torch.equal(planes_to_rgb(fmt, S, yuv), rgb)
    T = Surfaces(fmt, B, H, W, split=False, seed=5)
    rgb_to_planes(fmt, rgb, T, yuv)
    assert torch.equal(T.read(), rgb_to_dense(fmt, rgb, yuv)) and T.untouched()


# ---------------------------------------------------------------------------------------------------------------------------------
# whole forwards
FWD_CASES = ["window_72x104_r1p5", "window_64x80_x2", "fast_40x56_x2", "fast_36x52_x2_reflect", "fast_24x32_x6",
             "fast_40x56_res60x84", "residual_720p_1080p"]          # fast_40x56_res60x84: the Resize path, ending in the surfaces op


def _out_hw(dense_out):
    return dense_out.shape[1] * 2 // 3, dense_out.shape[2]


@pytest.mark.parametrize("name", FWD_CASES)
@pytest.mark.parametrize("path", ["bf16", "fp32"])
def test_forward_with_surfaces_equals_dense(name, path):
    c = CASES[name]
    B, _, H, W = c["shape"]
    kw = c["kw"]
    M = _model(name)
    M.engine_precision = path
    try:
        with torch.no_grad():
            f = natural_nv12(B, H, W, seed=c["xseed"], yuv="bt709").to(DEV)
            S = Surfaces("nv12", B, H, W, split=False, seed=c["xseed"])
            S.write(f)
            want = M(f, in_layout="nv12", out_layout="nv12", **kw)
            oh, ow = _out_hw(want)
            # surfaces in, dense out
            got = M(S.planes, in_layout="nv12", out_layout="nv12", **kw)
            assert got.dtype == U8 and torch.equal(got, want)
            # dense in, surfaces out: the same list comes back
            O = Surfaces("nv12", B, oh, ow, split=True, seed=c["xseed"] + 1)
            assert M(f, in_layout="nv12", out_layout="nv12", out=O.planes, **kw) is O.planes
            assert torch.equal(O.read(), want) and O.untouched()
            # surfaces on both sides
            O = Surfaces("nv12", B, oh, ow, split=False, seed=c["xseed"] + 2)
            M(S.planes, in_layout="nv12", out_layout="nv12", out=O.planes, **kw)
            assert torch.equal(O.read(), want) and O.untouched()
            # NV12 surfaces -> P010 surfaces
            want10 = M(f, in_layout="nv12", out_layout="p010", **kw)
            O10 = Surfaces("p010", B, oh, ow, split=True, seed=c["xseed"] + 3)
            M(S.planes, in_layout="nv12", out_layout="p010", out=O10.planes, **kw)
            assert torch.equal(O10.read(), want10) and O10.untouched()
            # NV12 surfaces -> HWC BGR
            bgr = M(S.planes, in_layout="nv12", out_layout="hwc_bgr", **kw)
            assert torch.equal(bgr, M(f, in_layout="nv12", out_layout="hwc_bgr", **kw))
            # P010 surfaces (BT.2020) in, P010 dense and surfaces out, and dense uint8 in -> P010 surfaces
            p = natural_p010(B, H, W, seed=c["xseed"] + 4, yuv="bt2020").to(DEV)
            P = Surfaces("p010", B, H, W, split=False, seed=c["xseed"] + 5)
            P.write(p)
            want = M(p, in_layout="p010", out_layout="p010", yuv="bt2020", **kw)
            assert torch.equal(M(P.planes, in_layout="p010", out_layout="p010", yuv="bt2020", **kw), want)
            O10 = Surfaces("p010", B, oh, ow, split=False, seed=c["xseed"] + 6)
            M(P.planes, in_layout="p010", out_layout="p010", yuv="bt2020", out=O10.planes, **kw)
            assert torch.equal(O10.read(), want) and O10.untouched()
            xu = (torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(3)) * 255).to(U8).to(DEV)
            O10 = Surfaces("p010", B, oh, ow, split=True, seed=c["xseed"] + 7)
            M(xu, out_layout="p010", out=O10.planes, **kw)
            assert torch.equal(O10.read(), M(xu, out_layout="p010", **kw)) and O10.untouched()
            assert S.untouched() and P.untouched()
    finally:
        M.engine_precision = None


def test_forward_batch_larger_than_one_launch():
    M = _model("window_72x104_r1p5")
    B = PLANES_PER_LAUNCH + 6
    f = natural_nv12(B, 72, 104, seed=5).to(DEV)
    S = Surfaces("nv12", B, 72, 104, split=True, seed=6)
    S.write(f)
    O = Surfaces("nv12", B, 108, 156, split=False, seed=7)
    with torch.no_grad():
        M(S.planes, in_layout="nv12", out_layout="nv12", out=O.planes, res_out=(108, 156))
        want = M(f, in_layout="nv12", out_layout="nv12", res_out=(108, 156))
    assert torch.equal(O.read(), want) and O.untouched()


@pytest.mark.parametrize("name,fmt,yuv", [("window_720p_1080p_b8", "nv12", "bt709"), ("residual_720p_4k", "p010", "bt2020")])
def test_fullsize_surfaces_to_surfaces_bf16(name, fmt, yuv):
    c = FULLSIZE[name]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    oh, ow = c["kw"]["res_out"]
    f = (natural_p010 if fmt == "p010" else natural_nv12)(B, H, W, seed=c["xseed"], yuv=yuv).to(DEV)
    S = Surfaces(fmt, B, H, W, split=False, seed=1)                      # chroma at the aligned height, as NVDEC maps it
    S.write(f)
    O = Surfaces(fmt, B, oh, ow, split=True, seed=2)
    with torch.no_grad():
        M(S.planes, in_layout=fmt, out_layout=fmt, yuv=yuv, out=O.planes, **c["kw"])
        want = M(f, in_layout=fmt, out_layout=fmt, yuv=yuv, **c["kw"])
    assert torch.equal(O.read(), want) and O.untouched()


# ---------------------------------------------------------------------------------------------------------------------------------
# graphs, torch.compile, wrappers
def test_graph_replays_surfaces_with_no_host_descriptors_alive():
    M = _model("window_72x104_r1p5")
    kw = dict(res_out=(108, 156), in_layout="nv12", out_layout="p010")
    f1, f2 = natural_nv12(2, 72, 104, seed=21).to(DEV), natural_nv12(2, 72, 104, seed=22).to(DEV)
    S = Surfaces("nv12", 2, 72, 104, split=False, seed=3)
    O = Surfaces("p010", 2, 108, 156, split=True, seed=4)
    S.write(f1)
    planes_in, planes_out = list(S.planes), list(O.planes)
    with torch.no_grad():
        s = torch.cuda.Stream(DEV)
        s.wait_stream(torch.cuda.current_stream(DEV))
        with torch.cuda.stream(s):
            M(planes_in, out=planes_out, **kw)                           # packs the weights outside the capture
        torch.cuda.current_stream(DEV).wait_stream(s)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            M(planes_in, out=planes_out, **kw)
    del planes_in, planes_out                                            # the descriptor lists (and their ctypes tables) are gone
    S.planes = O.planes = None
    gc.collect()
    S.write(f2)                                                          # new contents in the same surfaces
    O.write(torch.zeros(2, 162, 156, dtype=U16))
    g.replay()
    torch.cuda.synchronize()
    with torch.no_grad():
        want = M(f2, **kw)
    assert torch.equal(O.read(), want) and O.untouched()


def test_compile_with_out_equals_eager():
    M = _model("window_72x104_r1p5")
    f = natural_nv12(1, 72, 104, seed=31).to(DEV)
    S = Surfaces("nv12", 1, 72, 104, split=True, seed=1)
    S.write(f)
    A, Bo = Surfaces("nv12", 1, 108, 156, split=False, seed=2), Surfaces("nv12", 1, 108, 156, split=False, seed=3)
    kw = dict(res_out=(108, 156), in_layout="nv12", out_layout="nv12")
    with torch.no_grad():
        M(S.planes, out=A.planes, **kw)
        torch.compile(M)(S.planes, out=Bo.planes, **kw)
    assert torch.equal(A.read(), Bo.read()) and Bo.untouched()
    assert torch.equal(A.read(), M(f, **kw))


def test_graphed_model_and_frame_pipeline_reject_planes():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M = _model("window_72x104_r1p5")
    S = Surfaces("nv12", 1, 72, 104, split=True, seed=1)
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(M)(S.planes, in_layout="nv12", res_out=(108, 156))
    pipe = FramePipeline(M, depth=2, device=DEV, in_layout="nv12", res_out=(108, 156))
    with pytest.raises(TypeError, match="frame planes"):
        pipe.submit(S.planes, torch.empty(1, 3, 108, 156, dtype=U8).pin_memory())
