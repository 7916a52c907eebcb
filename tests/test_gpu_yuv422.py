"""GPU: 4:2:2 frames (yuv422p, nv16, p210, yuv422p10le) and LSB-aligned 10-bit planar frames (yuv420p10le, yuv422p10le, yuv444p10le),
dense and as per-frame surfaces.  Every comparison is bitwise: the kernels against the oracle of tests/test_yuv422_host.py, the identity
pairs (yuv420p10le = P010 >> 6, yuv444p10le = yuv444p16 >> 6, yuv422p = nv16 de-interleaved, yuv422p10le = p210 >> 6, the two 4:2:2
identities, LSB words above 1023 read as 1023) on the kernels and on whole forwards, 4:2:2 luma planes against NV12 / P010 outputs, and
surfaces against the dense path.  Surfaces are strided views into sentinel-filled pools (the rules of tests/test_gpu_yuvp.py: pitched
rows, a guard row above each plane, shuffled frame slots, 8-bit planar chroma at odd addresses); every byte outside the valid samples of
the planes' rows must keep its sentinel."""
import pytest
import torch

from tests.golden.cases import CASES, FULLSIZE
from tests.test_gpu_models import build
from tests.test_gpu_p010 import _model, natural_nv12, natural_p010
from tests.test_gpu_yuv_planes import Surfaces
from tests.test_gpu_yuvp import SENTINEL, Surfaces3, engine_fwd, eq, st
from tests.test_yuv422_host import (NEW, code, colours, dense_shape, from_planes, identity_pairs_image, is16, oracle_from_rgb,
                                    oracle_to_rgb, random_frames, to_planes)
from transformerupscaler_b200.synth import synth_frames

pytestmark = pytest.mark.gpu

F32, F16, U8, U16, I32 = torch.float32, torch.float16, torch.uint8, torch.uint16, torch.int32
DEV = torch.device("cuda:0")
PLANES_PER_LAUNCH = 64               # kPlanesPerLaunch of csrc/resample.cu


def _l():
    from transformerupscaler_b200 import _lib
    return _lib, _lib.load()


def hw_of(fmt, f):
    sub = NEW[fmt][0]
    return (f.shape[1] * 2 // 3, f.shape[2]) if sub == "420" else (f.shape[1] // 2, f.shape[2]) if sub == "422" else tuple(f.shape[2:])


class Pools(Surfaces3):
    """B frames of a new layout in strided views of sentinel-filled byte pools, one pool per plane, laid out by Surfaces3's rules: a row
    pitch of the row rounded up to 256 bytes plus an odd multiple of the plane's alignment, a guard row above each plane, shuffled frame
    slots, 8-bit planar chroma at odd addresses.  pitched=False: rows of exactly the row's bytes"""

    def __init__(self, fmt, B, H, W, seed, pitched=True):
        self.fmt, self.B, self.H = fmt, B, H
        sub, self.dt, self.semi = NEW[fmt]
        es = 2 if self.dt == U16 else 1
        if self.semi:
            dims, al = [(H, W), (H, W)], [2 * es, 2 * es]
        else:
            ch, cw = (H // 2 if sub == "420" else H), (W if sub == "444" else W // 2)
            dims, al = [(H, W), (ch, cw), (ch, cw)], [es if sub == "444" else 2 * es, es, es]
        self.perm = torch.randperm(B, generator=torch.Generator().manual_seed(seed)).tolist()
        self.idx = torch.tensor(self.perm, device=DEV)
        self.regions = []
        for p, ((h, w), a) in enumerate(zip(dims, al)):
            row = w * es
            off = (1 if (seed + p) % 2 else 3) if a == 1 and pitched else 0
            pitch = (-(-row // 256) * 256 + a * (2 * ((seed + p) % 3) + 1) + off) if pitched else row
            pool = torch.full((B, h + 2, pitch), SENTINEL, dtype=U8, device=DEV)
            self.regions.append((pool, slice(1, 1 + h), slice(off, off + row)))
        self.planes = [tuple(pool[s, rows, cols].view(self.dt) for pool, rows, cols in self.regions) for s in self.perm]

    def _split(self, f):
        return [f[:, :self.H], f[:, self.H:]] if self.semi else list(to_planes(f, self.fmt))

    def write(self, dense):
        for (pool, rows, cols), plane in zip(self.regions, self._split(dense.to(DEV))):
            pool[self.idx, rows, cols] = plane.contiguous().view(U8)

    def read(self):
        planes = [pool[self.idx, rows, cols].view(self.dt) for pool, rows, cols in self.regions]
        return torch.cat(planes, 1) if self.semi else from_planes(*planes, self.fmt)

    def descriptors(self):
        from transformerupscaler_b200 import engine
        return engine._descriptors(engine._flat(self.planes), code(self.fmt))


def rgb_dtype(fmt):
    return F32 if is16(fmt) else F16


def k_to_rgb(fmt, yuv, f=None, S=None, B=None, H=None, W=None):
    L, lib = _l()
    if f is not None:
        B, (H, W) = f.shape[0], hw_of(fmt, f)
    out = torch.empty(B, 3, H, W, dtype=rgb_dtype(fmt), device=DEV)
    fn = lib.tu_yuv422sp_to_rgb if NEW[fmt][2] else lib.tu_yuvp_to_rgb
    L.check(fn(f.data_ptr() if f is not None else None, S.descriptors() if S is not None else None, code(fmt, yuv), out.data_ptr(),
               B, H, W, st()))
    return out


def k_from_rgb(fmt, yuv, x, S=None):
    L, lib = _l()
    B, _, H, W = x.shape
    out = None if S is not None else torch.empty(dense_shape(fmt, B, H, W), dtype=NEW[fmt][1], device=DEV)
    fn = lib.tu_rgb_to_yuv422sp if NEW[fmt][2] else lib.tu_rgb_to_yuvp
    L.check(fn(x.data_ptr(), out.data_ptr() if out is not None else None, S.descriptors() if S is not None else None, code(fmt, yuv),
               B, H, W, st()))
    return out


def k_other(name, x, c, B, H, W, out_shape=None, out_dtype=None):
    """an existing conversion op (tu_nv12_to_rgb, tu_rgb_to_p010, tu_yuvp_to_rgb, ...) on dense buffers"""
    L, lib = _l()
    if name.endswith("_to_rgb"):
        out = torch.empty(B, 3, H, W, dtype=out_dtype, device=DEV)
        if name == "yuvp_to_rgb":
            L.check(lib.tu_yuvp_to_rgb(x.data_ptr(), None, c, out.data_ptr(), B, H, W, st()))
        else:
            L.check(getattr(lib, "tu_" + name)(x.data_ptr(), c, out.data_ptr(), B, H, W, st()))
    else:
        out = torch.empty(out_shape, dtype=out_dtype, device=DEV)
        if name == "rgb_to_yuvp":
            L.check(lib.tu_rgb_to_yuvp(x.data_ptr(), out.data_ptr(), None, c, B, H, W, st()))
        else:
            L.check(getattr(lib, "tu_" + name)(x.data_ptr(), out.data_ptr(), c, B, H, W, st()))
    return out


# conversions between the layouts of the identity pairs (int32 arithmetic, back to the frame dtype)
def as_words(t):
    return t.to(I32) & 0xFFFF


def p010_to_lsb420(p):
    B, R, W = p.shape
    H = R * 2 // 3
    c = as_words(p) >> 6
    ch = c[:, H:].reshape(B, H // 2, W // 2, 2)
    return from_planes(c[:, :H], ch[..., 0], ch[..., 1], "yuv420p10le").to(U16)


def lsb420_to_p010(f):
    y, u, v = (as_words(t) for t in to_planes(f, "yuv420p10le"))
    B, H, W = y.shape
    return (torch.cat([y, torch.stack([u, v], -1).reshape(B, H // 2, W)], 1) << 6).to(U16)


def p422_to_sp(f, fmt_from, fmt_to):
    """yuv422p <-> nv16 and yuv422p10le <-> p210 (words shifted by 6)"""
    y, u, v = (as_words(t) for t in to_planes(f, fmt_from))
    sh = 6 if fmt_to == "p210" else -6 if fmt_from == "p210" else 0
    if sh:
        y, u, v = ((t << sh) if sh > 0 else (t >> -sh) for t in (y, u, v))
    return from_planes(y, u, v, fmt_to).to(NEW[fmt_to][1])


def natural(fmt, B, H, W, seed, yuv="bt709"):
    rgb = synth_frames(B, H, W, seed=seed)
    return oracle_from_rgb(rgb if is16(fmt) else rgb.half(), fmt, yuv)


def with_stray_bits(f, seed):
    """LSB frames of codes (<= 1023) with random words above 1023 at random places, and the same frames with 1023 there"""
    g = torch.Generator().manual_seed(seed)
    mask = torch.rand(f.shape, generator=g) < 0.2
    hi = torch.randint(1024, 65536, f.shape, generator=g, dtype=I32)
    sat = torch.where(mask, torch.full_like(as_words(f.cpu()), 1023), as_words(f.cpu()))
    return torch.where(mask, hi, sat).to(U16), sat.to(U16)


SIZES = {"420": [(2, 2), (2, 6), (6, 10), (720, 1280), (1080, 1920)],
         "422": [(1, 2), (3, 2), (5, 6), (2, 10), (7, 1282), (720, 1280), (1080, 1920)],      # odd H; W = 2 mod 4
         "444": [(1, 1), (1, 2), (3, 5), (7, 9), (5, 1283), (720, 1280)]}
CASES_K = [(fmt, hw) for fmt in NEW for hw in SIZES[NEW[fmt][0]]]


# ---------------------------------------------------------------------------------------------------------------------------------
# the conversion kernels
@pytest.mark.parametrize("fmt,hw", CASES_K)
def test_kernels_match_oracle_dense_and_surfaces(fmt, hw):
    H, W = hw
    B = 2 if H * W > 100000 else 3
    f = random_frames(fmt, B, H, W, seed=H * 31 + W)
    g = torch.Generator().manual_seed(H * 7 + W)
    x = (torch.rand(B, 3, H, W, generator=g) * 1.6 - 0.3).to(rgb_dtype(fmt))        # values outside [0, 1] too
    cols = colours(fmt)
    if H * W > 100000:
        cols = (cols[0], cols[-1])
    for i, yuv in enumerate(cols):
        want = oracle_to_rgb(f, fmt, yuv).to(rgb_dtype(fmt))
        fd = f.to(DEV)
        assert eq(k_to_rgb(fmt, yuv, fd), want), yuv
        S = Pools(fmt, B, H, W, seed=i, pitched=i % 2 == 0)
        S.write(fd)
        assert eq(k_to_rgb(fmt, yuv, S=S, B=B, H=H, W=W), want) and S.untouched(), yuv
        want = oracle_from_rgb(x, fmt, yuv)
        xd = x.to(DEV)
        assert eq(k_from_rgb(fmt, yuv, xd), want), yuv
        T = Pools(fmt, B, H, W, seed=i + 1, pitched=i % 2 == 1)
        k_from_rgb(fmt, yuv, xd, T)
        assert eq(T.read(), want) and T.untouched(), yuv


@pytest.mark.parametrize("fmt", list(NEW))
def test_batch_larger_than_one_launch(fmt):
    B = PLANES_PER_LAUNCH + 6
    H, W = (6, 10) if NEW[fmt][0] != "422" else (5, 10)
    f = random_frames(fmt, B, H, W, seed=99).to(DEV)
    yuv = "bt2020" if is16(fmt) else "bt601_full"
    want = oracle_to_rgb(f, fmt, yuv).to(rgb_dtype(fmt))
    assert eq(k_to_rgb(fmt, yuv, f), want)
    S = Pools(fmt, B, H, W, seed=4)
    S.write(f)
    assert eq(k_to_rgb(fmt, yuv, S=S, B=B, H=H, W=W), want)
    x = want.to(DEV)
    back = oracle_from_rgb(x.cpu(), fmt, yuv)
    assert eq(k_from_rgb(fmt, yuv, x), back)
    T = Pools(fmt, B, H, W, seed=5, pitched=False)
    k_from_rgb(fmt, yuv, x, T)
    assert eq(T.read(), back) and T.untouched() and S.untouched()


@pytest.mark.parametrize("hw", [(2, 2), (6, 10), (720, 1280)])
def test_kernel_identity_pairs(hw):
    """yuv420p10le = P010 >> 6 and yuv444p10le = yuv444p16 >> 6 (stray high bits of LSB words read as 1023), yuv422p = nv16 and
    yuv422p10le = p210 >> 6, and the 4:2:2 luma planes are the NV12 / P010 luma planes"""
    H, W = hw
    B = 2
    g = torch.Generator().manual_seed(H + W)
    x32 = (torch.rand(B, 3, H, W, generator=g) * 1.4 - 0.2).to(DEV)
    x16 = x32.half()
    for yuv in ("bt709", "bt2020_full", "bt601"):
        from transformerupscaler_b200 import _lib as L, engine
        yc = engine.yuv_code(yuv)
        # yuv420p10le against P010
        stray, sat = with_stray_bits(random_frames("yuv420p10le", B, H, W, seed=1, hi=1024), seed=2)
        p010 = lsb420_to_p010(sat.to(DEV))
        assert eq(k_to_rgb("yuv420p10le", yuv, stray.to(DEV)), k_other("p010_to_rgb", p010, L.TU_U16 | L.TU_LAYOUT_P010 | yc, B, H, W,
                                                                           out_dtype=F32)), yuv
        assert eq(lsb420_to_p010(k_from_rgb("yuv420p10le", yuv, x32)),
                  k_other("rgb_to_p010", x32, L.TU_U16 | L.TU_LAYOUT_P010 | yc, B, H, W, (B, 3 * H // 2, W), U16)), yuv
        # yuv444p10le against yuv444p16
        stray, sat = with_stray_bits(random_frames("yuv444p10le", B, H, W, seed=3, hi=1024), seed=4)
        p16 = L.TU_U16 | L.TU_LAYOUT_YUV444P | yc
        assert eq(k_to_rgb("yuv444p10le", yuv, stray.to(DEV)),
                  k_other("yuvp_to_rgb", (as_words(sat) << 6).to(U16).to(DEV), p16, B, H, W, out_dtype=F32)), yuv
        assert eq((as_words(k_from_rgb("yuv444p10le", yuv, x32)) << 6).to(U16),
                  k_other("rgb_to_yuvp", x32, p16, B, H, W, (B, 3, H, W), U16)), yuv
        # yuv422p10le against p210, LSB stray bits included
        stray, sat = with_stray_bits(random_frames("yuv422p10le", B, H, W, seed=5, hi=1024), seed=6)
        assert eq(k_to_rgb("yuv422p10le", yuv, stray.to(DEV)), k_to_rgb("p210", yuv, p422_to_sp(sat.to(DEV), "yuv422p10le", "p210"))), yuv
        out10 = k_from_rgb("yuv422p10le", yuv, x32)
        out210 = k_from_rgb("p210", yuv, x32)
        assert eq(p422_to_sp(out10, "yuv422p10le", "p210"), out210), yuv
        # 4:2:2 luma = 4:2:0 luma
        assert eq(out210[:, :H], k_other("rgb_to_p010", x32, L.TU_U16 | L.TU_LAYOUT_P010 | yc, B, H, W, (B, 3 * H // 2, W), U16)[:, :H])
        if yuv.startswith("bt2020"):
            continue
        f8 = random_frames("yuv422p", B, H, W, seed=7).to(DEV)
        assert eq(k_to_rgb("yuv422p", yuv, f8), k_to_rgb("nv16", yuv, p422_to_sp(f8, "yuv422p", "nv16"))), yuv
        o8 = k_from_rgb("yuv422p", yuv, x16)
        assert eq(p422_to_sp(o8, "yuv422p", "nv16"), k_from_rgb("nv16", yuv, x16)), yuv
        assert eq(o8[:, :H], k_other("rgb_to_nv12", x16, L.TU_U8 | L.TU_LAYOUT_NV12 | yc, B, H, W, (B, 3 * H // 2, W), U8)[:, :H])


@pytest.mark.parametrize("fmt", ["nv16", "p210", "yuv422p", "yuv422p10le"])
def test_kernel_422_identities(fmt):
    """identity 1: an image whose rows come in equal pairs gives 4:2:2 chroma rows 2i, 2i+1 equal to the NV12 / P010 kernel's chroma row
    i; identity 2: a frame whose chroma is constant along each row converts to the RGB of the yuv444p / yuv444p16 kernel"""
    from transformerupscaler_b200 import _lib as L, engine
    B, H, W = 2, 720, 1282 if fmt != "p210" else 1280
    w16 = is16(fmt)
    rgb = identity_pairs_image(B, H, W, seed=3, w16=w16).to(DEV)
    for yuv in colours(fmt)[::2]:
        yc = engine.yuv_code(yuv)
        y, u, v = (as_words(t) for t in to_planes(k_from_rgb(fmt, yuv, rgb), fmt))
        if fmt == "p210":
            y, u, v = y >> 6, u >> 6, v >> 6
        if w16:
            f420 = as_words(k_other("rgb_to_p010", rgb, L.TU_U16 | L.TU_LAYOUT_P010 | yc, B, H, W, (B, 3 * H // 2, W), U16)) >> 6
        else:
            f420 = as_words(k_other("rgb_to_nv12", rgb, L.TU_U8 | L.TU_LAYOUT_NV12 | yc, B, H, W, (B, 3 * H // 2, W), U8))
        ch = f420[:, H:].reshape(B, H // 2, W // 2, 2)
        assert eq(y, f420[:, :H]), yuv
        assert eq(u, ch[..., 0].repeat_interleave(2, 1)) and eq(v, ch[..., 1].repeat_interleave(2, 1)), yuv
        # identity 2
        f = random_frames(fmt, B, H, W, seed=11).to(DEV)
        yy, uu, vv = to_planes(f, fmt)
        f = from_planes(yy, uu[..., :1].expand_as(uu), vv[..., :1].expand_as(vv), fmt).contiguous()
        yy, uu, vv = (as_words(t) for t in to_planes(f, fmt))
        if fmt.endswith("10le"):
            yy, uu, vv = yy.clamp(max=1023) << 6, uu.clamp(max=1023) << 6, vv.clamp(max=1023) << 6
        f444 = torch.stack([yy, uu[..., :1].expand(B, H, W), vv[..., :1].expand(B, H, W)], 1).to(U16 if w16 else U8)
        c444 = (L.TU_U16 if w16 else L.TU_U8) | L.TU_LAYOUT_YUV444P | yc
        assert eq(k_to_rgb(fmt, yuv, f), k_other("yuvp_to_rgb", f444.contiguous(), c444, B, H, W, out_dtype=F32 if w16 else F16)), yuv


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
            # yuv422p = nv16 de-interleaved, in and out; the forward is the fp16 one of the converted frame
            f8 = natural("yuv422p", B, H, W, seed=s, yuv="bt601").to(DEV)
            got = M(f8, in_layout="yuv422p", out_layout="yuv422p", yuv="bt601", **kw)
            oh, ow = got.shape[1] // 2, got.shape[2]
            want = M(p422_to_sp(f8, "yuv422p", "nv16"), in_layout="nv16", out_layout="nv16", yuv="bt601", **kw)
            assert got.dtype == U8 and eq(p422_to_sp(got, "yuv422p", "nv16"), want)
            assert eq(got, engine_fwd(M, k_to_rgb("yuv422p", "bt601", f8), bf16, U8, kw, out_layout="yuv422p", yuv="bt601"))
            assert eq(got, k_from_rgb("yuv422p", "bt601", engine_fwd(M, f8, bf16, F16, kw, in_layout="yuv422p", yuv="bt601")))
            # yuv420p10le = P010 >> 6, in and out
            p10 = natural_p010(B, H, W, seed=s + 1, yuv="bt2020").to(DEV)
            got = M(p010_to_lsb420(p10), in_layout="yuv420p10le", out_layout="yuv420p10le", yuv="bt2020", **kw)
            assert got.dtype == U16 and eq(lsb420_to_p010(got), M(p10, in_layout="p010", out_layout="p010", yuv="bt2020", **kw))
            # yuv422p10le = p210 >> 6; the forward is the fp32 one of the converted frame
            f10 = natural("yuv422p10le", B, H, W, seed=s + 2, yuv="bt709_full").to(DEV)
            got = M(f10, in_layout="yuv422p10le", out_layout="yuv422p10le", yuv="bt709_full", **kw)
            want = M(p422_to_sp(f10, "yuv422p10le", "p210"), in_layout="p210", out_layout="p210", yuv="bt709_full", **kw)
            assert got.dtype == U16 and eq(p422_to_sp(got, "yuv422p10le", "p210"), want)
            rgb32 = k_to_rgb("yuv422p10le", "bt709_full", f10)
            assert eq(got, engine_fwd(M, rgb32, bf16, U16, kw, out_layout="yuv422p10le", yuv="bt709_full"))
            assert eq(want, k_from_rgb("p210", "bt709_full", engine_fwd(M, f10, bf16, F32, kw, in_layout="yuv422p10le", yuv="bt709_full")))
            # yuv444p10le = yuv444p16 >> 6, and words above 1023 read as 1023
            f444 = natural("yuv444p10le", B, H, W, seed=s + 3, yuv="bt601").to(DEV)
            got = M(f444, in_layout="yuv444p10le", out_layout="yuv444p10le", yuv="bt601", **kw)
            want = M((as_words(f444) << 6).to(U16), in_layout="yuv444p16", out_layout="yuv444p16", yuv="bt601", **kw)
            assert got.dtype == U16 and got.shape == (B, 3, oh, ow) and eq((as_words(got) << 6).to(U16), want)
            stray, sat = with_stray_bits(f444, seed=s)
            assert eq(M(stray.to(DEV), in_layout="yuv444p10le", out_layout="hwc", **kw), M(sat.to(DEV), in_layout="yuv444p10le",
                                                                                          out_layout="hwc", **kw))
            # the luma planes of 4:2:2 outputs are those of the NV12 / P010 outputs of the same forward
            xu = (torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(s)) * 255).to(U8).to(DEV)
            assert eq(M(xu, out_layout="nv16", **kw)[:, :oh], M(xu, out_layout="nv12", **kw)[:, :oh])
            p010_y = M(xu, out_layout="p010", **kw)[:, :oh]
            assert eq(M(xu, out_layout="p210", **kw)[:, :oh], p010_y)
            assert eq((as_words(M(xu, out_layout="yuv422p10le", **kw)[:, :oh]) << 6).to(U16), p010_y)
            # identity 2 on a forward: row-constant 4:2:2 chroma is the yuv444p input holding it everywhere
            y, u, v = to_planes(f8, "yuv422p")
            fc = from_planes(y, u[..., :1].expand_as(u), v[..., :1].expand_as(v), "yuv422p").contiguous()
            f444c = torch.stack([y, u[..., :1].expand(B, H, W), v[..., :1].expand(B, H, W)], 1).contiguous()
            assert eq(M(fc, in_layout="yuv422p", **kw), M(f444c, in_layout="yuv444p", **kw))
            # mixed sides: dense yuv420p10le in -> BGRA out; NV12 surfaces in -> yuv422p10le surfaces out; p210 surfaces -> nv16 surfaces;
            # yuv420p10le surfaces -> yuv422p dense
            lsb = p010_to_lsb420(p10)
            assert eq(M(lsb, in_layout="yuv420p10le", out_layout="bgra", yuv="bt2020", **kw),
                      engine_fwd(M, k_to_rgb("yuv420p10le", "bt2020", lsb), bf16, U8, kw, out_layout="bgra"))
            nv = natural_nv12(B, H, W, seed=s + 4).to(DEV)
            S = Surfaces("nv12", B, H, W, split=True, seed=s)
            S.write(nv)
            O = Pools("yuv422p10le", B, oh, ow, seed=s)
            assert M(S.planes, in_layout="nv12", out_layout="yuv422p10le", out=O.planes, **kw) is O.planes
            assert eq(O.read(), M(nv, in_layout="nv12", out_layout="yuv422p10le", **kw)) and O.untouched() and S.untouched()
            p210 = p422_to_sp(f10, "yuv422p10le", "p210")
            P = Pools("p210", B, H, W, seed=s + 1)
            P.write(p210)
            O = Pools("nv16", B, oh, ow, seed=s + 2)
            M(P.planes, in_layout="p210", out_layout="nv16", yuv="bt709_full", out=O.planes, **kw)
            want = M(p210, in_layout="p210", out_layout="nv16", yuv="bt709_full", **kw)
            assert eq(O.read(), want) and O.untouched() and P.untouched()
            Q = Pools("yuv420p10le", B, H, W, seed=s + 3)
            Q.write(lsb)
            assert eq(M(Q.planes, in_layout="yuv420p10le", out_layout="yuv422p", **kw), M(lsb, in_layout="yuv420p10le", out_layout="yuv422p",
                                                                                            **kw))
            R = Pools("yuv444p10le", B, oh, ow, seed=s + 4)
            M(f8, in_layout="yuv422p", out_layout="yuv444p10le", out=R.planes, **kw)
            assert eq(R.read(), M(f8, in_layout="yuv422p", out_layout="yuv444p10le", **kw)) and R.untouched()
    finally:
        M.engine_precision = None


def test_forward_batch_larger_than_one_launch():
    M = _model("window_72x104_r1p5")
    B = PLANES_PER_LAUNCH + 6
    f = natural("yuv422p", B, 72, 104, seed=5).to(DEV)
    S = Pools("yuv422p", B, 72, 104, seed=6)
    S.write(f)
    O = Pools("p210", B, 108, 156, seed=7)
    with torch.no_grad():
        M(S.planes, in_layout="yuv422p", out_layout="p210", out=O.planes, res_out=(108, 156))
        want = M(f, in_layout="yuv422p", out_layout="p210", res_out=(108, 156))
    assert eq(O.read(), want) and O.untouched() and S.untouched()


def test_fullsize_window_yuv420p10le_is_p010_bf16():
    c = FULLSIZE["window_720p_1080p_b8"]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    p10 = natural_p010(B, H, W, seed=c["xseed"]).to(DEV)
    with torch.no_grad():
        want = M(p10, in_layout="p010", out_layout="p010", **c["kw"])
        got = M(p010_to_lsb420(p10), in_layout="yuv420p10le", out_layout="yuv420p10le", **c["kw"])
        assert eq(lsb420_to_p010(got), want)
        S = Pools("yuv420p10le", B, H, W, seed=1)
        S.write(p010_to_lsb420(p10))
        O = Pools("yuv420p10le", B, 1080, 1920, seed=2, pitched=False)
        M(S.planes, in_layout="yuv420p10le", out_layout="yuv420p10le", out=O.planes, **c["kw"])
    assert eq(O.read(), got) and O.untouched()
    assert int(as_words(got).max()) <= 1023                                            # top 6 bits zero


def test_fullsize_residual_yuv422p10le_bf16():
    c = FULLSIZE["residual_720p_4k"]
    B, _, H, W = c["shape"]
    M, _ = build(c["model"], c["wseed"])
    M.engine_precision = "bf16"
    f = natural("yuv422p10le", B, H, W, seed=c["xseed"], yuv="bt2020").to(DEV)
    kw = dict(in_layout="yuv422p10le", out_layout="yuv422p10le", yuv="bt2020", **c["kw"])
    with torch.no_grad():
        want = M(f, **kw)
        assert want.shape == (B, 4320, 3840)
        assert eq(p422_to_sp(want, "yuv422p10le", "p210"),
                  M(p422_to_sp(f, "yuv422p10le", "p210"), in_layout="p210", out_layout="p210", yuv="bt2020", **c["kw"]))
        S = Pools("yuv422p10le", B, H, W, seed=3)
        S.write(f)
        O = Pools("yuv422p10le", B, 2160, 3840, seed=4)
        M(S.planes, out=O.planes, **kw)
    assert eq(O.read(), want) and O.untouched()
    assert int(as_words(want).max()) <= 1023


# ---------------------------------------------------------------------------------------------------------------------------------
# wrappers
def test_graphed_model_frame_pipeline_and_compile():
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.pipeline import FramePipeline
    M = _model("window_72x104_r1p5")
    for fmt, ofmt, yuv, oshape in (("yuv420p10le", "yuv422p10le", "bt2020", (2, 216, 156)),
                                   ("p210", "yuv444p10le", "bt601_full", (2, 3, 108, 156)),
                                   ("nv16", "yuv422p", "bt709", (2, 216, 156))):
        kw = dict(res_out=(108, 156), in_layout=fmt, out_layout=ofmt, yuv=yuv)
        xs = [natural(fmt, 2, 72, 104, seed=700 + i, yuv=yuv) for i in range(4)]
        with torch.no_grad():
            eager = [M(x.to(DEV), **kw).clone() for x in xs]
        assert eager[0].shape == oshape and eager[0].dtype == NEW[ofmt][1]
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
    # surfaces out under torch.compile
    f = natural("yuv422p", 1, 72, 104, seed=9).to(DEV)
    kw = dict(in_layout="yuv422p", out_layout="p210", res_out=(108, 156))
    with torch.no_grad():
        want = M(f, **kw)
        O = Pools("p210", 1, 108, 156, seed=1)
        torch.compile(M)(f, out=O.planes, **kw)
    assert eq(O.read(), want) and O.untouched()
    # the Resize path ends in tu::rgb_to_yuv422sp / tu::rgb_to_yuvp (compiled) and their _planes forms (eager)
    Mf = _model("fast_40x56_res60x84")
    for fin, fout in (("nv16", "nv16"), ("yuv420p10le", "yuv422p10le"), ("p210", "yuv444p10le")):
        f = natural(fin, 1, 40, 56, seed=3).to(DEV)
        kw = dict(in_layout=fin, out_layout=fout, res_out=(60, 84))
        with torch.no_grad():
            want = Mf(f, **kw)
            assert want.shape == dense_shape(fout, 1, 60, 84) and eq(torch.compile(Mf)(f, **kw), want)
            O = Pools(fout, 1, 60, 84, seed=1)
            Mf(f, out=O.planes, **kw)
        assert eq(O.read(), want) and O.untouched()
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(M)(O.planes, in_layout=fout, res_out=(108, 156))
