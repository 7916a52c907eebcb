"""CPU: NV12 / P010 frames as per-frame decoder / encoder surfaces (TuFramePlanes) -- the C layout of the descriptor, every host-side
rejection of tu_yuv420_planes_to_rgb, tu_rgb_to_yuv420_planes and tu_forward_planes (all made before anything is enqueued, so they
run without a GPU), the workspace of a surfaces call, and the Python-side errors that need no device."""
import ctypes as C
import subprocess

import pytest
import torch

from tests.test_abi import HEADER
from tests.test_nv12_host import _packed

FAKE = 1 << 20                       # never dereferenced: every call below fails its checks before any launch


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from transformerupscaler_b200 import _lib
    return _lib.load()


def L():
    from transformerupscaler_b200 import _lib
    return _lib


def test_frame_planes_layout_matches_c(lib, tmp_path):
    src = tmp_path / "fp.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu %%zu %%zu %%zu\\n",'
                   'sizeof(TuFramePlanes),offsetof(TuFramePlanes,y),offsetof(TuFramePlanes,uv),offsetof(TuFramePlanes,y_pitch),'
                   'offsetof(TuFramePlanes,uv_pitch));return 0;}\n' % HEADER)
    exe = tmp_path / "fp"
    subprocess.check_call(["gcc", str(src), "-o", str(exe)])
    got = [int(t) for t in subprocess.check_output([str(exe)]).split()]
    P = L().TuFramePlanes
    assert got == [C.sizeof(P), P.y.offset, P.uv.offset, P.y_pitch.offset, P.uv_pitch.offset] == [32, 0, 8, 16, 24]


def frames(B, W, sample, pitch_extra=256):
    """B valid descriptors of W-sample rows (fake, aligned addresses)"""
    pitch = W * sample + pitch_extra
    return (L().TuFramePlanes * B)(*[L().TuFramePlanes(FAKE + b * (1 << 16), FAKE + b * (1 << 16) + 8192, pitch, pitch)
                                     for b in range(B)])


def codes():
    _l = L()
    return {"NV12": (_l.TU_U8 | _l.TU_LAYOUT_NV12, 1, 2), "P010": (_l.TU_U16 | _l.TU_LAYOUT_P010, 2, 4)}


def both_ops(lib, fr, code, B, H, W, rgb=FAKE):
    return [(lib.tu_yuv420_planes_to_rgb(fr, code, rgb, B, H, W, None), L().last_error()),
            (lib.tu_rgb_to_yuv420_planes(rgb, fr, code, B, H, W, None), L().last_error())]


def expect(results, *words):
    for rc, msg in results:
        assert rc == L().TU_ERR_ARG, msg
        for w in words:
            assert w in msg, (w, msg)


@pytest.mark.parametrize("fmt", ["NV12", "P010"])
def test_descriptor_rejections(lib, fmt):
    code, sb, al = codes()[fmt]
    B, H, W = 3, 8, 10
    # a NULL plane, frame 1
    for field in ("y", "uv"):
        fr = frames(B, W, sb)
        setattr(fr[1], field, None)
        expect(both_ops(lib, fr, code, B, H, W), "frame 1", f"{field} is NULL")
    # a pitch smaller than W samples, frame 2
    for field in ("y_pitch", "uv_pitch"):
        fr = frames(B, W, sb)
        setattr(fr[2], field, W * sb - al)
        expect(both_ops(lib, fr, code, B, H, W), "frame 2", field, "smaller than W samples")
        setattr(fr[2], field, -W * sb)                                   # bottom-up (negative) pitches are not surfaces here
        expect(both_ops(lib, fr, code, B, H, W), "frame 2", field)
    # alignment the pair accesses need: 2 bytes (NV12), 4 bytes (P010), of every plane pointer and pitch
    for field in ("y", "uv", "y_pitch", "uv_pitch"):
        for off in range(1, al):
            fr = frames(B, W, sb)
            setattr(fr[0], field, getattr(fr[0], field) + off)
            expect(both_ops(lib, fr, code, B, H, W), "frame 0", field, "multiple of %d bytes" % al)
    # a pitch of exactly W samples is a dense row and is fine: only the later frames' fault is reported
    fr = frames(B, W, sb, pitch_extra=0)
    fr[2].y = None
    expect(both_ops(lib, fr, code, B, H, W), "frame 2")
    # odd sizes, no array, a bad B, a NULL or misaligned RGB buffer
    fr = frames(B, W, sb)
    expect(both_ops(lib, fr, code, B, H + 1, W), "even")
    expect(both_ops(lib, fr, code, B, H, W + 1), "even")
    expect(both_ops(lib, None, code, B, H, W), "bad argument")
    expect(both_ops(lib, fr, code, 0, H, W), "bad argument")
    expect(both_ops(lib, fr, code, B, H, W, rgb=None), "RGB buffer")
    expect(both_ops(lib, fr, code, B, H, W, rgb=FAKE + 2), "RGB buffer")


def test_codes_that_are_not_4_2_0(lib):
    _l = L()
    fr = frames(2, 8, 2)
    for code in (_l.TU_U8, _l.TU_F16, _l.TU_F32, _l.TU_U16, _l.TU_U8 | _l.TU_LAYOUT_HWC, _l.TU_U8 | _l.TU_LAYOUT_P010,
                 _l.TU_U8 | _l.TU_LAYOUT_NV12 | _l.TU_YUV_BT2020,
                 _l.TU_U16 | _l.TU_LAYOUT_P010 | _l.TU_YUV_BT2020 | _l.TU_YUV_BT601):
        expect(both_ops(lib, fr, code, 2, 4, 8), "NV12", "P010")


def _weights():
    """packed WindowTransformer weights (host tensors: only the sizing pass reads the struct here)"""
    return _packed("WindowTransformer", torch.bfloat16)


def test_forward_planes_rejections_before_any_launch(lib):
    _l = L()
    pw = _weights()
    w = C.byref(pw.struct)
    nv12, p010 = _l.TU_U8 | _l.TU_LAYOUT_NV12, _l.TU_U16 | _l.TU_LAYOUT_P010
    B, H, W, oh, ow = 2, 72, 104, 108, 156
    xf, of = frames(B, W, 1), frames(B, ow, 2)

    def fwd(x, xfr, i, o, ofr, oc, Bn=B, ws=FAKE, nbytes=1 << 40):
        rc = lib.tu_forward_planes(w, x, xfr, i, o, ofr, oc, Bn, H, W, oh, ow, 0, _l.TU_BF16, 1, ws, nbytes, None)
        return rc, _l.last_error()

    expect([fwd(FAKE, xf, nv12, FAKE, None, _l.TU_F32)], "either x or x_frames")          # both given on a side
    expect([fwd(FAKE, None, nv12, FAKE, of, p010)], "either out or out_frames")
    expect([fwd(None, None, nv12, FAKE, None, _l.TU_F32)], "null buffer")                 # neither
    expect([fwd(FAKE, None, nv12, None, None, _l.TU_F32)], "null buffer")
    expect([fwd(None, xf, nv12, FAKE, None, _l.TU_F32, ws=None)], "null buffer")
    # a frames array on a side that is not NV12 / P010
    for i in (_l.TU_U8, _l.TU_F16, _l.TU_U8 | _l.TU_LAYOUT_HWC_BGR):
        expect([fwd(None, xf, i, FAKE, None, _l.TU_F32)], "x_frames", "NV12 / P010 input only")
    for o in (_l.TU_U8, _l.TU_F32, _l.TU_U8 | _l.TU_LAYOUT_HWC):
        expect([fwd(FAKE, None, nv12, None, of, o)], "out_frames", "NV12 / P010 output only")
    # bad descriptors: the frame index and field, on the side they belong to; output pitches are checked against outW
    bad = frames(B, W, 1)
    bad[1].uv_pitch = W - 2
    expect([fwd(None, bad, nv12, FAKE, None, _l.TU_F32)], "x_frames", "frame 1", "uv_pitch")
    short = frames(B, ow, 2, pitch_extra=0)
    short[1].y_pitch = 2 * ow - 4
    expect([fwd(None, xf, nv12, None, short, p010)], "out_frames", "frame 1", "y_pitch")
    odd = frames(B, ow, 2)
    odd[0].uv += 2
    expect([fwd(None, xf, nv12, None, odd, p010)], "out_frames", "frame 0", "uv", "multiple of 4 bytes")
    # the existing code rules hold for surfaces too
    expect([fwd(None, xf, nv12 | _l.TU_YUV_BT2020, FAKE, None, _l.TU_F32)], "TU_YUV_BT2020")
    expect([fwd(None, xf, _l.TU_U16, FAKE, None, _l.TU_F32)], "TU_U16")
    rc, msg = lib.tu_forward_planes(w, None, xf, nv12, FAKE, None, _l.TU_F32, B, H + 1, W, oh, ow, 0, _l.TU_BF16, 1, FAKE, 1 << 40,
                                    None), _l.last_error()
    expect([(rc, msg)], "even")
    rc, msg = lib.tu_forward_planes(w, FAKE, None, _l.TU_F32, None, of, p010, B, H, W, oh + 1, ow, 0, _l.TU_BF16, 1, FAKE, 1 << 40,
                                    None), _l.last_error()
    expect([(rc, msg)], "even")


def test_workspace_of_a_surfaces_call_is_the_io_query(lib):
    """surfaces do not change the arena: a surfaces call needs exactly tu_forward_workspace_bytes_io of its codes (one byte less is
    TU_ERR_WORKSPACE, reported by the sizing pass before any launch)"""
    _l = L()
    pw = _weights()
    w = C.byref(pw.struct)
    nv12, p010 = _l.TU_U8 | _l.TU_LAYOUT_NV12, _l.TU_U16 | _l.TU_LAYOUT_P010
    B, H, W, oh, ow = 2, 72, 104, 108, 156
    for i, o in ((nv12, nv12), (p010, p010), (nv12, p010), (nv12, _l.TU_U8 | _l.TU_LAYOUT_HWC_BGR), (_l.TU_U8, p010)):
        need = lib.tu_forward_workspace_bytes_io(w, B, H, W, oh, ow, 0, _l.TU_BF16, i, o)
        assert need > 0
        xf = frames(B, W, 2 if i == p010 else 1) if i in (nv12, p010) else None
        of = frames(B, ow, 2 if o == p010 else 1) if o in (nv12, p010) else None
        for planes_in, planes_out in ((True, True), (True, False), (False, True)):
            a = xf if planes_in and xf is not None else None
            b = of if planes_out and of is not None else None
            rc = lib.tu_forward_planes(w, None if a else FAKE, a, i, None if b else FAKE, b, o, B, H, W, oh, ow, 0, _l.TU_BF16, 1,
                                       FAKE, need - 1, None)
            assert rc == _l.TU_ERR_WORKSPACE and ("need %d bytes" % need) in _l.last_error(), (i, o, planes_in, planes_out)


# ---------------------------------------------------------------------------------------------------------------------------------
# Python
def test_plane_pairs_rejections():
    from transformerupscaler_b200 import engine
    y, uv = torch.zeros(8, 16, dtype=torch.uint8), torch.zeros(4, 16, dtype=torch.uint8)
    bad = [
        [],                                                               # empty
        (y, uv),                                                          # a pair, not a list of pairs
        [(y,)],                                                           # not a pair
        [(y, uv.numpy())],                                                # not tensors
        [(y.to(torch.uint16), uv.to(torch.uint16))],                      # P010 planes for NV12
        [(y[None], uv)],                                                  # 3-D
        [(torch.zeros(8, 32, dtype=torch.uint8)[:, ::2], uv)],            # non-unit stride along W
        [(y, torch.zeros(5, 16, dtype=torch.uint8))],                     # uv is not (H/2, W)
        [(torch.zeros(7, 16, dtype=torch.uint8), torch.zeros(3, 16, dtype=torch.uint8))],   # odd H
        [(torch.zeros(8, 15, dtype=torch.uint8), torch.zeros(4, 15, dtype=torch.uint8))],   # odd W
        [(y, uv)],                                                        # host tensors
    ]
    for fr in bad:
        with pytest.raises(ValueError):
            engine.plane_pairs(fr, "NV12", "frames")
    with pytest.raises(ValueError):
        engine.plane_pairs([(y, uv)], "P010", "frames")


def test_model_and_wrappers_reject_misplaced_planes():
    from transformerupscaler_b200 import engine
    from transformerupscaler_b200.graph import GraphedModel
    from transformerupscaler_b200.models.WindowTransformer.model import TransformerModel
    from transformerupscaler_b200.pipeline import FramePipeline
    m = TransformerModel().eval()
    y, uv = torch.zeros(8, 16, dtype=torch.uint8), torch.zeros(4, 16, dtype=torch.uint8)
    with pytest.raises(ValueError, match="in_layout"):                    # planes need in_layout 'nv12' / 'p010'
        m([(y, uv)], res_out=(12, 24))
    with pytest.raises(ValueError, match="in_layout"):
        m([(y, uv)], in_layout="hwc", res_out=(12, 24))
    x = torch.zeros(1, 12, 16, dtype=torch.uint8)
    for ol in ("chw", "hwc_bgr"):                                         # out= needs out_layout 'nv12' / 'p010'
        with pytest.raises(ValueError, match="out_layout"):
            engine.run_forward(0, "WindowTransformer", x, (12, 24), None, True, True, torch.uint8, in_layout="nv12", out_layout=ol,
                               out=[(y, uv)])
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(m)([(y, uv)], in_layout="nv12")
    with pytest.raises(TypeError, match="frame planes"):
        GraphedModel(m)(x, in_layout="nv12", out_layout="nv12", out=[(y, uv)])
    with pytest.raises(TypeError, match="out="):
        FramePipeline(m, device=torch.device("cpu"), in_layout="nv12", out_layout="nv12", out=[(y, uv)])
