#!/usr/bin/env python
"""4:2:2 frames (yuv422p, nv16, p210, yuv422p10le) and LSB-aligned 10-bit planar frames (yuv420p10le, yuv444p10le) at both ends of the
forward (profiles/yuv422_io_probe.log).

  python tools/probes/yuv422_io_probe.py [rounds]

1. The conversion kernels on dense batches, with their siblings in the same run: NV12, P010 (the MSB sibling of yuv420p10le) and
   yuv444p16 (that of yuv444p10le).  Alternating rounds, CUDA events over 400 launches a round, inputs rotating over four buffer sets so
   the working set (236 MB and more) does not stay in the 126 MB L2.  To RGB at 8 x 720p, from RGB at 8 x 1080p.  Bytes are the frame
   bytes read plus written, from the shapes; the lower bound is bytes / 7.7 TB/s.
2. Device-resident whole forwards of bf16 modules in alternating rounds of 10 forwards, medians: WindowTransformer 8 x 720p -> 1080p and
   ResidualTransformer 2 x 720p -> 4K, yuv422p10le -> yuv422p10le and yuv420p10le -> yuv420p10le against P010 -> P010 and uint8 CHW -> CHW.
3. The card's name, power limit and SM clock, read in the same run (first and last line).
"""
import importlib
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from transformerupscaler_b200 import _lib  # noqa: E402
from transformerupscaler_b200.synth import synth_state_dict, synth_frames  # noqa: E402

PEAK = 7.7e12
LSB = _lib.TU_YUV_LSB10
# name -> (code, chroma subsampling, 16-bit, entry points: "yuvp" planar, "sp" semi-planar 4:2:2, or the 4:2:0 op's name)
FMTS = {"yuv422p": (_lib.TU_U8 | _lib.TU_LAYOUT_YUV422P, "422", False, "yuvp"),
        "nv16": (_lib.TU_U8 | _lib.TU_LAYOUT_NV16, "422", False, "sp"),
        "yuv422p10le": (_lib.TU_U16 | _lib.TU_LAYOUT_YUV422P | LSB, "422", True, "yuvp"),
        "p210": (_lib.TU_U16 | _lib.TU_LAYOUT_NV16, "422", True, "sp"),
        "yuv420p10le": (_lib.TU_U16 | _lib.TU_LAYOUT_YUV420P | LSB, "420", True, "yuvp"),
        "p010": (_lib.TU_U16 | _lib.TU_LAYOUT_P010, "420", True, "p010"),
        "nv12": (_lib.TU_U8 | _lib.TU_LAYOUT_NV12, "420", False, "nv12"),
        "yuv444p10le": (_lib.TU_U16 | _lib.TU_LAYOUT_YUV444P | LSB, "444", True, "yuvp"),
        "yuv444p16": (_lib.TU_U16 | _lib.TU_LAYOUT_YUV444P, "444", True, "yuvp")}
ROWS = {"420": 1.5, "422": 2, "444": 3}


def shape(fmt, B, H, W):
    sub = FMTS[fmt][1]
    return (B, 3, H, W) if sub == "444" else (B, int(ROWS[sub] * H), W)


def convert(lib, fmt, to_rgb, yuv, rgb, B, H, W, st):
    """one conversion call on dense buffers"""
    code, _, _, kind = FMTS[fmt]
    if kind == "yuvp":
        return (lib.tu_yuvp_to_rgb(yuv, None, code, rgb, B, H, W, st) if to_rgb else lib.tu_rgb_to_yuvp(rgb, yuv, None, code, B, H, W, st))
    if kind == "sp":
        return (lib.tu_yuv422sp_to_rgb(yuv, None, code, rgb, B, H, W, st) if to_rgb
                else lib.tu_rgb_to_yuv422sp(rgb, yuv, None, code, B, H, W, st))
    return (getattr(lib, f"tu_{kind}_to_rgb")(yuv, code, rgb, B, H, W, st) if to_rgb
            else getattr(lib, f"tu_rgb_to_{kind}")(rgb, yuv, code, B, H, W, st))


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def alternate(fns, rounds, iters):
    """alternating rounds over the functions (the order rotates each round); {name: [ms per call of each round]}"""
    for f in fns.values():
        f(0)
        f(0)
    torch.cuda.synchronize()
    names = list(fns)
    ts = {k: [] for k in names}
    for r in range(rounds):
        for k in names[r % len(names):] + names[:r % len(names)]:
            ts[k].append(timed(fns[k], iters))
    return ts


def kernels(dev, rounds):
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    print(f"# 1. conversion kernels, dense batches: alternating rounds of 400 launches ({rounds} rounds), four rotating buffer sets; "
          "medians, bandwidth over 7.7 TB/s", flush=True)
    for to_rgb, (B, H, W) in ((True, (8, 720, 1280)), (False, (8, 1080, 1920))):
        n = B * H * W
        fns, nbytes = {}, {}
        for fmt, (code, sub, w16, _) in FMTS.items():
            if w16:
                yv = [torch.randint(0, 1024, shape(fmt, B, H, W), dtype=torch.int16, device=dev).view(torch.uint16) for _ in range(4)]
            else:
                yv = [torch.randint(0, 256, shape(fmt, B, H, W), dtype=torch.uint8, device=dev) for _ in range(4)]
            rgb = [torch.rand(B, 3, H, W, device=dev).to(torch.float32 if w16 else torch.float16) for _ in range(4)]
            nbytes[fmt] = ROWS[sub] * n * (2 if w16 else 1) + 3 * n * (4 if w16 else 2)
            fn = (lambda i, yv=yv, rgb=rgb, fmt=fmt: convert(lib, fmt, to_rgb, yv[i % 4].data_ptr(), rgb[i % 4].data_ptr(), B, H, W, st))
            _lib.check(fn(0))
            fns[f"{fmt}_to_rgb" if to_rgb else f"rgb_to_{fmt}"] = fn
        ts = alternate(fns, rounds, 400)
        for (name, v), fmt in zip(ts.items(), FMTS):
            ms = statistics.median(v)
            nb = nbytes[fmt]
            print(f"   {name:19s} {B} x {H}x{W}: {ms * 1e3:7.2f} us  ({nb / 1e6:.1f} MB, lower bound {nb / PEAK * 1e6:.1f} us: "
                  f"{nb / (ms * 1e-3) / 1e12:.2f} TB/s, {nb / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s; rounds {min(v) * 1e3:.2f}.."
                  f"{max(v) * 1e3:.2f} us)", flush=True)
        del fns
        torch.cuda.empty_cache()


def forwards(dev, rounds):
    print(f"# 2. device-resident forwards, bf16 modules; alternating rounds of 10 forwards ({rounds} rounds), medians", flush=True)
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    for model, B, kw in (("WindowTransformer", 8, dict(res_out=(1080, 1920))), ("ResidualTransformer", 2, dict(res_out=(2160, 3840)))):
        m = importlib.import_module(f"transformerupscaler_b200.models.{model}.model").TransformerModel().eval()
        m.load_state_dict(synth_state_dict(model, 0), strict=True)
        m = m.to(dev).bfloat16()
        rgb = synth_frames(B, 720, 1280, seed=1).to(dev)
        xs = {"chw": (rgb * 255).to(torch.uint8)}
        for fmt in ("yuv422p10le", "yuv420p10le", "p010"):
            xs[fmt] = torch.empty(shape(fmt, B, 720, 1280), dtype=torch.uint16, device=dev)
            _lib.check(convert(lib, fmt, False, xs[fmt].data_ptr(), rgb.data_ptr(), B, 720, 1280, st))
        arms = {f"{k} -> {k}": (lambda i, k=k: m(xs[k], in_layout=k, out_layout=k, **kw)) for k in xs}
        with torch.no_grad():
            ts = alternate(arms, rounds, 10)
        base = statistics.median(ts["chw -> chw"])
        print(f"{model} {B} x 720p -> {kw['res_out'][0]}p", flush=True)
        for k, v in ts.items():
            med = statistics.median(v)
            print(f"   {k:28s} {med:7.3f} ms  / CHW {med / base:6.4f}  (rounds {min(v):.3f}..{max(v):.3f})", flush=True)
        del m, xs, arms
        torch.cuda.empty_cache()


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 12
    dev = torch.device("cuda:0")
    print(f"# {card()} (name, power limit, SM clock now, max SM clock); {torch.cuda.device_count()} GPU(s); torch {torch.__version__}",
          flush=True)
    kernels(dev, rounds)
    forwards(dev, rounds)
    print(f"# after the run: {card()}", flush=True)


if __name__ == "__main__":
    main()
