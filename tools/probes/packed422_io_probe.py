#!/usr/bin/env python
"""Packed 4:2:2 frames (yuyv422, uyvy422, y210) at both ends of the forward (profiles/packed422_io_probe.log).

  python tools/probes/packed422_io_probe.py [rounds]

1. The conversion kernels on dense batches, with their semi-planar siblings (nv16, p210: the same samples in two planes) in the same
   run.  Alternating rounds, CUDA events over 400 launches a round, inputs rotating over four buffer sets so the working set (236 MB and
   more) does not stay in the 126 MB L2.  To RGB at 8 x 720p, from RGB at 8 x 1080p.  Bytes are the frame bytes read plus written, from
   the shapes; the lower bound is bytes / 7.7 TB/s.
2. Device-resident whole forwards of bf16 modules in alternating rounds of 10 forwards, medians: WindowTransformer 8 x 720p -> 1080p
   yuyv422 -> yuyv422 against nv16 -> nv16 and uint8 CHW -> CHW, and ResidualTransformer 2 x 720p -> 4K y210 -> y210 against p210 -> p210.
3. End to end through FramePipeline (pinned host frames in and out, depth 4, two compute streams): WindowTransformer 8 x 720p -> 1080p,
   pinned yuyv422 (B, H, W, 2) against pinned uint8 HWC (B, H, W, 3), alternating, median of 3.
4. The card's name, power limit and SM clock, read in the same run (first and last line).
"""
import importlib
import os
import statistics
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from transformerupscaler_b200 import _lib  # noqa: E402
from transformerupscaler_b200.synth import synth_state_dict, synth_frames  # noqa: E402

PEAK = 7.7e12
# name -> (code, 16-bit, packed)
FMTS = {"yuyv422": (_lib.TU_U8 | _lib.TU_LAYOUT_YUYV, False, True), "uyvy422": (_lib.TU_U8 | _lib.TU_LAYOUT_UYVY, False, True),
        "nv16": (_lib.TU_U8 | _lib.TU_LAYOUT_NV16, False, False),
        "y210": (_lib.TU_U16 | _lib.TU_LAYOUT_YUYV, True, True), "p210": (_lib.TU_U16 | _lib.TU_LAYOUT_NV16, True, False)}


def shape(fmt, B, H, W):
    return (B, H, W, 2) if FMTS[fmt][2] else (B, 2 * H, W)


def convert(lib, fmt, to_rgb, yuv, rgb, B, H, W, st):
    """one conversion call on dense buffers"""
    code, _, packed = FMTS[fmt]
    if packed:
        return (lib.tu_packed422_to_rgb(yuv, None, code, rgb, B, H, W, st) if to_rgb
                else lib.tu_rgb_to_packed422(rgb, yuv, None, code, B, H, W, st))
    return (lib.tu_yuv422sp_to_rgb(yuv, None, code, rgb, B, H, W, st) if to_rgb
            else lib.tu_rgb_to_yuv422sp(rgb, yuv, None, code, B, H, W, st))


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
        for fmt, (code, w16, _) in FMTS.items():
            if w16:
                yv = [torch.randint(0, 65536, shape(fmt, B, H, W), dtype=torch.int32, device=dev).to(torch.int16).view(torch.uint16)
                      for _ in range(4)]
            else:
                yv = [torch.randint(0, 256, shape(fmt, B, H, W), dtype=torch.uint8, device=dev) for _ in range(4)]
            rgb = [torch.rand(B, 3, H, W, device=dev).to(torch.float32 if w16 else torch.float16) for _ in range(4)]
            nbytes[fmt] = 2 * n * (2 if w16 else 1) + 3 * n * (4 if w16 else 2)
            fn = (lambda i, yv=yv, rgb=rgb, fmt=fmt: convert(lib, fmt, to_rgb, yv[i % 4].data_ptr(), rgb[i % 4].data_ptr(), B, H, W, st))
            _lib.check(fn(0))
            fns[f"{fmt}_to_rgb" if to_rgb else f"rgb_to_{fmt}"] = fn
        ts = alternate(fns, rounds, 400)
        meds = {fmt: statistics.median(v) for (name, v), fmt in zip(ts.items(), FMTS)}
        for (name, v), fmt in zip(ts.items(), FMTS):
            ms, nb = meds[fmt], nbytes[fmt]
            sib = "p210" if FMTS[fmt][1] else "nv16"
            rel = f"; / {sib} {ms / meds[sib]:.3f}" if FMTS[fmt][2] else ""
            print(f"   {name:16s} {B} x {H}x{W}: {ms * 1e3:7.2f} us  ({nb / 1e6:.1f} MB, lower bound {nb / PEAK * 1e6:.1f} us: "
                  f"{nb / (ms * 1e-3) / 1e12:.2f} TB/s, {nb / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s{rel}; rounds "
                  f"{min(v) * 1e3:.2f}..{max(v) * 1e3:.2f} us)", flush=True)
        del fns
        torch.cuda.empty_cache()


def model(name, dev):
    m = importlib.import_module(f"transformerupscaler_b200.models.{name}.model").TransformerModel().eval()
    m.load_state_dict(synth_state_dict(name, 0), strict=True)
    return m.to(dev).bfloat16()


def frames(fmt, B, H, W, rgb, dev):
    lib, st = _lib.load(), torch.cuda.current_stream().cuda_stream
    x = torch.empty(shape(fmt, B, H, W), dtype=torch.uint16 if FMTS[fmt][1] else torch.uint8, device=dev)
    _lib.check(convert(lib, fmt, False, x.data_ptr(), rgb.to(torch.float32 if FMTS[fmt][1] else torch.float16).data_ptr(), B, H, W, st))
    return x


def forwards(dev, rounds):
    print(f"# 2. device-resident forwards, bf16 modules; alternating rounds of 10 forwards ({rounds} rounds), medians", flush=True)
    for name, B, kw, fmts in (("WindowTransformer", 8, dict(res_out=(1080, 1920)), ("yuyv422", "nv16")),
                              ("ResidualTransformer", 2, dict(res_out=(2160, 3840)), ("y210", "p210"))):
        m = model(name, dev)
        rgb = synth_frames(B, 720, 1280, seed=1).to(dev)
        xs = {"chw": (rgb * 255).to(torch.uint8)}
        for fmt in fmts:
            xs[fmt] = frames(fmt, B, 720, 1280, rgb, dev)
        arms = {f"{k} -> {k}": (lambda i, k=k: m(xs[k], in_layout=k, out_layout=k, **kw)) for k in xs}
        with torch.no_grad():
            ts = alternate(arms, rounds, 10)
        base = statistics.median(ts["chw -> chw"])
        print(f"{name} {B} x 720p -> {kw['res_out'][0]}p", flush=True)
        for k, v in ts.items():
            med = statistics.median(v)
            print(f"   {k:20s} {med:7.3f} ms  / CHW {med / base:6.4f}  (rounds {min(v):.3f}..{max(v):.3f})", flush=True)
        del m, xs, arms
        torch.cuda.empty_cache()


def e2e_rate(dev, m, packed, steps=60, B=8):
    """frames/s of FramePipeline over `steps` batches of B frames, pinned host buffers both sides"""
    from transformerupscaler_b200.pipeline import FramePipeline
    if packed:
        hin = [frames("yuyv422", B, 720, 1280, synth_frames(B, 720, 1280, seed=i).to(dev), dev).cpu().pin_memory() for i in range(4)]
        hout = [torch.empty((B, 1080, 1920, 2), dtype=torch.uint8).pin_memory() for _ in range(4)]
        kw = dict(in_layout="yuyv422", out_layout="yuyv422")
    else:
        hin = [(synth_frames(B, 720, 1280, seed=i) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous().pin_memory()
               for i in range(4)]
        hout = [torch.empty((B, 1080, 1920, 3), dtype=torch.uint8).pin_memory() for _ in range(4)]
        kw = dict(in_layout="hwc", out_layout="hwc")
    pipe = FramePipeline(m, depth=4, device=dev, compute_streams=2, res_out=(1080, 1920), **kw)
    for i in range(8):
        pipe.submit(hin[i % 4], hout[i % 4])
    pipe.drain()
    t0 = time.perf_counter()
    for i in range(steps):
        pipe.submit(hin[i % 4], hout[i % 4])
    pipe.drain()
    return steps * B / (time.perf_counter() - t0)


def pipeline(dev):
    print("# 3. end to end, FramePipeline, WindowTransformer 8 x 720p -> 1080p, pinned host frames both sides, depth 4, 2 compute "
          "streams, 60 batches after 8 warm-up batches, alternating, median of 3", flush=True)
    m = model("WindowTransformer", dev)
    rates = {True: [], False: []}
    for r in range(3):
        for packed in ((True, False) if r % 2 == 0 else (False, True)):
            rates[packed].append(e2e_rate(dev, m, packed))
    for packed, label in ((True, "pinned yuyv422 -> yuyv422"), (False, "pinned uint8 HWC -> HWC")):
        v = rates[packed]
        mb = (2 if packed else 3) * (720 * 1280 + 1080 * 1920) / 1e6
        print(f"   {label:26s} {statistics.median(v):7.1f} frames/s  (host bytes a frame {mb:.1f} MB; rounds "
              f"{min(v):.1f}..{max(v):.1f})", flush=True)


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
    pipeline(dev)
    print(f"# after the run: {card()}", flush=True)


if __name__ == "__main__":
    main()
