#!/usr/bin/env python
"""Planar YUV frames (yuv420p, yuv444p, yuv444p16) at both ends of the forward (profiles/yuvp_io_probe.log).

  python tools/probes/yuvp_io_probe.py [rounds]

1. The conversion kernels of tu_yuvp_to_rgb / tu_rgb_to_yuvp on dense batches, with the NV12 kernels in the same run as the control:
   alternating rounds, CUDA events over 400 launches a round, inputs rotating over four buffer sets so the working set (265 MB and
   more) does not stay in the 126 MB L2.  To RGB at 8 x 720p, from RGB at 8 x 1080p.  Bytes are the frame bytes read plus written,
   from the shapes; the lower bound is bytes / 7.7 TB/s.
2. Device-resident whole forwards of the bf16 WindowTransformer, 8 x 720p -> 1080p, in alternating rounds of 20 forwards, medians:
   yuv420p -> yuv420p and yuv444p -> yuv444p against NV12 -> NV12 and uint8 CHW -> CHW.
3. The card's name, power limit and SM clock, read in the same run (first and last line).
"""
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from transformerupscaler_b200 import _lib  # noqa: E402
from transformerupscaler_b200.synth import synth_state_dict, synth_frames  # noqa: E402

PEAK = 7.7e12
NV12 = _lib.TU_U8 | _lib.TU_LAYOUT_NV12
CODES = {"yuv420p": _lib.TU_U8 | _lib.TU_LAYOUT_YUV420P, "yuv444p": _lib.TU_U8 | _lib.TU_LAYOUT_YUV444P,
         "yuv444p16": _lib.TU_U16 | _lib.TU_LAYOUT_YUV444P, "nv12": NV12}


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
        for fmt, code in CODES.items():
            w16 = fmt == "yuv444p16"
            frame_el = (1.5 if fmt in ("nv12", "yuv420p") else 3) * n
            shape = (B, 3 * H // 2, W) if fmt in ("nv12", "yuv420p") else (B, 3, H, W)
            if w16:
                yv = [torch.randint(-32768, 32768, shape, dtype=torch.int16, device=dev).view(torch.uint16) for _ in range(4)]
            else:
                yv = [torch.randint(0, 256, shape, dtype=torch.uint8, device=dev) for _ in range(4)]
            rgb = [torch.rand(B, 3, H, W, device=dev).to(torch.float32 if w16 else torch.float16) for _ in range(4)]
            nbytes[fmt] = frame_el * (2 if w16 else 1) + 3 * n * (4 if w16 else 2)
            name = (f"{fmt}_to_rgb" if to_rgb else f"rgb_to_{fmt}")
            if fmt == "nv12":
                fn = ((lambda i, yv=yv, rgb=rgb: lib.tu_nv12_to_rgb(yv[i % 4].data_ptr(), NV12, rgb[i % 4].data_ptr(), B, H, W, st))
                      if to_rgb else
                      (lambda i, yv=yv, rgb=rgb: lib.tu_rgb_to_nv12(rgb[i % 4].data_ptr(), yv[i % 4].data_ptr(), NV12, B, H, W, st)))
            else:
                fn = ((lambda i, yv=yv, rgb=rgb, c=code: lib.tu_yuvp_to_rgb(yv[i % 4].data_ptr(), None, c, rgb[i % 4].data_ptr(), B, H, W, st))
                      if to_rgb else
                      (lambda i, yv=yv, rgb=rgb, c=code: lib.tu_rgb_to_yuvp(rgb[i % 4].data_ptr(), yv[i % 4].data_ptr(), None, c, B, H, W,
                                                                            st)))
            _lib.check(fn(0))
            fns[name] = fn
        ts = alternate(fns, rounds, 400)
        for (name, v), fmt in zip(ts.items(), CODES):
            ms = statistics.median(v)
            nb = nbytes[fmt]
            print(f"   {name:17s} {B} x {H}x{W}: {ms * 1e3:7.2f} us  ({nb / 1e6:.1f} MB, lower bound {nb / PEAK * 1e6:.1f} us: "
                  f"{nb / (ms * 1e-3) / 1e12:.2f} TB/s, {nb / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s; rounds {min(v) * 1e3:.2f}.."
                  f"{max(v) * 1e3:.2f} us)", flush=True)
        del fns
        torch.cuda.empty_cache()


def forwards(dev, rounds):
    import importlib
    print(f"# 2. device-resident forward, bf16 module; alternating rounds of 20 forwards ({rounds} rounds), medians", flush=True)
    m = importlib.import_module("transformerupscaler_b200.models.WindowTransformer.model").TransformerModel().eval()
    m.load_state_dict(synth_state_dict("WindowTransformer", 0), strict=True)
    m = m.to(dev).bfloat16()
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    B, kw = 8, dict(res_out=(1080, 1920))
    rgb = synth_frames(B, 720, 1280, seed=1).to(dev).half()
    xs = {"chw": (rgb.float() * 255).to(torch.uint8)}
    xs["nv12"] = torch.empty(B, 1080, 1280, dtype=torch.uint8, device=dev)
    _lib.check(lib.tu_rgb_to_nv12(rgb.data_ptr(), xs["nv12"].data_ptr(), NV12, B, 720, 1280, st))
    xs["yuv420p"] = torch.empty(B, 1080, 1280, dtype=torch.uint8, device=dev)
    _lib.check(lib.tu_rgb_to_yuvp(rgb.data_ptr(), xs["yuv420p"].data_ptr(), None, CODES["yuv420p"], B, 720, 1280, st))
    xs["yuv444p"] = torch.empty(B, 3, 720, 1280, dtype=torch.uint8, device=dev)
    _lib.check(lib.tu_rgb_to_yuvp(rgb.data_ptr(), xs["yuv444p"].data_ptr(), None, CODES["yuv444p"], B, 720, 1280, st))
    arms = {f"{k} -> {k}": (lambda i, k=k: m(xs[k], in_layout=k, out_layout=k, **kw)) for k in ("yuv420p", "yuv444p", "nv12", "chw")}
    with torch.no_grad():
        ts = alternate(arms, rounds, 20)
    base = statistics.median(ts["chw -> chw"])
    print(f"WindowTransformer {B} x 720p -> 1080p", flush=True)
    for k, v in ts.items():
        med = statistics.median(v)
        print(f"   {k:20s} {med:7.3f} ms  / CHW {med / base:6.4f}  (rounds {min(v):.3f}..{max(v):.3f})", flush=True)


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
