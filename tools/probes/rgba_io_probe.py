#!/usr/bin/env python
"""Cost of RGBA / BGRA frame I/O (profiles/rgba_io_probe.log).

  python tools/probes/rgba_io_probe.py [rounds]

1. tu_frames_to_planar, 4-byte (BGRA) against 3-byte (HWC BGR) frames at 8 x 720p: CUDA events over many launches, alternating A / B
   rounds, medians; inputs rotate over four buffer sets (4 x 51.6 / 4 x 44.2 MB with the planar outputs, more than the 126 MB L2).
   Bytes from the shapes: 4 (3) read + 3 written a pixel.
2. tu_resample_alpha at 8 x 720p -> 1080p and 2 x 720p -> 4K, inputs rotating over four buffer sets, with its bytes and share of
   7.7 TB/s.  Bytes: the whole 4-byte input (the alpha byte of every pixel lies in every 32-byte sector) + 1 byte an output pixel.
3. Device-resident bf16 forwards, alternating rounds of 20, medians, inputs rotating over four sets: BGRA -> BGRA (A) against
   HWC BGR -> HWC BGR (B) against uint8 CHW -> CHW (C): WindowTransformer 8 x 720p -> 1080p, ResidualTransformer 2 x 720p -> 4K,
   FastTransformer 4 x 720p x2; and NV12 -> BGRA (A) against NV12 -> HWC BGR (B) against NV12 -> NV12 (C) for WindowTransformer.
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
NSETS = 4


def model(name, dev):
    import importlib
    m = importlib.import_module(f"transformerupscaler_b200.models.{name}.model").TransformerModel().eval()
    m.load_state_dict(synth_state_dict(name, 0), strict=True)
    return m.to(dev).bfloat16()


def bgra_frames(B, H, W, seed, dev):
    """smooth synthetic RGB content with a smooth alpha ramp, (B, H, W, 4) uint8 B G R A"""
    x = torch.empty(B, H, W, 4, dtype=torch.uint8)
    x[..., :3] = (synth_frames(B, H, W, seed=seed) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).flip(-1)
    x[..., 3] = (torch.arange(W) * 255 // max(W - 1, 1)).to(torch.uint8)
    return x.to(dev)


def nv12_frames(B, H, W, seed, dev):
    lib = _lib.load()
    rgb = synth_frames(B, H, W, seed=seed).half().to(dev)
    out = torch.empty(B, 3 * H // 2, W, dtype=torch.uint8, device=dev)
    _lib.check(lib.tu_rgb_to_nv12(rgb.data_ptr(), out.data_ptr(), _lib.TU_U8 | _lib.TU_LAYOUT_NV12, B, H, W,
                                  torch.cuda.current_stream().cuda_stream))
    return out


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def abn(tag, fns, rounds, iters):
    """alternating rounds over the variants (order rotated every round); returns the medians in ms"""
    for f in fns:
        f(0)
        f(1)
    torch.cuda.synchronize()
    ts = [[] for _ in fns]
    for r in range(rounds):
        order = list(range(len(fns)))
        order = order[r % len(fns):] + order[:r % len(fns)]
        for k in order:
            ts[k].append(timed(fns[k], iters))
    med = [statistics.median(t) for t in ts]
    names = "ABC"
    parts = "  ".join(f"{names[k]} {med[k]:8.4f} ms" for k in range(len(fns)))
    last = names[len(fns) - 1]
    ratios = "  ".join(f"{names[k]}/{last} {med[k] / med[-1]:6.4f}" for k in range(len(fns) - 1))
    spread = "; ".join(f"{names[k]} {min(t):.4f}..{max(t):.4f}" for k, t in enumerate(ts))
    print(f"{tag:44s} {parts}  {ratios}  ({spread})", flush=True)
    return med


def kernels(dev, rounds):
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    B, H, W = 8, 720, 1280
    n = B * H * W
    print(f"# 1. tu_frames_to_planar {B} x {H}x{W}: A = BGRA (4 bytes a pixel), B = HWC BGR (3 bytes); CUDA events, {rounds} alternating "
          f"rounds of 200 launches, {NSETS} rotating buffer sets, medians", flush=True)
    x4 = [torch.randint(0, 256, (B, H, W, 4), dtype=torch.uint8, device=dev) for _ in range(NSETS)]
    x3 = [t[..., :3].contiguous() for t in x4]
    pl = [torch.empty(B, 3, H, W, dtype=torch.uint8, device=dev) for _ in range(NSETS)]

    def f4(i):
        lib.tu_frames_to_planar(x4[i % NSETS].data_ptr(), _lib.TU_LAYOUT_BGRA, pl[i % NSETS].data_ptr(), B, H, W, st)

    def f3(i):
        lib.tu_frames_to_planar(x3[i % NSETS].data_ptr(), _lib.TU_LAYOUT_HWC_BGR, pl[i % NSETS].data_ptr(), B, H, W, st)
    ma, mb = abn("   frames_to_planar", [f4, f3], rounds, 200)
    for tag, ms, nb in (("BGRA", ma, n * 7), ("HWC BGR", mb, n * 6)):
        print(f"   {tag:8s} {ms * 1e3:7.2f} us  {nb / 1e6:6.1f} MB  {nb / (ms * 1e-3) / 1e12:.2f} TB/s  "
              f"{nb / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s", flush=True)
    del x4, x3, pl
    torch.cuda.empty_cache()

    print(f"# 2. tu_resample_alpha: CUDA events, {rounds} rounds of 200 launches, {NSETS} rotating buffer sets, medians", flush=True)
    for B, oh, ow in ((8, 1080, 1920), (2, 2160, 3840)):
        xs = [torch.randint(0, 256, (B, H, W, 4), dtype=torch.uint8, device=dev) for _ in range(NSETS)]
        outs = [torch.empty(B, oh, ow, dtype=torch.uint8, device=dev) for _ in range(NSETS)]

        def fa(i):
            lib.tu_resample_alpha(xs[i % NSETS].data_ptr(), _lib.TU_U8 | _lib.TU_LAYOUT_BGRA, outs[i % NSETS].data_ptr(), B, H, W, oh, ow, st)
        fa(0)
        ts = [timed(fa, 200) for _ in range(rounds)]
        ms = statistics.median(ts)
        nb = B * H * W * 4 + B * oh * ow
        print(f"   {B} x 720p -> {oh}x{ow}: {ms * 1e3:7.2f} us  ({nb / 1e6:.1f} MB: {nb / (ms * 1e-3) / 1e12:.2f} TB/s, "
              f"{nb / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s; runs {min(ts) * 1e3:.2f}..{max(ts) * 1e3:.2f} us)", flush=True)
        del xs, outs
        torch.cuda.empty_cache()


def forwards(dev, rounds):
    print(f"# 3. device-resident forward, bf16 module, {rounds} alternating rounds of 20, {NSETS} rotating input sets, medians", flush=True)
    print("#    A = BGRA -> BGRA (alpha resampled), B = HWC BGR -> HWC BGR, C = uint8 CHW -> CHW", flush=True)
    for name, B, kw in (("WindowTransformer", 8, dict(res_out=(1080, 1920))), ("ResidualTransformer", 2, dict(res_out=(2160, 3840))),
                        ("FastTransformer", 4, dict(upscale_factor=2))):
        m = model(name, dev)
        x4 = [bgra_frames(B, 720, 1280, 10 + s, dev) for s in range(NSETS)]
        x3 = [t[..., :3].contiguous() for t in x4]
        xc = [t.permute(0, 3, 1, 2).flip(1).contiguous() for t in x3]
        with torch.no_grad():
            abn(f"{name} {B} x 720p {kw}", [lambda i: m(x4[i % NSETS], in_layout="bgra", out_layout="bgra", **kw),
                                             lambda i: m(x3[i % NSETS], in_layout="hwc_bgr", out_layout="hwc_bgr", **kw),
                                             lambda i: m(xc[i % NSETS], **kw)], rounds, 20)
        del m, x4, x3, xc
        torch.cuda.empty_cache()
    print("#    A = NV12 -> BGRA, B = NV12 -> HWC BGR, C = NV12 -> NV12", flush=True)
    m = model("WindowTransformer", dev)
    xn = [nv12_frames(8, 720, 1280, 20 + s, dev) for s in range(NSETS)]
    kw = dict(res_out=(1080, 1920))
    with torch.no_grad():
        abn(f"WindowTransformer 8 x 720p {kw}", [lambda i: m(xn[i % NSETS], in_layout="nv12", out_layout="bgra", **kw),
                                                 lambda i: m(xn[i % NSETS], in_layout="nv12", out_layout="hwc_bgr", **kw),
                                                 lambda i: m(xn[i % NSETS], in_layout="nv12", out_layout="nv12", **kw)], rounds, 20)


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print(f"# {q}; {torch.cuda.device_count()} GPU(s); torch {torch.__version__}", flush=True)
    kernels(dev, rounds)
    forwards(dev, rounds)


if __name__ == "__main__":
    main()
