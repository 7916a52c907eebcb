#!/usr/bin/env python
"""Cost of P010 (10-bit) frame I/O (profiles/p010_io_probe.log).

  python tools/probes/p010_io_probe.py [rounds]

1. The conversion kernels alone (CUDA events over many launches; the inputs rotate over four buffer sets, 442 / 995 MB for P010, so
   the working set does not stay in the 126 MB L2): tu_p010_to_rgb at 8 x 720p, tu_rgb_to_p010 at 8 x 1080p, and the NV12 pair at the
   same sizes for comparison, with their bandwidth as a fraction of 7.7 TB/s.  Bytes from the shapes: P010 = 3 B read + 12 B written
   a pixel (8 x 720p: 22.1 + 88.5 MB), and the reverse (8 x 1080p: 199.1 + 49.8 MB); NV12 = 1.5 B + 6 B.
2. Device-resident whole forwards of the bf16 module, alternating rounds, medians: P010 -> P010 against NV12 -> NV12 and uint8 CHW ->
   CHW, for WindowTransformer 8 x 720p -> 1080p and ResidualTransformer 2 x 720p -> 4K.
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
P010 = _lib.TU_U16 | _lib.TU_LAYOUT_P010


def model(name, dev):
    import importlib
    m = importlib.import_module(f"transformerupscaler_b200.models.{name}.model").TransformerModel().eval()
    m.load_state_dict(synth_state_dict(name, 0), strict=True)
    return m.to(dev).bfloat16()


def frames(B, H, W, dev, p010):
    """smooth synthetic frames as NV12 / P010, converted on the device"""
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    rgb = synth_frames(B, H, W, seed=1).to(dev)
    if p010:
        out = torch.empty(B, 3 * H // 2, W, dtype=torch.uint16, device=dev)
        _lib.check(lib.tu_rgb_to_p010(rgb.data_ptr(), out.data_ptr(), P010, B, H, W, st))
    else:
        rgb = rgb.half()
        out = torch.empty(B, 3 * H // 2, W, dtype=torch.uint8, device=dev)
        _lib.check(lib.tu_rgb_to_nv12(rgb.data_ptr(), out.data_ptr(), NV12, B, H, W, st))
    return out


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def kernels(dev):
    lib = _lib.load()
    st = torch.cuda.current_stream().cuda_stream
    print("# 1. conversion kernels (CUDA events, 2000 launches, four rotating buffer sets), bandwidth over 7.7 TB/s", flush=True)
    for name, (B, H, W) in (("tu_p010_to_rgb", (8, 720, 1280)), ("tu_nv12_to_rgb", (8, 720, 1280)),
                            ("tu_rgb_to_p010", (8, 1080, 1920)), ("tu_rgb_to_nv12", (8, 1080, 1920))):
        n = B * H * W
        p010 = "p010" in name
        rgb_dt = torch.float32 if p010 else torch.float16
        yuv_b, rgb_b = (2, 4) if p010 else (1, 2)
        if p010:                                        # random 16-bit words
            yv = [torch.randint(-32768, 32768, (B, 3 * H // 2, W), dtype=torch.int16, device=dev).view(torch.uint16) for _ in range(4)]
        else:
            yv = [torch.randint(0, 256, (B, 3 * H // 2, W), dtype=torch.uint8, device=dev) for _ in range(4)]
        rgb = [torch.rand(B, 3, H, W, device=dev).to(rgb_dt) for _ in range(4)]
        code = P010 if p010 else NV12
        fn = getattr(lib, name)
        if "to_rgb" in name:
            def f(i):
                fn(yv[i % 4].data_ptr(), code, rgb[i % 4].data_ptr(), B, H, W, st)
            rd, wr = n * 1.5 * yuv_b, n * 3 * rgb_b
        else:
            def f(i):
                fn(rgb[i % 4].data_ptr(), yv[i % 4].data_ptr(), code, B, H, W, st)
            rd, wr = n * 3 * rgb_b, n * 1.5 * yuv_b
        _lib.check(fn(*((yv[0].data_ptr(), code, rgb[0].data_ptr()) if "to_rgb" in name else (rgb[0].data_ptr(), yv[0].data_ptr(), code)),
                      B, H, W, st))
        timed(f, 50)
        ts = [timed(f, 400) for _ in range(5)]
        ms = statistics.median(ts)
        nbytes = rd + wr
        print(f"   {name} {B} x {H}x{W}: {ms * 1e3:7.2f} us  ({rd / 1e6:.1f} MB read + {wr / 1e6:.1f} MB written = {nbytes / 1e6:.1f} MB: "
              f"{nbytes / (ms * 1e-3) / 1e12:.2f} TB/s, {nbytes / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s; "
              f"runs {min(ts) * 1e3:.2f}..{max(ts) * 1e3:.2f} us)", flush=True)
        del yv, rgb
        torch.cuda.empty_cache()


def abc(tag, fns, rounds, iters):
    """alternating rounds over the functions (the order rotates each round); medians"""
    for f in fns.values():
        f(0)
        f(0)
    torch.cuda.synchronize()
    names = list(fns)
    ts = {k: [] for k in names}
    for r in range(rounds):
        for k in names[r % len(names):] + names[:r % len(names)]:
            ts[k].append(timed(fns[k], iters))
    med = {k: statistics.median(v) for k, v in ts.items()}
    base = med[names[-1]]
    print(f"{tag}", flush=True)
    for k in names:
        print(f"   {k:22s} {med[k]:7.3f} ms  / {names[-1]} {med[k] / base:6.4f}  (min {min(ts[k]):.3f} max {max(ts[k]):.3f})", flush=True)


def forwards(dev, rounds):
    print(f"# 2. device-resident forward, bf16 module; alternating rounds of 20 forwards ({rounds} rounds), medians", flush=True)
    for name, B, kw in (("WindowTransformer", 8, dict(res_out=(1080, 1920))), ("ResidualTransformer", 2, dict(res_out=(2160, 3840)))):
        m = model(name, dev)
        xp = frames(B, 720, 1280, dev, True)
        xn = frames(B, 720, 1280, dev, False)
        xu = (synth_frames(B, 720, 1280, seed=1) * 255).round().to(torch.uint8).to(dev)
        with torch.no_grad():
            abc(f"{name} {B} x 720p {kw}", {
                "P010 -> P010": lambda i: m(xp, in_layout="p010", out_layout="p010", **kw),
                "NV12 -> NV12": lambda i: m(xn, in_layout="nv12", out_layout="nv12", **kw),
                "uint8 CHW -> CHW": lambda i: m(xu, **kw),
            }, rounds, 20)
        del m, xp, xn, xu
        torch.cuda.empty_cache()


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 12
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print(f"# {q}; {torch.cuda.device_count()} GPU(s); torch {torch.__version__}", flush=True)
    kernels(dev)
    forwards(dev, rounds)


if __name__ == "__main__":
    main()
