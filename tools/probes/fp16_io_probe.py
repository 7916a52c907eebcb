#!/usr/bin/env python
"""Cost of fp16 image I/O (a .half() module: fp16 frames in, fp16 image out, bf16 tensor-core compute) against the bf16 module with
bf16 I/O, which moves the same bytes.  Device-resident inputs, one process, A/B rounds alternated, medians.

  python tools/probes/fp16_io_probe.py [rounds]          (profiles/fp16_io_probe.log)

1. Whole forwards: WindowTransformer 8 x 720p -> 1080p, FastTransformer 720p x2 (4 frames), ResidualTransformer 720p -> 4K (2 frames):
   the fp16 module on fp16 frames vs the bf16 module on bf16 frames.
2. Per kernel (tu_profile, every kernel bracketed by events): conv1_conv2 and bicubic_add_clamp of the WindowTransformer forward,
   fp16 vs bf16 frames.
3. fp16 frames into a bf16 module: passed as they are vs an explicit x.float() first (what the library did before).
"""
import ctypes as C
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from transformerupscaler_b200 import _lib  # noqa: E402
from transformerupscaler_b200.synth import synth_state_dict, synth_frames  # noqa: E402

WORKLOADS = [("WindowTransformer", 8, 720, 1280, dict(res_out=(1080, 1920))),
             ("FastTransformer", 4, 720, 1280, dict(upscale_factor=2)),
             ("ResidualTransformer", 2, 720, 1280, dict(res_out=(2160, 3840)))]


def model(name, dev):
    import importlib
    m = importlib.import_module(f"transformerupscaler_b200.models.{name}.model").TransformerModel().eval()
    m.load_state_dict(synth_state_dict(name, 0), strict=True)
    return m.to(dev)


def timed(fn, iters):
    """ms per call of fn over `iters` back-to-back calls (device events)"""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def ab(tag, fa, fb, rounds, iters):
    for f in (fa, fb):
        f()
        f()
    torch.cuda.synchronize()
    ta, tb = [], []
    for r in range(rounds):
        pair = ((ta, fa), (tb, fb)) if r % 2 == 0 else ((tb, fb), (ta, fa))
        for lst, f in pair:
            lst.append(timed(f, iters))
    ma, mb = statistics.median(ta), statistics.median(tb)
    print(f"{tag:58s} A {ma:8.3f} ms  B {mb:8.3f} ms  A/B {ma / mb:6.4f}  "
          f"(A min {min(ta):.3f} max {max(ta):.3f}; B min {min(tb):.3f} max {max(tb):.3f})", flush=True)


def profile(lib, f, iters):
    f()
    torch.cuda.synchronize()
    lib.tu_profile_reset()
    lib.tu_profile_enable(2)
    for _ in range(iters):
        f()
    torch.cuda.synchronize()
    lib.tu_profile_enable(0)
    out = {}
    for name in (b"conv1_conv2", b"bicubic_add_clamp"):
        ms, n = C.c_double(), C.c_int()
        lib.tu_profile_collect(name, C.byref(ms), C.byref(n))
        out[name.decode()] = ms.value / max(n.value, 1)
    lib.tu_profile_reset()
    return out


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    try:
        gpu = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        gpu = torch.cuda.get_device_name(dev)
    print(f"# {gpu}; torch {torch.__version__}; {rounds} alternating rounds per comparison, medians", flush=True)
    print("# 1. whole forward: A = .half() module on fp16 frames, B = .bfloat16() module on bf16 frames", flush=True)
    with torch.no_grad():
        for name, B, H, W, kw in WORKLOADS:
            m = model(name, dev)
            m16, mb = m.half(), model(name, dev).bfloat16()
            x = synth_frames(B, H, W, seed=7).to(dev)
            x16, xb = x.half(), x.bfloat16()
            iters = 5 if name != "FastTransformer" else 10
            ab(f"{name} {B} x {H}x{W} {kw}", lambda: m16(x16, **kw), lambda: mb(xb, **kw), rounds, iters)
            if name == "WindowTransformer":
                print("# 2. per kernel (tu_profile, mean ms per launch): fp16 frames vs bf16 frames", flush=True)
                for r in range(3):
                    pa = profile(lib, lambda: m16(x16, **kw), 10)
                    pb = profile(lib, lambda: mb(xb, **kw), 10)
                    print("   " + "  ".join(f"{k}: fp16 {pa[k]:.4f} bf16 {pb[k]:.4f} ratio {pa[k] / pb[k]:.4f}" for k in pa), flush=True)
                print("# 3. fp16 frames into the bf16 module: A = passed as they are, B = x.float() first (the old path)", flush=True)
                ab(f"{name} {B} x {H}x{W} bf16 module", lambda: mb(x16, **kw), lambda: mb(x16.float(), **kw), rounds, iters)
            del m, m16, mb, x, x16, xb
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
