#!/usr/bin/env python
"""NV12 / P010 frames from and to per-frame decoder / encoder surfaces (profiles/yuv_surface_probe.log).

  python tools/probes/yuv_surface_probe.py [rounds]

Surfaces here are what a decoder's pool looks like: one allocation per plane kind, rows of W samples at a pitch of W rounded up to
512 bytes, the chroma plane at the aligned height (1088 rows for 1080p) behind the luma, and the frames of a batch at shuffled slots.

1. The four conversion kernels, dense (B, 3H/2, W) buffers against surfaces (tu_yuv420_planes_to_rgb / tu_rgb_to_yuv420_planes), in
   alternating rounds: CUDA events over 400 launches a round, inputs rotating over four buffer sets so the working set (442 MB and
   more) does not stay in the 126 MB L2.  Bytes from the shapes as in p010_io_probe.py.
2. Device-resident whole forwards of the bf16 module in alternating rounds of 20 forwards, medians.  Arm A: surfaces in, surfaces out
   (tu_forward_planes).  Arm B: what a caller has to do without surfaces: gather the B surfaces into one dense tensor with
   Tensor.copy_ (two copies a frame), the dense forward, and a scatter of the dense result into the B output surfaces.  Arm C: the dense
   forward alone.  WindowTransformer 8 x 720p NV12 -> 1080p NV12, ResidualTransformer 2 x 720p P010 -> 4K P010.
3. The card's name, power limit and SM clock, read in the same run (first line).
"""
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from transformerupscaler_b200 import _lib, engine  # noqa: E402
from transformerupscaler_b200.synth import synth_state_dict, synth_frames  # noqa: E402

PEAK = 7.7e12
NV12 = _lib.TU_U8 | _lib.TU_LAYOUT_NV12
P010 = _lib.TU_U16 | _lib.TU_LAYOUT_P010


def model(name, dev):
    import importlib
    m = importlib.import_module(f"transformerupscaler_b200.models.{name}.model").TransformerModel().eval()
    m.load_state_dict(synth_state_dict(name, 0), strict=True)
    return m.to(dev).bfloat16()


def pool(B, H, W, p010, dev, seed=0):
    """B surfaces of a decoder-style pool: [(y, uv)] strided views, 512-byte pitch, chroma at the 16-aligned height + 8 rows"""
    es = 2 if p010 else 1
    pitch = -(-W * es // 512) * 512
    Hal = -(-H // 16) * 16 + 8
    buf = torch.zeros(B, Hal + H // 2, pitch, dtype=torch.uint8, device=dev)
    slots = torch.randperm(B, generator=torch.Generator().manual_seed(seed)).tolist()
    dt = torch.uint16 if p010 else torch.uint8
    return [(buf[s, :H, :W * es].view(dt), buf[s, Hal:Hal + H // 2, :W * es].view(dt)) for s in slots]


def fill(planes, dense):
    H = planes[0][0].shape[0]
    for b, (y, uv) in enumerate(planes):
        y.copy_(dense[b, :H])
        uv.copy_(dense[b, H:])


def timed(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def abc(fns, rounds, iters):
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
    print(f"# 1. conversion kernels, dense buffers vs surfaces: alternating rounds of 400 launches ({rounds} rounds), four rotating "
          "buffer sets; medians, bandwidth over 7.7 TB/s", flush=True)
    for name, (B, H, W) in (("p010_to_rgb", (8, 720, 1280)), ("nv12_to_rgb", (8, 720, 1280)),
                            ("rgb_to_p010", (8, 1080, 1920)), ("rgb_to_nv12", (8, 1080, 1920))):
        n = B * H * W
        p010 = "p010" in name
        to_rgb = name.endswith("to_rgb")
        rgb_dt = torch.float32 if p010 else torch.float16
        yuv_b, rgb_b = (2, 4) if p010 else (1, 2)
        code = P010 if p010 else NV12
        if p010:
            yv = [torch.randint(-32768, 32768, (B, 3 * H // 2, W), dtype=torch.int16, device=dev).view(torch.uint16) for _ in range(4)]
        else:
            yv = [torch.randint(0, 256, (B, 3 * H // 2, W), dtype=torch.uint8, device=dev) for _ in range(4)]
        rgb = [torch.rand(B, 3, H, W, device=dev).to(rgb_dt) for _ in range(4)]
        surf = [pool(B, H, W, p010, dev, seed=k) for k in range(4)]
        for s, d in zip(surf, yv):
            fill(s, d)
        desc = [engine._descriptors(engine._flat(s)) for s in surf]
        dense_fn = getattr(lib, "tu_" + name)
        if to_rgb:
            def dense(i):
                dense_fn(yv[i % 4].data_ptr(), code, rgb[i % 4].data_ptr(), B, H, W, st)

            def planes(i):
                lib.tu_yuv420_planes_to_rgb(desc[i % 4], code, rgb[i % 4].data_ptr(), B, H, W, st)
            rd, wr = n * 1.5 * yuv_b, n * 3 * rgb_b
        else:
            def dense(i):
                dense_fn(rgb[i % 4].data_ptr(), yv[i % 4].data_ptr(), code, B, H, W, st)

            def planes(i):
                lib.tu_rgb_to_yuv420_planes(rgb[i % 4].data_ptr(), desc[i % 4], code, B, H, W, st)
            rd, wr = n * 3 * rgb_b, n * 1.5 * yuv_b
        _lib.check(lib.tu_yuv420_planes_to_rgb(desc[0], code, rgb[0].data_ptr(), B, H, W, st) if to_rgb else
                   lib.tu_rgb_to_yuv420_planes(rgb[0].data_ptr(), desc[0], code, B, H, W, st))
        ts = abc({"dense": dense, "surfaces": planes}, rounds, 400)
        nbytes = rd + wr
        for k, v in ts.items():
            ms = statistics.median(v)
            print(f"   {name:11s} {k:8s} {B} x {H}x{W}: {ms * 1e3:7.2f} us  ({nbytes / 1e6:.1f} MB: {nbytes / (ms * 1e-3) / 1e12:.2f} TB/s, "
                  f"{nbytes / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s; rounds {min(v) * 1e3:.2f}..{max(v) * 1e3:.2f} us)", flush=True)
        del yv, rgb, surf, desc
        torch.cuda.empty_cache()


def forwards(dev, rounds):
    print(f"# 2. device-resident forward, bf16 module; alternating rounds of 20 forwards ({rounds} rounds), medians", flush=True)
    for name, B, fmt, kw, (oh, ow) in (("WindowTransformer", 8, "nv12", dict(res_out=(1080, 1920)), (1080, 1920)),
                                       ("ResidualTransformer", 2, "p010", dict(res_out=(2160, 3840)), (2160, 3840))):
        p010 = fmt == "p010"
        m = model(name, dev)
        lib = _lib.load()
        st = torch.cuda.current_stream().cuda_stream
        rgb = synth_frames(B, 720, 1280, seed=1).to(dev)
        x = torch.empty(B, 1080, 1280, dtype=torch.uint16 if p010 else torch.uint8, device=dev)
        if p010:
            _lib.check(lib.tu_rgb_to_p010(rgb.data_ptr(), x.data_ptr(), P010, B, 720, 1280, st))
        else:
            rgb = rgb.half()
            _lib.check(lib.tu_rgb_to_nv12(rgb.data_ptr(), x.data_ptr(), NV12, B, 720, 1280, st))
        sin = pool(B, 720, 1280, p010, dev, seed=1)
        fill(sin, x)
        sout = pool(B, oh, ow, p010, dev, seed=2)
        xd = torch.empty_like(x)
        lk = dict(in_layout=fmt, out_layout=fmt, **kw)

        def arm_a(i):
            m(sin, out=sout, **lk)

        def arm_b(i):
            fill_dense(xd, sin)
            y = m(xd, **lk)
            fill(sout, y)

        def arm_c(i):
            m(x, **lk)

        def fill_dense(d, planes):
            H = planes[0][0].shape[0]
            for b, (yy, uv) in enumerate(planes):
                d[b, :H].copy_(yy)
                d[b, H:].copy_(uv)

        with torch.no_grad():
            want = m(x, **lk)
            arm_a(0)
            torch.cuda.synchronize()
            got = torch.stack([torch.cat([yy, uv], 0) for yy, uv in sout])
            assert torch.equal(got, want), "surfaces forward differs from the dense forward"
            ts = abc({"A surfaces -> surfaces": arm_a, "B gather + dense + scatter": arm_b, "C dense forward alone": arm_c}, rounds, 20)
        base = statistics.median(ts["C dense forward alone"])
        print(f"{name} {B} x 720p {fmt.upper()} -> {oh}p {fmt.upper()}", flush=True)
        for k, v in ts.items():
            med = statistics.median(v)
            print(f"   {k:28s} {med:7.3f} ms  / C {med / base:6.4f}  (rounds {min(v):.3f}..{max(v):.3f})", flush=True)
        del m, x, xd, sin, sout, rgb, want
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
