#!/usr/bin/env python
"""Cost and benefit of NV12 frame I/O (profiles/nv12_io_probe.log).

  python tools/probes/nv12_io_probe.py [rounds]

1. The two conversion kernels alone (CUDA events over many launches; the inputs rotate over four buffer sets, 220 / 500 MB, so the
   working set does not stay in the 126 MB L2): tu_nv12_to_rgb at 8 x 720p, tu_rgb_to_nv12 at 8 x 1080p, with their bandwidth as a
   fraction of 7.7 TB/s.  Bytes from the shapes: 1.5 B read + 6 B written a pixel, and the reverse.
2. Device-resident whole forwards of the bf16 module, NV12 -> NV12 (A) against uint8 CHW -> CHW (B), alternating rounds, medians:
   WindowTransformer 8 x 720p -> 1080p, ResidualTransformer 2 x 720p -> 4K.
3. End to end through FramePipeline (pinned host frames in and out, depth 4, two compute streams): WindowTransformer 8 x 720p ->
   1080p, pinned NV12 against pinned uint8 CHW, on one GPU; then, when the host has more, one process per GPU under torchrun (each
   rank upscales its own share of frames, as bench.py --gpus N shards them) with the aggregate frames/s.

  python -m torch.distributed.run --nproc-per-node N tools/probes/nv12_io_probe.py e2e     (what part 3 launches)
"""
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
NV12 = _lib.TU_U8 | _lib.TU_LAYOUT_NV12


def model(name, dev):
    import importlib
    m = importlib.import_module(f"transformerupscaler_b200.models.{name}.model").TransformerModel().eval()
    m.load_state_dict(synth_state_dict(name, 0), strict=True)
    return m.to(dev).bfloat16()


def nv12_frames(B, H, W, dev):
    """smooth synthetic frames as NV12, converted on the device"""
    lib = _lib.load()
    rgb = synth_frames(B, H, W, seed=1).half().to(dev)
    out = torch.empty(B, 3 * H // 2, W, dtype=torch.uint8, device=dev)
    _lib.check(lib.tu_rgb_to_nv12(rgb.data_ptr(), out.data_ptr(), NV12, B, H, W, torch.cuda.current_stream().cuda_stream))
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
    for name, (B, H, W) in (("tu_nv12_to_rgb", (8, 720, 1280)), ("tu_rgb_to_nv12", (8, 1080, 1920))):
        n = B * H * W
        nv = [torch.randint(0, 256, (B, 3 * H // 2, W), dtype=torch.uint8, device=dev) for _ in range(4)]
        rgb = [torch.rand(B, 3, H, W, device=dev).half() for _ in range(4)]
        if name == "tu_nv12_to_rgb":
            def f(i):
                lib.tu_nv12_to_rgb(nv[i % 4].data_ptr(), NV12, rgb[i % 4].data_ptr(), B, H, W, st)
        else:
            def f(i):
                lib.tu_rgb_to_nv12(rgb[i % 4].data_ptr(), nv[i % 4].data_ptr(), NV12, B, H, W, st)
        timed(f, 50)
        ts = [timed(f, 400) for _ in range(5)]
        ms = statistics.median(ts)
        nbytes = n * 7.5
        print(f"   {name} {B} x {H}x{W}: {ms * 1e3:7.2f} us  ({nbytes / 1e6:.1f} MB: {nbytes / (ms * 1e-3) / 1e12:.2f} TB/s, "
              f"{nbytes / (ms * 1e-3) / PEAK * 100:.0f} % of 7.7 TB/s; runs {min(ts) * 1e3:.2f}..{max(ts) * 1e3:.2f} us)", flush=True)
        del nv, rgb


def ab(tag, fa, fb, rounds, iters):
    for f in (fa, fb):
        f(0)
        f(0)
    torch.cuda.synchronize()
    ta, tb = [], []
    for r in range(rounds):
        pair = ((ta, fa), (tb, fb)) if r % 2 == 0 else ((tb, fb), (ta, fa))
        for lst, f in pair:
            lst.append(timed(f, iters))
    ma, mb = statistics.median(ta), statistics.median(tb)
    print(f"{tag:52s} A {ma:7.3f} ms  B {mb:7.3f} ms  A/B {ma / mb:6.4f}  "
          f"(A min {min(ta):.3f} max {max(ta):.3f}; B min {min(tb):.3f} max {max(tb):.3f})", flush=True)


def forwards(dev, rounds):
    print("# 2. device-resident forward, bf16 module: A = NV12 -> NV12, B = uint8 CHW -> CHW; alternating rounds of 20, medians",
          flush=True)
    for name, B, kw in (("WindowTransformer", 8, dict(res_out=(1080, 1920))), ("ResidualTransformer", 2, dict(res_out=(2160, 3840)))):
        m = model(name, dev)
        xn = nv12_frames(B, 720, 1280, dev)
        xu = (synth_frames(B, 720, 1280, seed=1) * 255).round().to(torch.uint8).to(dev)
        with torch.no_grad():
            ab(f"{name} {B} x 720p {kw}", lambda i: m(xn, in_layout="nv12", out_layout="nv12", **kw), lambda i: m(xu, **kw), rounds, 20)
        del m, xn, xu
        torch.cuda.empty_cache()


def e2e_rate(dev, nv12, steps=60, B=8):
    """frames/s of FramePipeline over `steps` batches of B frames, pinned host buffers both sides"""
    from transformerupscaler_b200.pipeline import FramePipeline
    m = model("WindowTransformer", dev)
    if nv12:
        hin = [nv12_frames(B, 720, 1280, dev).cpu().pin_memory() for _ in range(4)]
        hout = [torch.empty((B, 1620, 1920), dtype=torch.uint8).pin_memory() for _ in range(4)]
        kw = dict(in_layout="nv12", out_layout="nv12")
    else:
        hin = [(synth_frames(B, 720, 1280, seed=i) * 255).round().to(torch.uint8).pin_memory() for i in range(4)]
        hout = [torch.empty((B, 3, 1080, 1920), dtype=torch.uint8).pin_memory() for _ in range(4)]
        kw = {}
    pipe = FramePipeline(m, depth=4, device=dev, compute_streams=2, res_out=(1080, 1920), **kw)
    for i in range(8):
        pipe.submit(hin[i % 4], hout[i % 4])
    pipe.drain()
    if torch.distributed.is_initialized():
        torch.distributed.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        pipe.submit(hin[i % 4], hout[i % 4])
    pipe.drain()
    return steps * B / (time.perf_counter() - t0)


def e2e_rank():
    import torch.distributed as dist
    local, world = int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    rates = {}
    for r in range(3):                                  # alternate the two formats; median of three per format
        for nv in ((True, False) if r % 2 == 0 else (False, True)):
            rates.setdefault(nv, []).append(e2e_rate(dev, nv))
    out = {}
    for nv, rs in rates.items():
        t = torch.tensor([statistics.median(rs)], device=dev, dtype=torch.float64)
        dist.all_reduce(t)
        out[nv] = t.item()
    if dist.get_rank() == 0:
        print(f"   N={world}: NV12 {out[True]:8.0f} frames/s   uint8 CHW {out[False]:8.0f} frames/s   NV12/uint8 {out[True] / out[False]:.3f}",
              flush=True)
    dist.destroy_process_group()


def main():
    rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 10
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print(f"# {q}; {torch.cuda.device_count()} GPU(s); torch {torch.__version__}", flush=True)
    kernels(dev)
    forwards(dev, rounds)
    print("# 3. end to end, FramePipeline, WindowTransformer 8 x 720p -> 1080p, pinned host frames both sides, depth 4, 2 compute "
          "streams, 60 batches after 8 warm-up batches, alternating, median of 3", flush=True)
    rates = {True: [], False: []}
    for r in range(3):
        for nv in ((True, False) if r % 2 == 0 else (False, True)):
            rates[nv].append(e2e_rate(dev, nv))
    a, b = statistics.median(rates[True]), statistics.median(rates[False])
    print(f"   N=1: NV12 {a:8.0f} frames/s   uint8 CHW {b:8.0f} frames/s   NV12/uint8 {a / b:.3f}", flush=True)
    n = torch.cuda.device_count()
    if n > 1:
        torch.cuda.empty_cache()
        subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr=127.0.0.1",
                        "--master-port=29613", os.path.abspath(__file__), "e2e"], check=True)
    else:
        print("   N>1: not measured (one GPU on this host)", flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "e2e":
        e2e_rank()
    else:
        main()
