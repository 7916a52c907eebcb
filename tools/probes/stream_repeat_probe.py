#!/usr/bin/env python
"""Run-to-run repeatability of the bench.py headline workload (WindowTransformer 720p -> 1080p, batch 8, bf16) when several
forwards are in flight on alternating CUDA streams, the way bench.py's headline loop issues them.

  python tools/probes/stream_repeat_probe.py [steps]          (profiles/stream_repeat_probe.log)

For each configuration: a one-stream forward of each of the two input buffers is the reference (same debug switches); then
`steps` forwards alternate between N streams and each output is compared with its reference on its own stream.  Prints, per
configuration, how many steps differ and, for the first few, the differing values per frame, the largest difference and the
output rows / columns they span.
"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from transformerupscaler_b200 import _lib  # noqa: E402
from transformerupscaler_b200.synth import synth_state_dict, synth_frames  # noqa: E402
from transformerupscaler_b200.models.WindowTransformer.model import TransformerModel  # noqa: E402

DEFAULTS = {b"unembed_overlap": 1, b"pdl": 1, b"fuse_dec12": 1, b"fused_stack": 1}


def main():
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 60
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    try:
        gpu = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        gpu = torch.cuda.get_device_name(dev)
    print(f"# {gpu}; torch {torch.__version__}; {steps} steps per configuration", flush=True)
    m = TransformerModel().eval()
    m.load_state_dict(synth_state_dict("WindowTransformer", 0), strict=True)
    m = m.to(dev).bfloat16()
    x_own = torch.cat([synth_frames(1, 720, 1280, seed=1000 + f) for f in range(8)], 0).to(dev).bfloat16()
    xs = [x_own, x_own.flip(0).contiguous()]          # bench.py's two input buffers

    def run(tag, nstreams, keys=()):
        for k, v in keys:
            lib.tu_debug_set(k, v)
        refs = [m(xs[0]).clone(), m(xs[1]).clone()]
        side = [torch.cuda.Stream(dev) for _ in range(nstreams)]
        for i in range(3 * nstreams):
            with torch.cuda.stream(side[i % nstreams]):
                m(xs[i & 1])
        torch.cuda.synchronize()
        e0 = torch.cuda.Event()
        e0.record()
        for s in side:
            s.wait_event(e0)
        outs = []
        for i in range(steps):
            with torch.cuda.stream(side[i % nstreams]):
                y = m(xs[i & 1])
                mk = y != refs[i & 1]
                outs.append((mk.sum(dim=(1, 2, 3)), (y.float() - refs[i & 1].float()).abs().amax(dim=(1, 2, 3)),
                             mk.any(dim=1).any(dim=2), mk.any(dim=1).any(dim=1)))
                del y, mk
        torch.cuda.synchronize()
        bad = [i for i, o in enumerate(outs) if int(o[0].sum())]
        print(f"{tag}: {len(bad)} of {steps} steps differ from the one-stream forward", flush=True)
        for i in bad[:3]:
            cnt, mx, rows, cols = (t.cpu() for t in outs[i])
            print(f"   step {i}: values per frame {cnt.tolist()}, max |diff| {mx.max().item():.4f}", flush=True)
            for f in range(8):
                if cnt[f]:
                    r, c = rows[f].nonzero().flatten(), cols[f].nonzero().flatten()
                    print(f"      frame {f}: rows {int(r.min())}-{int(r.max())}, cols {int(c.min())}-{int(c.max())}", flush=True)
        for k, _ in keys:
            lib.tu_debug_set(k, DEFAULTS[k])

    with torch.no_grad():
        run("1 stream", 1)
        run("2 streams", 2)
        run("4 streams", 4)
        run("4 streams, pdl off", 4, [(b"pdl", 0)])
        run("4 streams, unembed_overlap off", 4, [(b"unembed_overlap", 0)])
        run("4 streams, fuse_dec12 off", 4, [(b"fuse_dec12", 0)])
        run("4 streams, fused_stack off", 4, [(b"fused_stack", 0)])


if __name__ == "__main__":
    main()
