"""Host-buffer frame pipeline: pinned host frames -> device -> TransformerModel.forward -> pinned host frames,
with the H2D copy, the forward and the D2H copy of consecutive batches overlapped on three CUDA streams.

This is the end-to-end entry a video caller uses (the reference's speed_test.py / app_overlay.py do a
synchronous batch-1 `.to(device)` -> model -> `.cpu()` loop, speed_test.py:60-67, app_overlay.py:365-391).

Buffer lifetime contract: `submit(host_in, host_out)` returns as soon as the work is ENQUEUED.  The caller may overwrite
`host_in` only after `ticket.input_consumed()` (or `ticket.wait_input()`), and may read `host_out` only after `ticket.wait()`;
`drain()` waits for everything submitted so far.
"""
from __future__ import annotations

from typing import List, Optional

import torch


class Ticket:
    """Handle of one submitted batch: tells when its pinned input has been read and when its pinned output is complete."""

    __slots__ = ("_ev_in", "_ev_out", "index")

    def __init__(self, index: int, ev_in: torch.cuda.Event, ev_out: torch.cuda.Event):
        self.index, self._ev_in, self._ev_out = index, ev_in, ev_out

    def input_consumed(self) -> bool:
        """True once the H2D copy has read host_in (the buffer may be reused)."""
        return self._ev_in.query()

    def wait_input(self) -> None:
        self._ev_in.synchronize()

    def done(self) -> bool:
        """True once host_out holds the upscaled frames."""
        return self._ev_out.query()

    def wait(self) -> None:
        self._ev_out.synchronize()


class FramePipeline:
    def __init__(self, model, depth: int = 2, device: Optional[torch.device] = None, compute_streams: int = 2, **forward_kw):
        """compute_streams > 1: consecutive batches run their forwards on alternating streams, so the kernels of one batch
        can fill the SMs the other batch's partly filled waves leave idle (needs depth >= compute_streams)"""
        if forward_kw.get("out") is not None:
            raise TypeError("FramePipeline writes dense host frames: out= (frame planes) is not supported; call the model itself")
        self.model, self.kw, self.depth = model, forward_kw, depth
        self.device = device or next(model.parameters()).device
        self.s_in, self.s_out = (torch.cuda.Stream(self.device) for _ in range(2))
        self.s_comps = [torch.cuda.Stream(self.device) for _ in range(max(1, min(compute_streams, depth)))]
        self.dev_in: List[Optional[torch.Tensor]] = [None] * depth
        self.dev_out: List[Optional[torch.Tensor]] = [None] * depth
        self.ev_comp = [torch.cuda.Event() for _ in range(depth)]
        self.tickets: List[Optional[Ticket]] = [None] * depth
        self.n = 0

    @torch.no_grad()
    def submit(self, host_in: torch.Tensor, host_out: torch.Tensor) -> Ticket:
        """Enqueue one batch: host_in (pinned) is upscaled into host_out (pinned).  Returns immediately with the batch's Ticket
        (see the buffer lifetime contract in the module docstring)."""
        if not isinstance(host_in, torch.Tensor) or not isinstance(host_out, torch.Tensor):
            raise TypeError("FramePipeline takes dense pinned frame tensors only, not lists of (y, uv) frame planes")
        slot = self.n % self.depth
        if self.tickets[slot] is not None:
            self.tickets[slot].wait()                # slot's previous result has left the device
        # fresh events per batch: a Ticket stays valid after its slot has been reused
        ev_in, ev_out = torch.cuda.Event(), torch.cuda.Event()
        with torch.cuda.stream(self.s_in):
            if self.dev_in[slot] is None or self.dev_in[slot].shape != host_in.shape or self.dev_in[slot].dtype != host_in.dtype:
                # allocated on the stream that fills it (the caching allocator orders reuse per stream)
                self.dev_in[slot] = torch.empty(host_in.shape, dtype=host_in.dtype, device=self.device)
            self.dev_in[slot].copy_(host_in, non_blocking=True)
            ev_in.record(self.s_in)
        s_comp = self.s_comps[self.n % len(self.s_comps)]
        with torch.cuda.stream(s_comp):
            s_comp.wait_event(ev_in)
            out = self.model(self.dev_in[slot], **self.kw)
            self.ev_comp[slot].record(s_comp)
        with torch.cuda.stream(self.s_out):
            self.s_out.wait_event(self.ev_comp[slot])
            host_out.copy_(out, non_blocking=True)
            ev_out.record(self.s_out)
        out.record_stream(self.s_out)
        self.dev_out[slot] = out
        t = Ticket(self.n, ev_in, ev_out)
        self.tickets[slot] = t
        self.n += 1
        return t

    def drain(self) -> None:
        for s in (self.s_in, *self.s_comps, self.s_out):
            s.synchronize()
