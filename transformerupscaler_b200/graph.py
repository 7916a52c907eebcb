"""CUDA-graph replay of one TransformerModel.forward per input shape (SURVEY.md n3: low-latency entry point).

The reference's speed_test.py / app_overlay.py call the model once per frame at batch 1 (speed_test.py:60-67,
app_overlay.py:365-372).  At that size a forward is ~0.4 ms of GPU time behind ~0.15 ms of host work (Python dispatch, the
packed-weights key, eight tensor-map encodes, eight launches).  `GraphedModel` captures the whole forward -- every kernel of
tu_forward with its programmatic-dependent-launch edges, the tile-flag memset and the workspace -- into one CUDA graph per
(shape, dtype, keyword) signature and replays it with a single cudaGraphLaunch.

The library itself never allocates or synchronises, so tu_forward is capturable as is; the workspace and the output live in the
graph's private memory pool.  Results are bitwise those of the eager call (tests/test_zz_gpu_pipeline.py).
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch


class GraphedModel:
    """model(x, **kw) through a captured CUDA graph.  The returned tensor is the graph's static output buffer: it is overwritten
    by the next call with the same signature (clone it to keep it)."""

    def __init__(self, model, warmup: int = 2):
        self.model, self.warmup = model, warmup
        self._graphs: Dict[Tuple, Tuple[torch.cuda.CUDAGraph, torch.Tensor, torch.Tensor]] = {}

    def _key(self, x: torch.Tensor, kw: dict) -> Tuple:
        ac = torch.is_autocast_enabled("cuda")
        return (tuple(x.shape), x.dtype, x.device.index, ac, torch.get_autocast_dtype("cuda") if ac else None,
                tuple(sorted((k, tuple(v) if isinstance(v, (list, tuple)) else v) for k, v in kw.items())))

    @torch.no_grad()
    def __call__(self, x: torch.Tensor, **kw) -> torch.Tensor:
        if isinstance(x, (list, tuple)) or kw.get("out") is not None:
            # a graph replays from a static input buffer, so frame planes would be copied into it: call the model directly instead
            raise TypeError("GraphedModel takes dense frame tensors only, not lists of (y, uv) frame planes or out=; call the model "
                            "itself with frame planes")
        if not x.is_cuda:
            raise RuntimeError("transformerupscaler_b200 has no CPU path: move the input to a CUDA device")
        key = self._key(x, kw)
        hit = self._graphs.get(key)
        if hit is None:
            static_in = torch.empty_like(x)
            static_in.copy_(x)
            # warm-up on a side stream: packs the weights (a host-synchronising step that must not happen under capture) and
            # sets the kernels' shared-memory attributes
            s = torch.cuda.Stream(x.device)
            s.wait_stream(torch.cuda.current_stream(x.device))
            with torch.cuda.stream(s):
                for _ in range(max(1, self.warmup)):
                    self.model(static_in, **kw)
            torch.cuda.current_stream(x.device).wait_stream(s)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                static_out = self.model(static_in, **kw)
            hit = (g, static_in, static_out)
            self._graphs[key] = hit
        g, static_in, static_out = hit
        static_in.copy_(x, non_blocking=True)
        g.replay()
        return static_out

    def invalidate(self) -> None:
        """drop the captured graphs (after the model's weights changed: a graph replays the weights it was captured with)"""
        self._graphs.clear()
