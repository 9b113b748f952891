"""CUDA-graph capture of one training step (forward + loss + backward [+ gradient all-reduce]).

A step of the hot path is ~300 kernel launches of 3-2000 us each plus a few dozen tiny torch kernels; launched
eagerly from Python the GPU idles ~15 % of the time between them.  All shapes are static for a fixed batch size
(the reference's DataLoader yields one short last batch: use the eager path for it), so the whole step is captured
once into a CUDA graph and replayed: ``GraphedStep(model, criterion, x, y, supports)`` then ``loss = step(x, y)``.

The kernels launched through the C ABI take the stream from ``torch.cuda.current_stream()``, so they are captured
like any torch op; every buffer they touch comes from torch's allocator and therefore from the graph's private pool.
Gradients are accumulated into ``GradBucket`` views (static addresses).  The optimizer step stays outside the graph.
"""
from __future__ import annotations

from typing import Callable, Optional, Sequence

import torch

from .dp import GradBucket


class GraphedStep:
    def __init__(self, model: torch.nn.Module, criterion: Callable, x: torch.Tensor, y: torch.Tensor,
                 supports: Sequence, bucket: Optional[GradBucket] = None, all_reduce: bool = False,
                 warmup: int = 3):
        self.model, self.criterion, self.supports = model, criterion, list(supports)
        self.bucket = bucket if bucket is not None else GradBucket(model)
        self.all_reduce = all_reduce
        self.x = torch.empty_like(x)
        self.y = torch.empty_like(y)
        self.x.copy_(x)
        self.y.copy_(y)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                 # warm-up on a side stream (allocator + lazy inits)
            for _ in range(warmup):
                self._eager()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out, self.loss = self._eager()

    def _eager(self):
        self.bucket.zero_()
        out = self.model(obs_seq=self.x, sta_adj_list=self.supports)
        loss = self.criterion(out, self.y)
        loss.backward()
        if self.all_reduce:
            self.bucket.all_reduce_mean_()
        return out, loss

    def __call__(self, x: Optional[torch.Tensor] = None, y: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Copy the batch into the static buffers (host or device source) and replay. Returns the loss tensor
        (static buffer: read it before the next call); the replay's model output is the static buffer ``self.out``."""
        if x is not None and tuple(x.shape) != tuple(self.x.shape):
            # a batch of another size (the reference's DataLoader yields one short last batch, Data_Container.py:122):
            # shapes are baked into the captured graph, so this batch runs eagerly
            self.bucket.zero_()
            out = self.model(obs_seq=x.to(self.x.device, non_blocking=True), sta_adj_list=self.supports)
            loss = self.criterion(out, y.to(self.y.device, non_blocking=True))
            loss.backward()
            if self.all_reduce:
                self.bucket.all_reduce_mean_()
            return loss
        if x is not None:
            self.x.copy_(x, non_blocking=True)
        if y is not None:
            self.y.copy_(y, non_blocking=True)
        self.graph.replay()
        return self.loss
