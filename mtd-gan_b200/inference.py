"""Generator inference as a first-class path: `test.py:74-104` / `engine.test_MTD_GAN_Ours` (engine.py:124-129)
call `model.Generator(x)` on 1x1x512x512 slices under `torch.no_grad()`.  `GraphedGenerator` records that forward
once for a fixed micro-batch shape as a CUDA graph (43 tcgen05 conv launches + 21 fused FFT blocks of 3 passes each,
~110 kernels) and replays it per micro-batch; a batch of slices is walked in micro-batches so that one layer's
activations (33.5 MB per 512x512 slice at 32 channels) stay L2-resident between the producing and the consuming
kernel.  Slices are independent, so multi-GPU inference shards the slice list by rank with no collective
(SURVEY §8e; BASELINE configs[4]).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _ext, ops


class GraphedGenerator:
    """G: ResFFT_Generator in eval mode on a CUDA device; slices of height x width, each from 1 to 512 (512 x 512 is
    the full CT slice, smaller ones are crops).  `micro_batch` slices per graph replay."""

    def __init__(self, G, height: int = 512, width: int = 512, micro_batch: int = 1):
        self.G, self.H, self.W, self.mb = G, int(height), int(width), int(micro_batch)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.x = self.out = None
        self._versions = None

    def _param_versions(self):
        return tuple((p._version, p.data_ptr()) for p in self.G.parameters())

    @torch.no_grad()
    def capture(self, warmup: int = 2):
        dev = next(self.G.parameters()).device
        _ext.require_cuda_extension()
        self.G.eval()
        self.x = torch.zeros(self.mb, 1, self.H, self.W, device=dev)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):          # weight packs, tensor maps and workspaces are built here, once
                self.G(self.x)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = self.G(self.x)
        self._versions = self._param_versions()
        return self

    @torch.no_grad()
    def __call__(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x: (B, 1, H, W) CUDA fp32, any B (the tail micro-batch is zero padded).  Returns (B, 1, H, W)."""
        x = ops.check_input(x, "GraphedGenerator")
        if self.graph is None:
            self.capture()
        if tuple(x.shape[1:]) != (1, self.H, self.W):
            raise _ext.MtdError(f"GraphedGenerator was captured for (*, 1, {self.H}, {self.W}) inputs, got {tuple(x.shape)}")
        if self._versions != self._param_versions():
            # weights changed since the capture (load_state_dict, an optimizer step): the packed copies the graph reads are
            # rebuilt in place, the graph itself stays valid (same buffers)
            ops.repack_stale(list(self.G.parameters()))
            self._versions = self._param_versions()
        B = x.shape[0]
        if out is None:
            out = torch.empty_like(x)
        for b0 in range(0, B, self.mb):
            n = min(self.mb, B - b0)
            self.x[:n].copy_(x[b0:b0 + n], non_blocking=True)
            if n < self.mb:
                self.x[n:].zero_()
            self.graph.replay()
            out[b0:b0 + n].copy_(self.out[:n], non_blocking=True)
        return out


def shard_slices(n_slices: int, world_size: int, rank: int):
    """Contiguous slice range of `rank` when `n_slices` independent slices are sharded over `world_size` GPUs."""
    per = (n_slices + world_size - 1) // world_size
    return min(n_slices, rank * per), min(n_slices, (rank + 1) * per)
