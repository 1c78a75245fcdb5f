"""Inference path (SURVEY.md 8f-2, BASELINE.json configs[1]): the eval-mode generator forward as ONE CUDA-graph replay.

Eval mode already removes the per-call work of training (no power iteration: sigma = u.(W v) from the stored vectors; BatchNorm uses
running statistics and, where it follows a convolution directly, is folded into that convolution's epilogue -- common._conv_bn_relu_eval).
What is left is ~600 dependent kernel launches for a 4->18-frame forecast, most of them the latency-bound ConvGRU steps; a CUDA graph
removes the per-launch host cost (Python + ctypes + tensor-map encoding, ~20 us each) so the GPU runs them back to back.

The latent z is still drawn on the CPU default generator in the reference's order (ref: dgmr/common.py:481) and copied into a static
device buffer before every replay, so seeded forecasts equal the eager path's.

`train_mode=True` captures the TRAIN-mode forward without autograd instead -- what the discriminator phase of a GAN step runs twice
(ref: dgmr/dgmr.py:159-160: `self(images)` under the generator's train mode, its gradients discarded): BatchNorm batch statistics, running
statistics and the spectral-norm power iteration all advance on the device inside the replay, exactly as in the eager call.

`num_samples=K > 1` captures the eval-mode ensemble forward `generator.sample(x, K)` instead -- every sampler pass of it in the one graph;
each call draws the K latents in the reference's order into a static [K, ...] buffer and replays.
"""
from __future__ import annotations

import torch

from . import _lib


class GraphedGenerator:
    """`out = GraphedGenerator(generator, example_x)(x)`: generator(x) in eval mode, replayed from a captured CUDA graph.

    `x` must have the example's shape; the returned tensor is a static buffer that the next call overwrites (clone it to keep it).
    train_mode: capture the train-mode, no-grad forward (see the module docstring); the warm-up forwards needed before the capture would
    advance the module's buffers (spectral-norm u / v, BatchNorm running statistics), so they are saved and restored around it.
    num_samples: K > 1 replays `generator.sample(x, K)` ([B,K,T,C,H,W], eval mode only).
    `launches`: C-ABI kernel launches recorded into the graph (what one replay executes without host calls)."""

    def __init__(self, generator: torch.nn.Module, example_x: torch.Tensor, warmup: int = 2, train_mode: bool = False,
                 num_samples: int = 1):
        self.num_samples = int(num_samples)
        if self.num_samples < 1:
            raise RuntimeError(f"GraphedGenerator: num_samples must be >= 1, got {num_samples}")
        if train_mode and self.num_samples > 1:
            raise RuntimeError("GraphedGenerator: num_samples > 1 is eval-mode only (train_mode=True replays single forwards)")
        if not example_x.is_cuda:
            raise RuntimeError("GraphedGenerator needs CUDA tensors (there is no CPU path)")
        be = _lib.backend()
        self.train_mode = bool(train_mode)
        if self.train_mode:
            from . import ops
            if ops.config.precision != ops.PREC_TF32:
                # the graph reads the packed weights at fixed addresses: the optimiser step refreshes the 1xTF32 packs in place, the
                # 3xTF32 (hi, lo) packs are rebuilt (ops.refresh_packs)
                raise RuntimeError("GraphedGenerator(train_mode=True) needs the 1xTF32 mode (packed weights refreshed in place)")
        self.generator = generator.train() if self.train_mode else generator.eval()
        self.x = example_x.detach().clone()
        self._latent = generator.latent_stack
        self.z = self._latent.sample_z(self.x, self.num_samples)   # static device buffer, refilled before every replay
        saved = [(b, b.detach().clone()) for b in generator.buffers()] if self.train_mode else []
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                     # warm-up off the default stream: packs weights, sets kernel attributes
            for _ in range(max(1, warmup)):
                self._forward_static()
            with torch.no_grad():
                for b, v in saved:
                    b.copy_(v)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        n0 = be.launches
        cur = torch.cuda.current_stream()
        try:
            with torch.cuda.graph(self.graph):
                self.out = self._forward_static()
        except BaseException:
            torch.cuda.set_stream(cur)                    # a failed capture leaves torch's capture stream current: put the caller's back
            be.launches = n0
            raise
        self.launches = be.launches - n0
        be.launches = n0                                  # recorded, not executed

    def _forward_static(self):
        orig = self._latent.sample_z
        self._latent.sample_z = lambda like, k=1: self.z  # the graph reads the static buffer; the draw itself happens outside
        try:
            with torch.no_grad():
                return self.generator(self.x) if self.num_samples == 1 else self.generator.sample(self.x, self.num_samples)
        finally:
            self._latent.sample_z = orig

    def __call__(self, x: torch.Tensor) -> torch.Tensor:
        if tuple(x.shape) != tuple(self.x.shape):
            raise RuntimeError(f"GraphedGenerator was captured for input shape {tuple(self.x.shape)}, got {tuple(x.shape)}")
        if self.generator.training != self.train_mode:
            raise RuntimeError("GraphedGenerator: the generator's train / eval mode changed since the capture")
        z = self._latent.sample_z(self.x, self.num_samples)   # CPU draws in the reference's RNG order + host->device copy
        self.z.copy_(z, non_blocking=True)
        self.x.copy_(x, non_blocking=True)
        self.graph.replay()
        return self.out
