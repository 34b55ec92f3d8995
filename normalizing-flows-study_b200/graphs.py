"""CUDA-graph replay of a whole training step (forward, backward, optimizer).

Small batches are launch-bound: RealNVP(2, 8, 64) on 5 000 rows (the reference's README quickstart, README.md:105-123)
issues ~510 kernels per step and spends 11 ms in eager mode, 2.7 ms when the same launches are replayed as one graph.
Every kernel of the step goes through the C ABI on torch's current stream, so stream capture records them; tensors are
allocated from the capture's private pool, and the TMA descriptors baked into the tensor-core launches stay valid
because replays reuse the same addresses.

    step = GraphedTrainStep(model, optimizer, loss_fn, example_x)     # optimizer built with capturable=True
    for x in loader:
        loss = step(x)            # copies x into the static input, replays, returns the static loss tensor

Reverse-KL / variational training draws its own samples: with a DeviceGenerator the draw reads and advances its seed
and offset in device memory, so every replay takes fresh samples (and generator.manual_seed makes the replays
reproducible); the example input is then only a placeholder.

    g = nfb200.DeviceGenerator()
    def loss_fn(m, _):
        x, lq = m.sample_and_log_prob(n, generator=g)
        return (lq - target_log_prob(x)).mean()
    step = GraphedTrainStep(model, optimizer, loss_fn, torch.empty(1, device="cuda"))
"""
from __future__ import annotations

import torch

from . import packing


class GraphedTrainStep:
    def __init__(self, model, optimizer, loss_fn, example_input, warmup=3, sync_gradients=None):
        if not example_input.is_cuda:
            raise RuntimeError("GraphedTrainStep needs CUDA tensors (libnfb200 has no CPU path)")
        self.model, self.optimizer, self.loss_fn = model, optimizer, loss_fn
        self.static_input = example_input.detach().clone()
        self._sync = sync_gradients

        def eager():
            optimizer.zero_grad(set_to_none=True)
            loss = loss_fn(model, self.static_input)
            loss.backward()
            if self._sync is not None:
                self._sync()
            optimizer.step()
            return loss

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):          # builds every cached weight layout and the optimizer state outside the graph
                eager()
        torch.cuda.current_stream().wait_stream(side)
        optimizer.zero_grad(set_to_none=True)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.static_loss = eager()

    def __call__(self, x=None):
        if x is not None:
            self.static_input.copy_(x, non_blocking=True)
        self.graph.replay()
        # the replay moved the weights (and BatchNorm statistics) without running any Python: no version counter
        # changed, so the derived weight layouts cached by the eval routes must be dropped explicitly
        packing.invalidate_caches()
        return self.static_loss.detach()
