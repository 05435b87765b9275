"""CUDA-graph decode loop for ``Mamba.step`` (cross_atten/mamba.py:69-89, 342-405).

One decode step of an n-layer stack is ~10 tiny launches per layer (in_proj GEMV, conv step, x_proj, dt_proj, ssm step,
out_proj, RMSNorm, residual add): launch-bound by construction.  ``GraphedDecoder`` captures one whole-model step into a
CUDA graph over static buffers -- the token embedding, the output and every layer's (h, conv window) cache -- and replays
it per token, so the step costs one graph launch.  Same kernels, same arithmetic as ``Mamba.step``; the caches are updated
in place.  No CPU fallback.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch

from .mamba import Mamba


class GraphedDecoder:
    """decoder = GraphedDecoder(model, batch);  y = decoder.step(x)  with x: (batch, d_model) on the model's device.

    ``caches`` start as the reference's initial cache (h = zeros, conv window = zeros, mamba.py:342-373 with h=None) or can
    be seeded from a prefill with ``load_caches``: a P-token prompt costs one ``Mamba.prefill`` instead of P steps,

        _, caches = model.prefill(prompt)      # prompt: (batch, P, d_model)
        decoder.load_caches(caches)
        y = decoder.step(next_token)           # continues exactly where the prompt ended
    """

    def __init__(self, model: Mamba, batch: int, dtype: Optional[torch.dtype] = None, warmup: int = 3):
        p = next(model.parameters())
        if not p.is_cuda:
            raise RuntimeError("gfe_mamba_b200: GraphedDecoder needs the model on a CUDA device (no CPU fallback)")
        cfg = model.config
        self.model, self.batch = model, batch
        dt = dtype or p.dtype
        dev = p.device
        self.x = torch.zeros(batch, cfg.d_model, dtype=dt, device=dev)
        self.h: List[torch.Tensor] = [torch.zeros(batch, cfg.d_inner, cfg.d_state, dtype=torch.float32, device=dev) for _ in range(cfg.n_layers)]
        self.win: List[torch.Tensor] = [torch.zeros(batch, cfg.d_inner, cfg.d_conv - 1, dtype=dt, device=dev) for _ in range(cfg.n_layers)]
        self.y = torch.zeros(batch, cfg.d_model, dtype=dt, device=dev)
        self.graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.no_grad(), torch.cuda.stream(side):
            saved = [t.clone() for t in self.h + self.win]
            for _ in range(warmup):          # warm the allocator and cuBLAS handles outside the capture
                self._one_step()
            for t, s in zip(self.h + self.win, saved):
                t.copy_(s)
        torch.cuda.current_stream(dev).wait_stream(side)
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self._one_step()

    def _one_step(self) -> None:
        caches = [(self.h[i], self.win[i]) for i in range(len(self.h))]
        y, new = self.model.step(self.x, caches)
        for i, (h, w) in enumerate(new):     # ops.ssm_step / conv1d_step return fresh tensors: fold them back in place
            self.h[i].copy_(h)
            self.win[i].copy_(w)
        self.y.copy_(y)

    @torch.no_grad()
    def load_caches(self, caches: List[Tuple[Optional[torch.Tensor], torch.Tensor]]) -> None:
        for i, (h, w) in enumerate(caches):
            if h is None:
                self.h[i].zero_()
            else:
                self.h[i].copy_(h)
            self.win[i].copy_(w)

    @torch.no_grad()
    def step(self, x: torch.Tensor) -> torch.Tensor:
        """x: (batch, d_model).  Returns a view of the static output buffer (valid until the next step)."""
        self.x.copy_(x)
        self.graph.replay()
        return self.y
