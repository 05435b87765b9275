"""Drop-in for the reference's ``cross_atten/mamba.py``: same classes, constructor arguments, parameter
names/shapes (state-dict compatible) and call signatures; the work under ``MambaBlock`` is done by the
sm_100a kernels behind ``gfe_mamba_b200.ops``.

What stays in torch (by design, SURVEY 8a): the four projections (cuBLAS GEMMs).
What moved into hand-written CUDA: causal depthwise conv + SiLU, softplus(+bias), discretisation, the scan,
the C contraction, the D skip, the SiLU(z) gate, their backward passes, the decode step, and (SURVEY 8f rank 1) the
residual add fused with the next layer's RMSNorm in ``Mamba.forward``.

Reference line numbers below refer to cross_atten/mamba.py of Tinysqua/GFE-Mamba.
"""
import math
from dataclasses import dataclass
from typing import Union

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import ops
from .ops import add_rmsnorm
from .pscan import pscan


def _fusable_norm(x: torch.Tensor, config) -> bool:
    """The fused add + RMSNorm kernels move rows as 16-byte vectors (ops.add_rmsnorm; rows of up to 256 vectors stay in
    registers, wider ones take two passes); a d_model that is not a multiple of the vector width takes the module-by-module
    path."""
    vec = 16 // x.element_size()
    return x.dtype in (torch.float32, torch.bfloat16, torch.float16) and config.d_model % vec == 0


@dataclass
class MambaConfig:
    """Field-for-field the reference's dataclass (mamba.py:31-59)."""
    d_model: int  # D
    n_layers: int
    dt_rank: Union[int, str] = 'auto'
    d_state: int = 16  # N
    expand_factor: int = 2  # E
    d_conv: int = 4

    dt_min: float = 0.001
    dt_max: float = 0.1
    dt_init: str = "random"  # "random" or "constant"
    dt_scale: float = 1.0
    dt_init_floor = 1e-4  # un-annotated in the reference too: a class attribute, not a field (mamba.py:44)

    rms_norm_eps: float = 1e-5

    bias: bool = False
    conv_bias: bool = True
    inner_layernorms: bool = False

    pscan: bool = True  # kept for API compatibility; both modes run the same fused kernel here
    use_cuda: bool = False  # accepted (mamba_transformer.py:65 passes True); never needs mamba_ssm here

    def __post_init__(self):
        self.d_inner = self.expand_factor * self.d_model  # ED

        if self.dt_rank == 'auto':
            self.dt_rank = math.ceil(self.d_model / 16)


class Mamba(nn.Module):
    """mamba.py:61-89."""

    def __init__(self, config: MambaConfig):
        super().__init__()
        self.config = config
        self.layers = nn.ModuleList(ResidualBlock(config) for _ in range(config.n_layers))

    def forward(self, x):
        # x : (B, L, D) -> (B, L, D)
        if not x.is_cuda:
            raise RuntimeError("gfe_mamba_b200.Mamba: CUDA tensors required (this library has no CPU fallback); "
                               f"got input on {x.device}")
        if len(self.layers) == 0:
            return x
        if not _fusable_norm(x, self.config):
            # d_model not a multiple of the fused add + RMSNorm kernels' 16-byte vector: the reference's module-by-module
            # form, same CUDA kernels in the mixer
            for layer in self.layers:
                x = layer(x)
            return x
        # Same arithmetic as `x = mixer(norm(x)) + x` per layer (mamba.py:103), with every residual add fused into the
        # NEXT layer's RMSNorm: one pass over the residual stream per layer instead of an add and a five-kernel norm.
        resid, branch = x, None
        for layer in self.layers:
            resid, normed = add_rmsnorm(resid, branch, layer.norm.weight, layer.norm.eps)
            branch = layer.mixer(normed)
        return branch + resid

    def forward_mean(self, x):
        """``torch.mean(self(x), dim=1, keepdim=True)`` -- what the classifier head does with the stack's output
        (mamba_transformer.py:122-123) -- with the last residual add fused into the pooling: the (B, L, D) output is never
        written.  Extension of the reference API (SURVEY 8f rank 4); INTEGRATION.md shows the one-line caller change."""
        if not x.is_cuda:
            raise RuntimeError("gfe_mamba_b200.Mamba: CUDA tensors required (this library has no CPU fallback); "
                               f"got input on {x.device}")
        if len(self.layers) == 0 or not _fusable_norm(x, self.config):
            return ops.add_mean_pool(self(x), None)
        resid, branch = x, None
        for layer in self.layers:
            resid, normed = add_rmsnorm(resid, branch, layer.norm.weight, layer.norm.eps)
            branch = layer.mixer(normed)
        return ops.add_mean_pool(branch, resid)

    def step(self, x, caches):
        # x : (B, D); caches : [(h, inputs)] per layer
        for idx in range(len(self.layers)):
            x, caches[idx] = self.layers[idx].step(x, caches[idx])
        return x, caches

    def prefill(self, x, caches=None):
        """Many tokens of decoding at once.  x: (B, L, D); caches: [(h (B, ED, N) fp32 or None, inputs (B, ED, d_conv-1))] per
        layer in the convention of ``step``, or None for the reference's initial cache (h = None, a zero conv window in the
        activation dtype).  Returns (y (B, L, D), caches).

        Gives the same output rows and the same caches as ``x.shape[1]`` calls of ``step`` from ``caches``; when ``caches`` is
        what a prefix left, ``y`` equals the last rows of ``forward`` over prefix + ``x``.  So a prompt can be prefilled in one
        call (``_, caches = model.prefill(prompt)``, then ``step`` or ``GraphedDecoder.load_caches(caches)``), in chunks of
        bounded memory, or continued after decoding.  Extension of the reference API (like ``forward_mean``); the layers take
        the scan and conv kernels from the carried state where they are compiled and fall back to ``step`` token by token
        otherwise (see ``MambaBlock.prefill``).  ``caches`` is not modified."""
        if not x.is_cuda:
            raise RuntimeError("gfe_mamba_b200.Mamba: CUDA tensors required (this library has no CPU fallback); "
                               f"got input on {x.device}")
        cfg = self.config
        if caches is None:
            dt = torch.get_autocast_dtype("cuda") if torch.is_autocast_enabled("cuda") else x.dtype
            caches = [(None, torch.zeros(x.shape[0], cfg.d_inner, cfg.d_conv - 1, dtype=dt, device=x.device))
                      for _ in self.layers]
        caches = list(caches)
        if len(self.layers) == 0:
            return x, caches
        if not _fusable_norm(x, cfg):
            for i, layer in enumerate(self.layers):
                x, caches[i] = layer.prefill(x, caches[i])
            return x, caches
        # the add + RMSNorm structure of forward
        resid, branch = x, None
        for i, layer in enumerate(self.layers):
            resid, normed = add_rmsnorm(resid, branch, layer.norm.weight, layer.norm.eps)
            branch, caches[i] = layer.mixer.prefill(normed, caches[i])
        return branch + resid, caches


class ResidualBlock(nn.Module):
    """mamba.py:91-117: output = mixer(norm(x)) + x."""

    def __init__(self, config: MambaConfig):
        super().__init__()
        self.mixer = MambaBlock(config)
        self.norm = RMSNorm(config.d_model, config.rms_norm_eps)

    def forward(self, x):
        return self.mixer(self.norm(x)) + x

    def step(self, x, cache):
        y, cache = self.mixer.step(self.norm(x), cache)
        return y + x, cache

    def prefill(self, x, cache):
        """x: (B, L, D); ``step`` over the L tokens (see Mamba.prefill)."""
        y, cache = self.mixer.prefill(self.norm(x), cache)
        return y + x, cache


class MambaBlock(nn.Module):
    """mamba.py:119-405.  Parameter creation order and initialisation are the reference's (mamba.py:126-168) so
    a seeded construction draws the same values and reference checkpoints load with strict=True."""

    def __init__(self, config: MambaConfig):
        super().__init__()
        self.config = config

        self.in_proj = nn.Linear(config.d_model, 2 * config.d_inner, bias=config.bias)
        self.conv1d = nn.Conv1d(in_channels=config.d_inner, out_channels=config.d_inner,
                                kernel_size=config.d_conv, bias=config.conv_bias,
                                groups=config.d_inner, padding=config.d_conv - 1)
        self.x_proj = nn.Linear(config.d_inner, config.dt_rank + 2 * config.d_state, bias=False)
        self.dt_proj = nn.Linear(config.dt_rank, config.d_inner, bias=True)

        # dt_proj.weight: constant or uniform in +-dt_rank^-0.5 * dt_scale (mamba.py:141-148)
        std = config.dt_rank ** -0.5 * config.dt_scale
        initialisers = {"constant": lambda wt: nn.init.constant_(wt, std), "random": lambda wt: nn.init.uniform_(wt, -std, std)}
        if config.dt_init not in initialisers:
            raise NotImplementedError
        initialisers[config.dt_init](self.dt_proj.weight)

        # dt_proj.bias = softplus^-1(dt), dt log-uniform in [dt_min, dt_max], floored (mamba.py:150-157)
        log_lo, log_hi = math.log(config.dt_min), math.log(config.dt_max)
        dt = torch.exp(torch.rand(config.d_inner) * (log_hi - log_lo) + log_lo).clamp(min=config.dt_init_floor)
        with torch.no_grad():
            self.dt_proj.bias.copy_(dt + torch.log(-torch.expm1(-dt)))

        # S4D-real initialisation A[c, n] = n + 1, stored as its logarithm (mamba.py:160-161)
        self.A_log = nn.Parameter(torch.log(torch.arange(1, config.d_state + 1, dtype=torch.float32)).expand(config.d_inner, -1).clone())
        self.A_log._no_weight_decay = True

        self.D = nn.Parameter(torch.ones(config.d_inner))
        self.D._no_weight_decay = True

        self.out_proj = nn.Linear(config.d_inner, config.d_model, bias=config.bias)

        # optional RMSNorm on dt, B, C (mamba.py:169-176); registration order dt, B, C as in the reference
        widths = (config.dt_rank, config.d_state, config.d_state) if config.inner_layernorms else (0, 0, 0)
        self.dt_layernorm, self.B_layernorm, self.C_layernorm = (
            RMSNorm(n, config.rms_norm_eps) if n else None for n in widths)
        # config.use_cuda is accepted as-is: the fused sm_100a kernel *is* the CUDA path (no mamba_ssm import,
        # no fallback message, mamba.py:179-186).

    def _apply_layernorms(self, dt, B, C):
        norms = (self.dt_layernorm, self.B_layernorm, self.C_layernorm)
        return tuple(t if norm is None else norm(t) for norm, t in zip(norms, (dt, B, C)))

    # ------------------------------------------------------------------ training / prefill
    def forward(self, x):
        # x : (B, L, D) -> (B, L, D)          mamba.py:197-225
        xz = self.in_proj(x)                                  # (B, L, 2*ED)   GEMM
        if self._inner_fusable(xz):                           # conv -> x_proj -> dt_proj -> scan -> gate as one autograd node
            y = ops.mamba_inner_fn(xz, self.conv1d.weight, self.conv1d.bias, self.x_proj.weight, self.dt_proj.weight,
                                   self.dt_proj.bias, self.A_log, self.D)
            return self.out_proj(y)                           # GEMM
        xin, z = xz.chunk(2, dim=-1)                          # strided halves, consumed in place by the kernels
        if 2 <= self.config.d_conv <= 4:
            u = ops.causal_conv1d_silu(xin, self.conv1d.weight, self.conv1d.bias)   # conv + bias + SiLU fused (:208-212)
        else:   # filter lengths the conv kernel is not compiled for (jamba.py passes arbitrary mamba_d_conv): cuDNN
            u = F.silu(self.conv1d(xin.transpose(1, 2))[:, :, :x.shape[1]].transpose(1, 2))
        y = self._ssm_fused(u, z)                             # scan + D skip + SiLU(z) gate fused (:213-222)
        return self.out_proj(y)                               # GEMM

    def _inner_fusable(self, xz):
        """The one-node inner path serves the shapes the fused kernels are compiled for and the plain configuration (no
        inner layernorms); everything else takes the op-by-op composition below."""
        cfg = self.config
        return (xz.is_cuda and xz.dim() == 3 and cfg.d_state in ops.FUSED_D_STATES and 2 <= cfg.d_conv <= 4 and not cfg.inner_layernorms
                and xz.dtype in (torch.float32, torch.bfloat16, torch.float16) and self.x_proj.bias is None)

    def _project(self, x):
        """x_proj / split / optional layernorms / dt_proj without bias (mamba.py:235-238).  delta comes out
        channel-last (B, L, ED); the reference forms the same product as W @ delta^T."""
        deltaBC = self.x_proj(x)
        delta, B, C = torch.split(deltaBC, [self.config.dt_rank, self.config.d_state, self.config.d_state], dim=-1)
        delta, B, C = self._apply_layernorms(delta, B, C)
        delta = F.linear(delta, self.dt_proj.weight)
        return delta, B, C

    def _ssm_fused(self, x, z):
        delta, B, C = self._project(x)
        if self.config.d_state in ops.FUSED_D_STATES:
            return ops.selective_scan_fn(x, delta, self.A_log, B, C, self.D, z=z, dt_bias=self.dt_proj.bias,
                                         delta_softplus=True)
        # other state sizes: the reference's own composition on top of the CUDA pscan kernel
        delta = F.softplus(delta + self.dt_proj.bias)
        y = self.selective_scan(x, delta, -torch.exp(self.A_log.float()), B, C, self.D.float())
        return y if z is None else y * F.silu(z)

    def ssm(self, x, z):
        """mamba.py:227-263.  As in the reference the gate is applied here only when ``config.use_cuda`` is set
        (mamba.py:243-252); otherwise ``forward`` owns it.  ``forward`` itself always uses the fused form."""
        return self._ssm_fused(x, z if self.config.use_cuda else None)

    def selective_scan(self, x, delta, A, B, C, D):
        """mamba.py:265-286: x, delta (B, L, ED) with delta already softplus'ed; A (ED, N) negative; B, C (B, L, N);
        D (ED) -> y (B, L, ED) without gate."""
        if A.shape[1] in ops.FUSED_D_STATES:
            return ops.selective_scan_fn(x, delta, torch.log(-A), B, C, D, z=None, dt_bias=None, delta_softplus=False)
        deltaA = torch.exp(delta.unsqueeze(-1) * A)           # (B, L, ED, N)
        BX = (delta.unsqueeze(-1) * B.unsqueeze(2)) * x.unsqueeze(-1)
        hs = pscan(deltaA, BX)
        y = (hs @ C.unsqueeze(-1)).squeeze(3)
        return y + D * x

    def selective_scan_seq(self, x, delta, A, B, C, D):
        """mamba.py:288-318.  The reference's sequential mode is a second formulation of the same recurrence; on
        the GPU both names run the same sequential-in-time kernel."""
        return self.selective_scan(x, delta, A, B, C, D)

    # ------------------------------------------------------------------ decode
    def step(self, x, cache):
        # x : (B, D); cache : (h (B, ED, N) or None, inputs (B, ED, d_conv-1))      mamba.py:342-373
        h, inputs = cache
        xz = self.in_proj(x)                                  # (B, 2*ED)
        xin, z = xz.chunk(2, dim=1)
        if self._step_kernels_usable(xin, inputs, h) and 2 <= self.config.d_conv <= 4:
            u, inputs = ops.conv1d_step(xin, inputs, self.conv1d.weight, self.conv1d.bias)
        else:   # the reference's own window form (:357-358, 370): differentiable, any d_conv
            x_cache = xin.unsqueeze(2)
            u = F.silu(self.conv1d(torch.cat([inputs, x_cache], dim=2))[:, :, self.config.d_conv - 1])
            inputs = torch.cat([inputs[:, :, 1:], x_cache], dim=2)
        y, h = self.ssm_step(u, h, z=z)
        output = self.out_proj(y)
        return output, (h, inputs)

    def prefill(self, x, cache):
        """x: (B, L, D); cache: (h, inputs) as for ``step``.  Returns (y (B, L, D), cache): the outputs and the cache of L
        calls of ``step`` from ``cache``.  Where the kernels are compiled (d_state in ops.FUSED_D_STATES, 2 <= d_conv <= 4) and
        no gradient is asked for, the forward path runs once over the L tokens from the carried state: in_proj ->
        conv1d_prefill -> x_proj / dt_proj (inner layernorms included) -> ssm_prefill (gate fused) -> out_proj.  Otherwise
        ``step`` runs token by token: the reference's semantics, differentiable, any configuration."""
        h, inputs = cache
        cfg = self.config
        if cfg.d_state in ops.FUSED_D_STATES and 2 <= cfg.d_conv <= 4 and self._step_kernels_usable(x, h, inputs):
            y, cache = self._prefill_inner(x, h, inputs)
            return self.out_proj(y), cache
        ys = []
        for t in range(x.shape[1]):
            y, cache = self.step(x[:, t], cache)
            ys.append(y)
        return torch.stack(ys, 1), cache

    def _prefill_inner(self, x, h, inputs):
        """prefill between in_proj and out_proj: (y (B, L, ED), (h, inputs)).  A function of its own so that xz, u, delta and
        x_proj's output are freed before out_proj runs: the peak stays that of forward (whose inner node frees them too)."""
        xz = self.in_proj(x)                                  # (B, L, 2*ED)
        xin, z = xz.chunk(2, dim=-1)                          # strided halves, consumed in place
        u, inputs = ops.conv1d_prefill(xin, inputs, self.conv1d.weight, self.conv1d.bias)
        delta, B, C = self._project(u)
        y, h = ops.ssm_prefill(u, delta, self.A_log, B, C, self.D, h, z=z, dt_bias=self.dt_proj.bias, delta_softplus=True)
        return y, (h, inputs)

    def _step_kernels_usable(self, *tensors):
        """The decode kernels are inference-only: a caller that backpropagates through ``step`` (the reference's step is
        ordinary differentiable torch code) gets the torch composition instead of a silently detached graph."""
        if not torch.is_grad_enabled():
            return True
        return not (any(t is not None and t.requires_grad for t in tensors) or any(p.requires_grad for p in self.parameters()))

    def ssm_step(self, x, h, z=None):
        """mamba.py:375-405 (+ the gate of :364-367 when ``z`` is given).  Returns (y, h_new)."""
        deltaBC = self.x_proj(x)
        delta, B, C = torch.split(deltaBC, [self.config.dt_rank, self.config.d_state, self.config.d_state], dim=-1)
        delta, B, C = self._apply_layernorms(delta, B, C)
        delta = F.linear(delta, self.dt_proj.weight)
        if self.config.d_state in ops.FUSED_D_STATES and self._step_kernels_usable(x, h, z):
            return ops.ssm_step(x, delta, self.A_log, B, C, self.D, h, z=z, dt_bias=self.dt_proj.bias, delta_softplus=True)
        # other state sizes, or a caller that differentiates through the step: the reference's composition (:391-403)
        A = -torch.exp(self.A_log.float())
        delta = F.softplus(delta + self.dt_proj.bias)
        deltaA = torch.exp(delta.unsqueeze(-1) * A)
        BX = (delta.unsqueeze(-1) * B.unsqueeze(1)) * x.unsqueeze(-1)
        if h is None:
            h = torch.zeros(x.size(0), self.config.d_inner, self.config.d_state, device=deltaA.device)
        h = deltaA * h + BX
        y = (h @ C.unsqueeze(-1)).squeeze(2) + self.D.float() * x
        return (y if z is None else y * F.silu(z)), h


class RMSNorm(nn.Module):
    """mamba.py:408-418."""

    def __init__(self, d_model: int, eps: float = 1e-5):
        super().__init__()
        self.eps = eps
        self.weight = nn.Parameter(torch.ones(d_model))

    def forward(self, x):
        return x * torch.rsqrt(x.pow(2).mean(-1, keepdim=True) + self.eps) * self.weight
