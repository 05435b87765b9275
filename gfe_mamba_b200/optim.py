"""Multi-tensor gradient clipping + Adam behind the C ABI (csrc/optim.cu, SURVEY 8f rank 3).

Host-side mirror of the reference training loop's tail (classify_mamba.py:64, 104-109)::

    optimizer = torch.optim.Adam(all_params, lr=1e-4)
    ...
    for param in all_params:
        torch.nn.utils.clip_grad_norm_(param, max_norm=1.0)
    optimizer.step()
    optimizer.zero_grad()

``ClipAdam(all_params, lr=1e-4, max_norm=1.0).step()`` does all of it in three kernel launches for the whole list,
whatever the number of parameter tensors, and is CUDA-graph capturable (the step counter lives on the device).

``state_dict()`` / ``load_state_dict()`` use torch.optim.Adam's format (``exp_avg``, ``exp_avg_sq`` and a float32 ``step`` per
parameter), so a run resumes with its moments and bias corrections, and the state dicts of the two optimisers load into each
other.
"""
from __future__ import annotations

import ctypes
from typing import Iterable, List, Optional, Tuple

import torch

from . import _native as nat


class ClipAdam(torch.optim.Optimizer):
    """Adam (torch.optim.Adam defaults: betas (0.9, 0.999), eps 1e-8, no weight decay, no amsgrad) with the gradient
    clipping of the reference loop fused in.

    max_norm            clip threshold; ``None`` or <= 0 disables clipping.
    per_parameter_clip  True: every tensor is clipped to ``max_norm`` on its own (the reference's loop over
                        ``clip_grad_norm_(param, ...)``); False: one norm over the whole list
                        (``clip_grad_norm_(all_params, ...)``).
    zero_grad           True: ``step`` leaves every gradient zeroed in place (the loop's ``optimizer.zero_grad()``, with
                        the buffers kept so that their addresses stay fixed for CUDA graphs); False: gradients are left
                        clipped, as after the reference's clip loop.
    """

    def __init__(self, params: Iterable, lr: float = 1e-3, betas: Tuple[float, float] = (0.9, 0.999), eps: float = 1e-8,
                 max_norm: Optional[float] = 1.0, per_parameter_clip: bool = True, zero_grad: bool = False):
        if lr < 0 or eps < 0 or not (0 <= betas[0] < 1) or not (0 <= betas[1] < 1):
            raise ValueError("ClipAdam: invalid hyper-parameters")
        defaults = dict(lr=lr, betas=betas, eps=eps, max_norm=max_norm, per_parameter_clip=per_parameter_clip,
                        zero_grad=zero_grad)
        super().__init__(params, defaults)
        self._tables = {}        # group index -> (key, table dict)
        self._loaded_steps = {}  # group index -> step counter loaded before the group's table existed

    def __setstate__(self, state):
        super().__setstate__(state)
        for group in self.param_groups:   # groups of a torch.optim.Adam state dict lack ClipAdam's own settings
            for k, v in self.defaults.items():
                group.setdefault(k, v)

    # ------------------------------------------------------------------------------------------------
    @staticmethod
    def plan_chunks(numels: List[int], chunk: int):
        """Chunk table of a tensor list: (chunk_tensor, chunk_start, tensor_chunk0).  Pure host logic."""
        chunk_tensor, chunk_start, tensor_chunk0 = [], [], [0]
        for t, n in enumerate(numels):
            for s in range(0, n, chunk):
                chunk_tensor.append(t)
                chunk_start.append(s)
            tensor_chunk0.append(len(chunk_tensor))
        return chunk_tensor, chunk_start, tensor_chunk0

    def _key(self, params: List[torch.Tensor]):
        """The addresses a table holds: parameters, gradients and -- so that a table never writes through the addresses of
        replaced state tensors -- the moment buffers."""
        return tuple((p.data_ptr(), p.grad.data_ptr(), p.numel(),
                      *(t.data_ptr() if t is not None else 0 for t in (self.state[p].get("exp_avg"), self.state[p].get("exp_avg_sq"))))
                     for p in params)

    def _table(self, gi: int, params: List[torch.Tensor]):
        key = self._key(params)
        cached = self._tables.get(gi)
        if cached is not None and cached[0] == key:
            return cached[1]
        dev = params[0].device
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("ClipAdam: the parameter/gradient tables must exist before a CUDA-graph capture (their upload and the "
                               "step counter's initialisation would be replayed): run one step with the same gradient buffers first")
        for p in params:
            if p.device != dev or p.dtype != torch.float32 or p.grad.dtype != torch.float32 \
                    or not p.is_contiguous() or not p.grad.is_contiguous():
                raise RuntimeError("ClipAdam: parameters and gradients must be contiguous fp32 CUDA tensors on one device")
            st = self.state[p]
            if "exp_avg" not in st:
                st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        key = self._key(params)   # with the moment buffers just created
        chunk = nat.lib().gfe_clip_adam_chunk_elems()
        numels = [p.numel() for p in params]
        ct, cs, tc0 = self.plan_chunks(numels, chunk)

        def dev_i64(v):
            return torch.tensor(v, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)

        tb = dict(
            p=dev_i64([p.data_ptr() for p in params]), g=dev_i64([p.grad.data_ptr() for p in params]),
            m=dev_i64([self.state[p]["exp_avg"].data_ptr() for p in params]),
            v=dev_i64([self.state[p]["exp_avg_sq"].data_ptr() for p in params]),
            numel=dev_i64(numels),
            chunk_tensor=torch.tensor(ct, dtype=torch.int32).pin_memory().to(dev, non_blocking=True),
            chunk_start=dev_i64(cs),
            tensor_chunk0=torch.tensor(tc0, dtype=torch.int32).pin_memory().to(dev, non_blocking=True),
            partial=torch.empty(max(len(ct), 1), dtype=torch.float32, device=dev),
            coef=torch.empty(len(params), dtype=torch.float32, device=dev),
            ntensors=len(params), nchunks=len(ct), dev=dev,
        )
        if gi in self._loaded_steps:
            tb["step"] = torch.full((1,), self._loaded_steps.pop(gi), dtype=torch.int32, device=dev)
        elif cached is not None:
            tb["step"] = cached[1]["step"]
        else:
            tb["step"] = torch.zeros(1, dtype=torch.int32, device=dev)
        self._tables[gi] = (key, tb)
        return tb

    def _group_step(self, gi: int) -> int:
        cached = self._tables.get(gi)
        if cached is not None:
            return int(cached[1]["step"].item())
        return self._loaded_steps.get(gi, 0)

    def state_dict(self):
        """torch.optim.Adam's layout: every parameter with state carries its group's step counter as a float32 CPU scalar
        ``step``, and every group ``weight_decay = 0`` (ClipAdam has none), so that torch.optim.Adam can load the dict."""
        sd = super().state_dict()
        for gi, g in enumerate(sd["param_groups"]):
            g.setdefault("weight_decay", 0.0)
            step = None
            for i in g["params"]:
                if i in sd["state"]:
                    if step is None:
                        step = torch.tensor(float(self._group_step(gi)), dtype=torch.float32)
                    sd["state"][i] = {**sd["state"][i], "step": step.clone()}   # a copy: the live state keeps no "step"
        return sd

    @torch.no_grad()
    def load_state_dict(self, state_dict):
        """Loads a ClipAdam or torch.optim.Adam state dict.  The moments are copied INTO the existing buffers and the device
        step counter is overwritten, so the device tables -- and a CUDA graph captured over ``step`` -- stay valid.  The
        parameters of one group share one step counter: a group whose parameters carry different steps raises ValueError.  A
        group without any saved ``step`` restarts its bias correction."""
        for g in state_dict["param_groups"]:
            if g.get("weight_decay", 0) or g.get("amsgrad", False) or g.get("maximize", False):
                raise ValueError("ClipAdam: weight decay, amsgrad and maximize are not supported")
        steps = []
        for g in state_dict["param_groups"]:
            vals = {float(state_dict["state"][i]["step"]) for i in g["params"] if "step" in state_dict["state"].get(i, {})}
            if len(vals) > 1:
                raise ValueError(f"ClipAdam: one step counter serves a whole parameter group, but its parameters carry the "
                                 f"steps {sorted(vals)}")
            steps.append(int(vals.pop()) if vals else 0)
        old = {p: (st["exp_avg"], st["exp_avg_sq"]) for p, st in self.state.items() if "exp_avg" in st}
        super().load_state_dict(state_dict)
        for p, (m, v) in old.items():
            st = self.state[p]
            for buf, new in ((m, st.get("exp_avg")), (v, st.get("exp_avg_sq"))):
                if new is None:
                    buf.zero_()
                elif new is not buf:
                    buf.copy_(new)
            self.state[p] = {"exp_avg": m, "exp_avg_sq": v}
        for st in self.state.values():
            st.pop("step", None)
        for gi, step in enumerate(steps):
            cached = self._tables.get(gi)
            if cached is not None:
                cached[1]["step"].fill_(step)
                self._loaded_steps.pop(gi, None)
            else:
                self._loaded_steps[gi] = step

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        l = nat.lib()
        for gi, group in enumerate(self.param_groups):
            params = [p for p in group["params"] if p.grad is not None]
            if not params:
                continue
            if not params[0].is_cuda:
                raise RuntimeError("gfe_mamba_b200.ClipAdam: CUDA tensors required (this library has no CPU fallback)")
            tb = self._table(gi, params)
            dev = tb["dev"]
            mx = group["max_norm"]
            with torch.cuda.device(dev):
                nat.check(l.gfe_clip_adam_step(
                    *(ctypes.c_void_p(tb[k].data_ptr()) for k in ("p", "g", "m", "v", "numel", "chunk_tensor", "chunk_start",
                                                                  "tensor_chunk0", "partial", "coef", "step")),
                    tb["ntensors"], tb["nchunks"], float(group["lr"]), float(group["betas"][0]), float(group["betas"][1]),
                    float(group["eps"]), float(mx) if mx else 0.0, 0 if group["per_parameter_clip"] else 1,
                    1 if group["zero_grad"] else 0, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "clip_adam_step")
        return loss

    def zero_grad(self, set_to_none: bool = False):
        """Keeps the gradient buffers (fixed addresses) unless ``set_to_none`` is asked for explicitly; a no-op after a
        ``step`` with ``zero_grad=True``."""
        if set_to_none:
            return super().zero_grad(set_to_none=True)
        if all(g["zero_grad"] for g in self.param_groups) and self._tables:
            return
        return super().zero_grad(set_to_none=False)
