"""torch.autograd wrappers around the C ABI (include/gfe_mamba_b200.h).

PyTorch is plumbing here: it owns device memory, streams and autograd bookkeeping; every number is
produced by the sm_100a kernels in csrc/.  CPU tensors are rejected -- there is no fallback path.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _native as nat

_DT = {torch.float32: nat.GFE_F32, torch.bfloat16: nat.GFE_BF16, torch.float16: nat.GFE_F16}

# d_state values the fused scan, the one-node inner path and the decode kernel are compiled for (fused_d_state in
# csrc/common.cuh); MambaBlock takes the reference's composition on top of the pscan kernel for every other value
FUSED_D_STATES = (16, 32, 64)


def _require_cuda(*ts: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("gfe_mamba_b200: CUDA tensors required (this library has no CPU fallback); "
                               f"got a tensor on {t.device}")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"gfe_mamba_b200: tensors on different devices ({dev} vs {t.device})")
    return dev


def _ptr(t: Optional[torch.Tensor]) -> ctypes.c_void_p:
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream(dev: torch.device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _bytes(n: int, dev: torch.device) -> Optional[torch.Tensor]:
    return torch.empty(n, dtype=torch.uint8, device=dev) if n > 0 else None


def _rows(t: torch.Tensor) -> torch.Tensor:
    """(B, L, C) with unit channel stride; batch/row strides are passed to the kernels as they are."""
    return t if t.stride(-1) == 1 else t.contiguous()


_SIZE_CACHE = {}


def _sizes(B: int, L: int, ED: int, N: int, dev: torch.device, dtype: int):
    """(ckpt, fwd workspace, bwd workspace) bytes of one shape ON ONE DEVICE (the launch plan depends on the device's
    SM count, so the key carries the device); asked once.  Call with ``dev`` current."""
    key = (B, L, ED, N, dev.index, dtype)
    v = _SIZE_CACHE.get(key)
    if v is None:
        l = nat.lib()
        v = (l.gfe_selscan_ckpt_bytes_dt(B, L, ED, N, dtype), l.gfe_selscan_fwd_workspace_bytes(B, L, ED, N),
             l.gfe_selscan_bwd_workspace_bytes(B, L, ED, N))
        _SIZE_CACHE[key] = v
    return v


def _as(t: torch.Tensor, dt: torch.dtype) -> torch.Tensor:
    """detach + dtype + unit channel stride, touching the tensor only when something has to change."""
    t = t.detach()
    if t.dtype != dt:
        t = t.to(dt)
    return t if t.stride(-1) == 1 else t.contiguous()


def _f32(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------------------------------ pscan
class _PScanFn(torch.autograd.Function):
    """pscan(A, X) -- cross_atten/pscan.py:152-224 (PScan.forward / PScan.backward)."""

    @staticmethod
    def forward(ctx, A_in: torch.Tensor, X_in: torch.Tensor) -> torch.Tensor:
        dev = _require_cuda(A_in, X_in)
        if A_in.dim() != 4 or A_in.shape != X_in.shape:
            raise ValueError(f"pscan expects A, X of identical shape (B, L, D, N); got {tuple(A_in.shape)}, {tuple(X_in.shape)}")
        A = A_in.detach().float().contiguous()
        X = X_in.detach().float().contiguous()
        B, L, D, N = A.shape
        H = torch.empty_like(X)
        l = nat.lib()
        with torch.cuda.device(dev):
            nws = l.gfe_pscan_workspace_bytes(B, L, D, N)
            ws = _bytes(nws, dev)
            nat.check(l.gfe_pscan_fwd(_ptr(A), _ptr(X), _ptr(H), B, L, D, N, _ptr(ws), nws, _stream(dev)), "pscan_fwd")
        ctx.save_for_backward(A, H)
        ctx.in_dtypes = (A_in.dtype, X_in.dtype)
        return H if X_in.dtype == torch.float32 else H.to(X_in.dtype)

    @staticmethod
    def backward(ctx, dH_in: torch.Tensor):
        A, H = ctx.saved_tensors
        dev = A.device
        dH = dH_in.detach().float().contiguous()
        B, L, D, N = A.shape
        dA, dX = torch.empty_like(A), torch.empty_like(A)
        l = nat.lib()
        with torch.cuda.device(dev):
            nws = l.gfe_pscan_workspace_bytes(B, L, D, N)
            ws = _bytes(nws, dev)
            nat.check(l.gfe_pscan_bwd(_ptr(A), _ptr(H), _ptr(dH), _ptr(dA), _ptr(dX), B, L, D, N, _ptr(ws), nws, _stream(dev)),
                      "pscan_bwd")
        return dA.to(ctx.in_dtypes[0]), dX.to(ctx.in_dtypes[1])


def pscan(A: torch.Tensor, X: torch.Tensor) -> torch.Tensor:
    """H[t] = A[t] * H[t-1] + X[t] over dim 1 of (B, L, D, N) tensors; differentiable in both arguments."""
    return _PScanFn.apply(A, X)


# ------------------------------------------------------------------------------- selective scan
def _fill_common(a: nat.SelscanArgs, u, delta, z, Bm, Cm, A_log, D, dt_bias, softplus: bool):
    B, L, ED = u.shape
    a.batch, a.seqlen, a.d_inner, a.d_state = B, L, ED, A_log.shape[1]
    a.dtype = _DT[u.dtype]
    a.flags = nat.GFE_FLAG_DELTA_SOFTPLUS if softplus else 0
    a.u, a.u_bs, a.u_rs = u.data_ptr(), u.stride(0), u.stride(1)
    a.delta, a.delta_bs, a.delta_rs = delta.data_ptr(), delta.stride(0), delta.stride(1)
    if z is not None:
        a.z, a.z_bs, a.z_rs = z.data_ptr(), z.stride(0), z.stride(1)
    a.Bm, a.B_bs, a.B_rs = Bm.data_ptr(), Bm.stride(0), Bm.stride(1)
    a.Cm, a.C_bs, a.C_rs = Cm.data_ptr(), Cm.stride(0), Cm.stride(1)
    a.A_log, a.D = A_log.data_ptr(), D.data_ptr()
    a.dt_bias = 0 if dt_bias is None else dt_bias.data_ptr()


class _SelectiveScanFn(torch.autograd.Function):
    """Fused MambaBlock.ssm tail: softplus(delta + bias) -> discretise -> scan -> C contraction -> D skip -> * silu(z)
    (cross_atten/mamba.py:255-256, 265-286, 220-222; the contract of the selective_scan_fn call at mamba.py:251)."""

    @staticmethod
    def forward(ctx, u, delta, A_log, Bm, Cm, D, z, dt_bias, softplus: bool, return_last_state: bool, grad_mode: bool):
        dev = _require_cuda(u, delta, A_log, Bm, Cm, D, z, dt_bias)
        if u.dim() != 3:
            raise ValueError(f"selective_scan: u must be (B, L, ED); got {tuple(u.shape)}")
        B, L, ED = u.shape
        N = A_log.shape[1]
        if u.dtype not in _DT:
            raise TypeError(f"selective_scan: unsupported activation dtype {u.dtype}")
        if tuple(delta.shape) != (B, L, ED) or tuple(Bm.shape) != (B, L, N) or tuple(Cm.shape) != (B, L, N) \
                or tuple(A_log.shape) != (ED, N) or tuple(D.shape) != (ED,):
            raise ValueError("selective_scan: inconsistent shapes")
        dt = u.dtype
        u_, delta_, Bm_, Cm_ = (_as(t, dt) for t in (u, delta, Bm, Cm))
        z_ = None if z is None else _as(z, dt)
        A_log_, D_, bias_ = _f32(A_log), _f32(D), _f32(dt_bias)
        out = torch.empty((B, L, ED), dtype=dt, device=dev)
        last = torch.empty((B, ED, N), dtype=torch.float32, device=dev) if return_last_state else None
        # needs_input_grad mirrors requires_grad and ignores the grad mode: under no_grad / eval with trainable parameters
        # nothing is checkpointed (the checkpoint stream is larger than the forward's own traffic)
        need_grad = grad_mode and any(ctx.needs_input_grad)
        l = nat.lib()
        a = nat.SelscanArgs()
        _fill_common(a, u_, delta_, z_, Bm_, Cm_, A_log_, D_, bias_, softplus)
        a.out, a.out_bs, a.out_rs = out.data_ptr(), out.stride(0), out.stride(1)
        a.last_state = 0 if last is None else last.data_ptr()
        with torch.cuda.device(dev):
            sz = _sizes(B, L, ED, N, dev, _DT[dt])
            nck = sz[0] if need_grad else 0
            ckpt = _bytes(nck, dev)
            nws = sz[1]
            ws = _bytes(nws, dev)
            a.ckpt, a.ckpt_bytes = (0 if ckpt is None else ckpt.data_ptr()), nck
            a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), nws
            nat.check(l.gfe_selscan_fwd(ctypes.byref(a), _stream(dev)), "selscan_fwd")
        if need_grad:
            ctx.save_for_backward(u_, delta_, A_log_, Bm_, Cm_, D_, z_, bias_, ckpt)
            ctx.softplus = softplus
            ctx.in_dtypes = tuple(None if t is None else t.dtype for t in (u, delta, A_log, Bm, Cm, D, z, dt_bias))
        if return_last_state:
            ctx.mark_non_differentiable(last)
            return out, last
        return out

    @staticmethod
    def backward(ctx, dout, *unused):
        u, delta, A_log, Bm, Cm, D, z, bias, ckpt = ctx.saved_tensors
        dev = u.device
        B, L, ED = u.shape
        N = A_log.shape[1]
        dt = u.dtype
        dout = _as(dout, dt)
        du = torch.empty((B, L, ED), dtype=dt, device=dev)
        ddelta = torch.empty((B, L, ED), dtype=dt, device=dev)
        dz = None if z is None else torch.empty((B, L, ED), dtype=dt, device=dev)
        dBm = torch.empty((B, L, N), dtype=dt, device=dev)
        dCm = torch.empty((B, L, N), dtype=dt, device=dev)
        dA_log = torch.empty((ED, N), dtype=torch.float32, device=dev)
        dD = torch.empty((ED,), dtype=torch.float32, device=dev)
        dbias = None if bias is None else torch.empty((ED,), dtype=torch.float32, device=dev)
        l = nat.lib()
        a = nat.SelscanArgs()
        _fill_common(a, u, delta, z, Bm, Cm, A_log, D, bias, ctx.softplus)
        a.ckpt, a.ckpt_bytes = ckpt.data_ptr(), ckpt.numel()
        a.dout, a.dout_bs, a.dout_rs = dout.data_ptr(), dout.stride(0), dout.stride(1)
        a.du, a.du_bs, a.du_rs = du.data_ptr(), du.stride(0), du.stride(1)
        a.ddelta, a.ddelta_bs, a.ddelta_rs = ddelta.data_ptr(), ddelta.stride(0), ddelta.stride(1)
        if dz is not None:
            a.dz, a.dz_bs, a.dz_rs = dz.data_ptr(), dz.stride(0), dz.stride(1)
        a.dBm, a.dB_bs, a.dB_rs = dBm.data_ptr(), dBm.stride(0), dBm.stride(1)
        a.dCm, a.dC_bs, a.dC_rs = dCm.data_ptr(), dCm.stride(0), dCm.stride(1)
        a.dA_log, a.dD = dA_log.data_ptr(), dD.data_ptr()
        a.ddt_bias = 0 if dbias is None else dbias.data_ptr()
        with torch.cuda.device(dev):
            nws = _sizes(B, L, ED, N, dev, _DT[dt])[2]
            ws = _bytes(nws, dev)
            a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), nws
            nat.check(l.gfe_selscan_bwd(ctypes.byref(a), _stream(dev)), "selscan_bwd")
        dts = ctx.in_dtypes

        def cast(g, i):
            return None if (g is None or dts[i] is None) else (g if g.dtype == dts[i] else g.to(dts[i]))

        return (cast(du, 0), cast(ddelta, 1), cast(dA_log, 2), cast(dBm, 3), cast(dCm, 4), cast(dD, 5),
                cast(dz, 6), cast(dbias, 7), None, None, None)


def selective_scan_fn(u: torch.Tensor, delta: torch.Tensor, A_log: torch.Tensor, Bm: torch.Tensor, Cm: torch.Tensor,
                      D: torch.Tensor, z: Optional[torch.Tensor] = None, dt_bias: Optional[torch.Tensor] = None,
                      delta_softplus: bool = True, return_last_state: bool = False):
    """Fused selective scan, channel-last.

    u, delta, z: (B, L, ED) (any batch/row strides, unit channel stride); Bm, Cm: (B, L, N); A_log: (ED, N);
    D, dt_bias: (ED).  Returns out (B, L, ED) in u's dtype:
        delta' = softplus(delta + dt_bias);  h_t = exp(delta' A) h_{t-1} + delta' B_t u_t,  A = -exp(A_log)
        out_t  = (C_t . h_t + D u_t) * silu(z_t)
    """
    return _SelectiveScanFn.apply(u, delta, A_log, Bm, Cm, D, z, dt_bias, bool(delta_softplus), bool(return_last_state),
                                  torch.is_grad_enabled())


# ----------------------------------------------------------------------- causal conv1d + SiLU
class _CausalConv1dSiluFn(torch.autograd.Function):
    """silu(Conv1d(groups=ED, k=K, padding=K-1)(x^T)[:, :, :L]^T) -- cross_atten/mamba.py:128-131, 208-212."""

    @staticmethod
    def forward(ctx, xin, weight, bias):
        dev = _require_cuda(xin, weight, bias)
        if xin.dim() != 3:
            raise ValueError(f"causal_conv1d_silu: x must be (B, L, ED); got {tuple(xin.shape)}")
        B, L, ED = xin.shape
        K = weight.shape[-1]
        if weight.numel() != ED * K:
            raise ValueError("causal_conv1d_silu: weight must be (ED, 1, K) / (ED, K)")
        x_ = _rows(xin.detach())
        w_ = weight.detach().float().reshape(ED, K).contiguous()
        b_ = _f32(bias)
        u = torch.empty((B, L, ED), dtype=xin.dtype, device=dev)
        l = nat.lib()
        with torch.cuda.device(dev):
            nat.check(l.gfe_conv1d_silu_fwd(_ptr(x_), x_.stride(0), x_.stride(1), _ptr(w_), _ptr(b_), _ptr(u), u.stride(0),
                                            u.stride(1), B, L, ED, K, _DT[xin.dtype], _stream(dev)), "conv1d_silu_fwd")
        ctx.save_for_backward(x_, w_, b_)
        ctx.meta = (weight.shape, weight.dtype, None if bias is None else bias.dtype)
        return u

    @staticmethod
    def backward(ctx, du):
        x_, w_, b_ = ctx.saved_tensors
        dev = x_.device
        B, L, ED = x_.shape
        K = w_.shape[1]
        du = _rows(du.detach().to(x_.dtype))
        dx = torch.empty((B, L, ED), dtype=x_.dtype, device=dev)
        dw = torch.empty((ED, K), dtype=torch.float32, device=dev)
        db = None if b_ is None else torch.empty((ED,), dtype=torch.float32, device=dev)
        l = nat.lib()
        with torch.cuda.device(dev):
            nws = l.gfe_conv1d_bwd_workspace_bytes(B, L, ED, K)
            ws = _bytes(nws, dev)
            nat.check(l.gfe_conv1d_silu_bwd(_ptr(x_), x_.stride(0), x_.stride(1), _ptr(w_), _ptr(b_), _ptr(du), du.stride(0),
                                            du.stride(1), _ptr(dx), dx.stride(0), dx.stride(1), _ptr(dw), _ptr(db),
                                            B, L, ED, K, _DT[x_.dtype], _ptr(ws), nws, _stream(dev)), "conv1d_silu_bwd")
        wshape, wdt, bdt = ctx.meta
        return dx, dw.reshape(wshape).to(wdt), (None if db is None else db.to(bdt))


def causal_conv1d_silu(xin: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor]) -> torch.Tensor:
    """Channel-last causal depthwise conv + bias + SiLU.  xin: (B, L, ED), weight: (ED, 1, K), bias: (ED) or None."""
    return _CausalConv1dSiluFn.apply(xin, weight, bias)


# ------------------------------------------------ conv -> x_proj -> dt_proj -> scan as ONE autograd node
class _MambaInnerFn(torch.autograd.Function):
    """MambaBlock.forward between in_proj and out_proj (cross_atten/mamba.py:204-223: split, conv1d + SiLU, x_proj, split,
    dt_proj, selective scan, gate) as one autograd node.  The kernels are the ones behind causal_conv1d_silu and
    selective_scan_fn; what the node removes is torch glue between them (SURVEY 8f rank 2):
      * the u|z halves of in_proj's output and the delta|B|C slices of x_proj's output are consumed in place (as before), and in
        backward their gradients are WRITTEN in place -- dz and d(conv input) into the two halves of one (B, L, 2 ED) tensor,
        dB / dC into the slices of one (B L, R + 2 N) tensor -- instead of being concatenated by autograd's split backward
        (a zero-fill plus two copies of 2 ED columns per token);
      * the two gradients that flow into the conv output (from the scan and from x_proj) meet in the GEMM epilogue
        (addmm_ with beta = 1) instead of a separate elementwise add over (B, L, ED).
    """

    @staticmethod
    def forward(ctx, xz, conv_w, conv_b, x_proj_w, dt_proj_w, dt_bias, A_log, D, grad_mode: bool):
        dev = _require_cuda(xz, conv_w, conv_b, x_proj_w, dt_proj_w, dt_bias, A_log, D)
        B, L, ED2 = xz.shape
        ED, N = A_log.shape
        K = conv_w.shape[-1]
        R = dt_proj_w.shape[1]
        dt = xz.dtype
        if ED2 != 2 * ED or tuple(x_proj_w.shape) != (R + 2 * N, ED) or tuple(dt_proj_w.shape) != (ED, R) or dt not in _DT:
            raise ValueError("mamba_inner: inconsistent shapes / dtype")
        xz_ = _rows(xz.detach())
        xin, z = xz_[..., :ED], xz_[..., ED:]
        cw = conv_w.detach().float().reshape(ED, K).contiguous()
        cb = _f32(conv_b)
        Wx, Wdt = x_proj_w.detach().to(dt), dt_proj_w.detach().to(dt)
        A_log_, D_, bias_ = _f32(A_log), _f32(D), _f32(dt_bias)
        need_grad = grad_mode and any(ctx.needs_input_grad)
        l = nat.lib()
        u = torch.empty((B, L, ED), dtype=dt, device=dev)
        out = torch.empty((B, L, ED), dtype=dt, device=dev)
        # the GEMMs run in the activation dtype chosen above whatever the ambient autocast state (the kernels need one dtype)
        with torch.cuda.device(dev), torch.autocast("cuda", enabled=False):
            nat.check(l.gfe_conv1d_silu_fwd(_ptr(xin), xin.stride(0), xin.stride(1), _ptr(cw), _ptr(cb), _ptr(u), u.stride(0),
                                            u.stride(1), B, L, ED, K, _DT[dt], _stream(dev)), "conv1d_silu_fwd")
            dbc = torch.mm(u.view(B * L, ED), Wx.t())                 # (B L, R + 2N): delta_low | B | C
            delta = torch.mm(dbc[:, :R], Wdt.t()).view(B, L, ED)      # dt_proj without its bias (added inside the scan)
            dbc3 = dbc.view(B, L, R + 2 * N)
            Bm, Cm = dbc3[..., R:R + N], dbc3[..., R + N:]
            a = nat.SelscanArgs()
            _fill_common(a, u, delta, z, Bm, Cm, A_log_, D_, bias_, True)
            a.out, a.out_bs, a.out_rs = out.data_ptr(), out.stride(0), out.stride(1)
            sz = _sizes(B, L, ED, N, dev, _DT[dt])
            nck = sz[0] if need_grad else 0
            ckpt = _bytes(nck, dev)
            ws = _bytes(sz[1], dev)
            a.ckpt, a.ckpt_bytes = (0 if ckpt is None else ckpt.data_ptr()), nck
            a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), sz[1]
            nat.check(l.gfe_selscan_fwd(ctypes.byref(a), _stream(dev)), "selscan_fwd")
        if need_grad:
            ctx.save_for_backward(xz_, cw, cb, x_proj_w, dt_proj_w, A_log_, D_, bias_, u, dbc, delta, ckpt)
            ctx.meta = (conv_w.shape, conv_w.dtype, None if conv_b is None else conv_b.dtype, x_proj_w.dtype, dt_proj_w.dtype,
                        None if dt_bias is None else dt_bias.dtype, A_log.dtype, D.dtype)
        return out

    @staticmethod
    def backward(ctx, dout):
        xz_, cw, cb, x_proj_w, dt_proj_w, A_log_, D_, bias_, u, dbc, delta, ckpt = ctx.saved_tensors
        dev = xz_.device
        B, L, ED2 = xz_.shape
        ED, N = A_log_.shape
        K = cw.shape[1]
        R = dt_proj_w.shape[1]
        dt = xz_.dtype
        dout = _as(dout, dt)
        xin, z = xz_[..., :ED], xz_[..., ED:]
        Wx, Wdt = x_proj_w.detach().to(dt), dt_proj_w.detach().to(dt)
        dxz = torch.empty((B, L, 2 * ED), dtype=dt, device=dev)
        dxin, dz = dxz[..., :ED], dxz[..., ED:]
        ddbc = torch.empty((B * L, R + 2 * N), dtype=dt, device=dev)
        ddbc3 = ddbc.view(B, L, R + 2 * N)
        dBm, dCm = ddbc3[..., R:R + N], ddbc3[..., R + N:]
        du = torch.empty((B, L, ED), dtype=dt, device=dev)
        ddelta = torch.empty((B, L, ED), dtype=dt, device=dev)
        dA_log = torch.empty((ED, N), dtype=torch.float32, device=dev)
        dD = torch.empty((ED,), dtype=torch.float32, device=dev)
        dbias = None if bias_ is None else torch.empty((ED,), dtype=torch.float32, device=dev)
        dcw = torch.empty((ED, K), dtype=torch.float32, device=dev)
        dcb = None if cb is None else torch.empty((ED,), dtype=torch.float32, device=dev)
        dbc3 = dbc.view(B, L, R + 2 * N)
        l = nat.lib()
        with torch.cuda.device(dev), torch.autocast("cuda", enabled=False):
            a = nat.SelscanArgs()
            _fill_common(a, u, delta, z, dbc3[..., R:R + N], dbc3[..., R + N:], A_log_, D_, bias_, True)
            a.ckpt, a.ckpt_bytes = ckpt.data_ptr(), ckpt.numel()
            a.dout, a.dout_bs, a.dout_rs = dout.data_ptr(), dout.stride(0), dout.stride(1)
            a.du, a.du_bs, a.du_rs = du.data_ptr(), du.stride(0), du.stride(1)
            a.ddelta, a.ddelta_bs, a.ddelta_rs = ddelta.data_ptr(), ddelta.stride(0), ddelta.stride(1)
            a.dz, a.dz_bs, a.dz_rs = dz.data_ptr(), dz.stride(0), dz.stride(1)
            a.dBm, a.dB_bs, a.dB_rs = dBm.data_ptr(), dBm.stride(0), dBm.stride(1)
            a.dCm, a.dC_bs, a.dC_rs = dCm.data_ptr(), dCm.stride(0), dCm.stride(1)
            a.dA_log, a.dD = dA_log.data_ptr(), dD.data_ptr()
            a.ddt_bias = 0 if dbias is None else dbias.data_ptr()
            nws = _sizes(B, L, ED, N, dev, _DT[dt])[2]
            ws = _bytes(nws, dev)
            a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), nws
            nat.check(l.gfe_selscan_bwd(ctypes.byref(a), _stream(dev)), "selscan_bwd")
            # dt_proj: d delta_low into its slice of d(dbc); weight gradient
            dd2 = ddelta.view(B * L, ED)
            ddbc[:, :R] = torch.mm(dd2, Wdt)
            dWdt = torch.mm(dd2.t(), dbc[:, :R])
            # x_proj: its input gradient lands on top of the scan's du in the GEMM epilogue; weight gradient
            du2 = du.view(B * L, ED)
            du2.addmm_(ddbc, Wx)
            dWx = torch.mm(ddbc.t(), u.view(B * L, ED))
            # conv + SiLU: d(conv input) straight into the first half of d(xz)
            nws = l.gfe_conv1d_bwd_workspace_bytes(B, L, ED, K)
            ws = _bytes(nws, dev)
            nat.check(l.gfe_conv1d_silu_bwd(_ptr(xin), xin.stride(0), xin.stride(1), _ptr(cw), _ptr(cb), _ptr(du), du.stride(0),
                                            du.stride(1), _ptr(dxin), dxin.stride(0), dxin.stride(1), _ptr(dcw), _ptr(dcb),
                                            B, L, ED, K, _DT[dt], _ptr(ws), nws, _stream(dev)), "conv1d_silu_bwd")
        cw_shape, cw_dt, cb_dt, wx_dt, wdt_dt, bias_dt, alog_dt, d_dt = ctx.meta
        return (dxz, dcw.reshape(cw_shape).to(cw_dt), None if dcb is None else dcb.to(cb_dt), dWx.to(wx_dt), dWdt.to(wdt_dt),
                None if dbias is None else dbias.to(bias_dt), dA_log.to(alog_dt), dD.to(d_dt), None)


def mamba_inner_fn(xz: torch.Tensor, conv_w: torch.Tensor, conv_b: Optional[torch.Tensor], x_proj_w: torch.Tensor,
                   dt_proj_w: torch.Tensor, dt_bias: Optional[torch.Tensor], A_log: torch.Tensor, D: torch.Tensor) -> torch.Tensor:
    """y (B, L, ED) = gate(scan(conv(xz[..., :ED]), ...), xz[..., ED:]) for d_state in FUSED_D_STATES, d_conv in 2..4; see
    _MambaInnerFn."""
    return _MambaInnerFn.apply(xz, conv_w, conv_b, x_proj_w, dt_proj_w, dt_bias, A_log, D, torch.is_grad_enabled())


# ----------------------------------------------------------------- residual add + RMSNorm
class _AddRMSNormFn(torch.autograd.Function):
    """resid = x (+ a);  y = (resid * rsqrt(mean(resid^2) + eps)) * w -- the residual add of ResidualBlock.forward
    (cross_atten/mamba.py:103) fused with the next RMSNorm (mamba.py:408-418).  SURVEY 8f rank 1.

    Two element types: the residual stream (x, resid and their gradients) keeps x's dtype; the branch side (a, y and their
    gradients) may be 16-bit next to an fp32 stream -- the stack under autocast -- so that neither the mixer's 16-bit output
    nor the normed input of the next mixer passes through a cast kernel."""

    @staticmethod
    def forward(ctx, x, a, weight, eps: float, grad_mode: bool, io_dtype):
        dev = _require_cuda(x, a, weight)
        if x.dtype not in _DT:
            raise TypeError(f"add_rmsnorm: unsupported activation dtype {x.dtype}")
        D = x.shape[-1]
        if weight.shape != (D,) or (a is not None and a.shape != x.shape):
            raise ValueError("add_rmsnorm: inconsistent shapes")
        if io_dtype != x.dtype and not (x.dtype == torch.float32 and io_dtype in (torch.bfloat16, torch.float16)):
            raise TypeError(f"add_rmsnorm: stream {x.dtype} with branch {io_dtype} is not supported")
        x_ = x.detach().contiguous()
        a_ = None if a is None else a.detach().to(io_dtype).contiguous()
        w_ = _f32(weight)
        rows = x_.numel() // D
        resid = torch.empty_like(x_) if a_ is not None else x_
        y = torch.empty(x_.shape, dtype=io_dtype, device=dev)
        need_grad = grad_mode and any(ctx.needs_input_grad)
        rstd = torch.empty(rows, dtype=torch.float32, device=dev) if need_grad else None
        l = nat.lib()
        with torch.cuda.device(dev):
            nat.check(l.gfe_add_rmsnorm_fwd_mixed(_ptr(x_), _ptr(a_), _ptr(w_), _ptr(resid if a_ is not None else None), _ptr(y),
                                                  _ptr(rstd), rows, D, float(eps), _DT[x.dtype], _DT[io_dtype], _stream(dev)),
                      "add_rmsnorm_fwd")
        # an output nothing downstream used arrives in backward as None, not as a zero-filled (rows, D) tensor: an unused
        # resid runs the kernels without the dres stream, an unused y reads zeros
        ctx.set_materialize_grads(False)
        if need_grad:
            ctx.save_for_backward(resid, w_, rstd)
            ctx.a_dtype = None if a is None else a.dtype
            ctx.io_dtype = io_dtype
            ctx.wdtype = weight.dtype
        return resid, y

    @staticmethod
    def backward(ctx, dresid, dy):
        resid, w_, rstd = ctx.saved_tensors
        dev = resid.device
        D = resid.shape[-1]
        rows = resid.numel() // D
        io = ctx.io_dtype
        dy_ = torch.zeros(resid.shape, dtype=io, device=dev) if dy is None else dy.detach().to(io).contiguous()
        dres_ = None if dresid is None else dresid.detach().to(resid.dtype).contiguous()
        dx = torch.empty_like(resid)
        # the branch operand's gradient in ITS dtype comes out of the same pass when that dtype differs from the stream's
        da = torch.empty(resid.shape, dtype=io, device=dev) if (ctx.a_dtype is not None and io != resid.dtype) else None
        dw = torch.empty(D, dtype=torch.float32, device=dev)
        l = nat.lib()
        with torch.cuda.device(dev):
            nws = l.gfe_add_rmsnorm_bwd_workspace_bytes(rows, D)
            ws = _bytes(nws, dev)
            nat.check(l.gfe_add_rmsnorm_bwd_mixed(_ptr(resid), _ptr(w_), _ptr(rstd), _ptr(dy_), _ptr(dres_), _ptr(dx), _ptr(da),
                                                  _ptr(dw), rows, D, _DT[resid.dtype], _DT[io], _ptr(ws), nws, _stream(dev)),
                      "add_rmsnorm_bwd")
        if ctx.a_dtype is None:
            ga = None
        elif da is not None:
            ga = da if ctx.a_dtype == io else da.to(ctx.a_dtype)
        else:
            ga = dx if ctx.a_dtype == dx.dtype else dx.to(ctx.a_dtype)
        return dx, ga, dw.to(ctx.wdtype), None, None, None


def add_rmsnorm(x: torch.Tensor, a: Optional[torch.Tensor], weight: torch.Tensor, eps: float = 1e-5,
                out_dtype: Optional[torch.dtype] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Returns (resid, y): resid = x + a (or x itself when a is None) in x's dtype, y = RMSNorm(resid) * weight.  x, a: (..., D).

    ``out_dtype`` is the dtype of ``y`` (and the dtype ``a`` is read in).  By default it is x's dtype, except for an fp32
    stream under CUDA autocast whose branch ``a`` is absent or already in the autocast dtype: then ``y`` comes out in that
    dtype -- what the next ``nn.Linear`` would cast it to anyway (same rounding of the same fp32 value) -- and ``a`` is
    consumed as it is."""
    if out_dtype is None:
        out_dtype = x.dtype
        if x.dtype == torch.float32 and x.is_cuda and torch.is_autocast_enabled("cuda"):
            ad = torch.get_autocast_dtype("cuda")
            if ad in (torch.bfloat16, torch.float16) and (a is None or a.dtype == ad):
                out_dtype = ad
    return _AddRMSNormFn.apply(x, a, weight, eps, torch.is_grad_enabled(), out_dtype)


# --------------------------------------------------------- final residual add + mean over L
class _AddMeanPoolFn(torch.autograd.Function):
    """mean over dim 1 of (a + r) -- the last residual add of the stack (cross_atten/mamba.py:103) fused with the head's
    pooling (cross_atten/mamba_transformer.py:123).  SURVEY 8f rank 4.

    a and r may differ in dtype as torch allows: fp32 next to bf16 / fp16, in either order (the stack under autocast: a 16-bit
    last branch on the fp32 residual stream).  Each operand is read in its own dtype, the output is fp32 like ``a + r`` in torch,
    and each operand's gradient comes out in its own dtype from one backward pass."""

    @staticmethod
    def forward(ctx, a, r):
        dev = _require_cuda(a, r)
        if a.dim() != 3 or (r is not None and r.shape != a.shape):
            raise ValueError("add_mean_pool: (B, L, D) operands of identical shape expected")
        rdt = a.dtype if r is None else r.dtype
        if a.dtype not in _DT or rdt not in _DT:
            raise TypeError(f"add_mean_pool: unsupported dtype {a.dtype if a.dtype not in _DT else rdt}")
        if rdt != a.dtype and torch.float32 not in (a.dtype, rdt):
            raise TypeError(f"add_mean_pool: operands in {a.dtype} and {rdt}: only fp32 may meet a 16-bit dtype")
        out_dt = torch.promote_types(a.dtype, rdt)
        B, L, D = a.shape
        a_ = a.detach().contiguous()
        r_ = None if r is None else r.detach().contiguous()
        out = torch.empty((B, 1, D), dtype=out_dt, device=dev)
        l = nat.lib()
        with torch.cuda.device(dev):
            nws = l.gfe_add_mean_pool_workspace_bytes(B, L, D)
            ws = _bytes(nws, dev)
            nat.check(l.gfe_add_mean_pool_fwd_mixed(_ptr(a_), _ptr(r_), _ptr(out), B, L, D, _DT[a.dtype], _DT[rdt], _ptr(ws), nws,
                                                    _stream(dev)), "add_mean_pool_fwd")
        ctx.shape, ctx.has_r, ctx.dtypes = (B, L, D), r is not None, (a.dtype, rdt, out_dt)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, L, D = ctx.shape
        adt, rdt, out_dt = ctx.dtypes
        dev = dout.device
        d_ = dout.detach().to(out_dt).contiguous()
        da = torch.empty((B, L, D), dtype=adt, device=dev)
        # equal dtypes: both operands share one gradient tensor; else r's own, written by the same pass
        dr = torch.empty((B, L, D), dtype=rdt, device=dev) if (ctx.has_r and rdt != adt and ctx.needs_input_grad[1]) else None
        l = nat.lib()
        with torch.cuda.device(dev):
            nat.check(l.gfe_mean_pool_bwd_mixed(_ptr(d_), _ptr(da), _ptr(dr), B, L, D, _DT[adt], _DT[rdt], _stream(dev)),
                      "mean_pool_bwd")
        if not ctx.has_r:
            return da, None
        return da, (dr if rdt != adt else da)


def add_mean_pool(a: torch.Tensor, r: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B, 1, D) = mean over L of (a + r); a, r: (B, L, D).  Equals ``torch.mean(a + r, dim=1, keepdim=True)``, dtype included:
    fp32 with bf16 / fp16 gives fp32; other dtype mixes raise TypeError."""
    return _AddMeanPoolFn.apply(a, r)


# ------------------------------------------------------------------------------- decode step
def _no_autograd(name: str, *ts):
    """The decode and prefill kernels have no backward: refuse to silently detach a graph (MambaBlock.step / .prefill fall
    back to the reference's differentiable torch composition in that case)."""
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts):
        raise RuntimeError(f"gfe_mamba_b200.{name}: inputs require grad but the decode kernels are inference-only; "
                           "call under torch.no_grad() or use MambaBlock.step, which falls back to torch ops")


def conv1d_step(xin: torch.Tensor, inputs: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor]
                ) -> Tuple[torch.Tensor, torch.Tensor]:
    """One token of the causal conv (mamba.py:357-358, 370).  xin: (B, ED); inputs: (B, ED, K-1).
    Returns (u, new_inputs); ``inputs`` is not modified."""
    dev = _require_cuda(xin, inputs, weight, bias)
    _no_autograd("conv1d_step", xin, inputs, weight, bias)
    xin, inputs, weight = xin.detach(), inputs.detach(), weight.detach()
    B, ED = xin.shape
    K = weight.shape[-1]
    dt = xin.dtype
    x_ = xin if xin.stride(-1) == 1 else xin.contiguous()
    new_inputs = inputs.to(dt).contiguous().clone()
    w_ = weight.float().reshape(ED, K).contiguous()
    b_ = _f32(bias)
    u = torch.empty((B, ED), dtype=dt, device=dev)
    l = nat.lib()
    with torch.cuda.device(dev):
        nat.check(l.gfe_conv1d_step(_ptr(x_), x_.stride(0), _ptr(new_inputs), _ptr(w_), _ptr(b_), _ptr(u), u.stride(0),
                                    B, ED, K, _DT[dt], _stream(dev)), "conv1d_step")
    return u, new_inputs


def conv1d_prefill(xin: torch.Tensor, inputs: Optional[torch.Tensor], weight: torch.Tensor, bias: Optional[torch.Tensor]
                   ) -> Tuple[torch.Tensor, torch.Tensor]:
    """L tokens of the causal conv continuing a decode cache: the multi-token ``conv1d_step``.  xin: (B, L, ED) (any
    batch / row strides, unit channel stride); inputs: (B, ED, K-1) or None (zeros).  Returns (u (B, L, ED),
    new_inputs (B, ED, K-1)): u equals causal_conv1d_silu over cat(inputs, xin) without its first K-1 rows, new_inputs is
    the cache L calls of ``conv1d_step`` would leave.  Inference only; ``inputs`` is not modified."""
    dev = _require_cuda(xin, inputs, weight, bias)
    _no_autograd("conv1d_prefill", xin, inputs, weight, bias)
    if xin.dim() != 3:
        raise ValueError(f"conv1d_prefill: x must be (B, L, ED); got {tuple(xin.shape)}")
    B, L, ED = xin.shape
    K = weight.shape[-1]
    dt = xin.dtype
    if dt not in _DT:
        raise TypeError(f"conv1d_prefill: unsupported activation dtype {dt}")
    if weight.numel() != ED * K or (inputs is not None and tuple(inputs.shape) != (B, ED, K - 1)):
        raise ValueError("conv1d_prefill: weight must be (ED, 1, K) / (ED, K) and inputs (B, ED, K-1)")
    x_ = _rows(xin.detach())
    in_ = None if inputs is None else inputs.detach().to(dt).contiguous()
    w_ = weight.detach().float().reshape(ED, K).contiguous()
    b_ = _f32(bias)
    u = torch.empty((B, L, ED), dtype=dt, device=dev)
    new_inputs = torch.empty((B, ED, K - 1), dtype=dt, device=dev)
    l = nat.lib()
    with torch.cuda.device(dev):
        nat.check(l.gfe_conv1d_silu_fwd_state(_ptr(x_), x_.stride(0), x_.stride(1), _ptr(w_), _ptr(b_), _ptr(in_), _ptr(new_inputs),
                                              _ptr(u), u.stride(0), u.stride(1), B, L, ED, K, _DT[dt], _stream(dev)),
                  "conv1d_silu_fwd_state")
    return u, new_inputs


def ssm_prefill(u, delta, A_log, Bm, Cm, D, h, z=None, dt_bias=None, delta_softplus: bool = True):
    """L tokens of the selective scan from a carried state: the multi-token ``ssm_step``.  u, delta, z: (B, L, ED); Bm, Cm:
    (B, L, N) (any batch / row strides, unit channel stride: the halves of in_proj's and the slices of x_proj's output are
    read in place); h: (B, ED, N) or None (zeros).  Returns (out (B, L, ED), h_new (B, ED, N) fp32): the outputs and final
    state of ``selective_scan_fn`` over the L tokens started from h instead of zero -- what L calls of ``ssm_step`` give.
    Inference only (no checkpoints are written); ``h`` is not modified."""
    dev = _require_cuda(u, delta, A_log, Bm, Cm, D, h, z, dt_bias)
    _no_autograd("ssm_prefill", u, delta, A_log, Bm, Cm, D, h, z, dt_bias)
    if u.dim() != 3:
        raise ValueError(f"ssm_prefill: u must be (B, L, ED); got {tuple(u.shape)}")
    B, L, ED = u.shape
    N = A_log.shape[1]
    dt = u.dtype
    if dt not in _DT:
        raise TypeError(f"ssm_prefill: unsupported activation dtype {dt}")
    if tuple(delta.shape) != (B, L, ED) or tuple(Bm.shape) != (B, L, N) or tuple(Cm.shape) != (B, L, N) \
            or tuple(A_log.shape) != (ED, N) or tuple(D.shape) != (ED,) or (h is not None and tuple(h.shape) != (B, ED, N)):
        raise ValueError("ssm_prefill: inconsistent shapes")
    u_, delta_, Bm_, Cm_ = (_as(t, dt) for t in (u, delta, Bm, Cm))
    z_ = None if z is None else _as(z, dt)
    A_log_, D_, bias_ = _f32(A_log), _f32(D), _f32(dt_bias)
    h_ = None if h is None else _f32(h)
    if h_ is not None and h_.data_ptr() % 16:   # the kernels read the state as 16-byte vectors
        h_ = h_.clone()
    out = torch.empty((B, L, ED), dtype=dt, device=dev)
    h_new = torch.empty((B, ED, N), dtype=torch.float32, device=dev)
    l = nat.lib()
    a = nat.SelscanArgs()
    _fill_common(a, u_, delta_, z_, Bm_, Cm_, A_log_, D_, bias_, delta_softplus)
    a.out, a.out_bs, a.out_rs = out.data_ptr(), out.stride(0), out.stride(1)
    a.last_state = h_new.data_ptr()
    with torch.cuda.device(dev):
        nws = _sizes(B, L, ED, N, dev, _DT[dt])[1]
        ws = _bytes(nws, dev)
        a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), nws
        nat.check(l.gfe_selscan_fwd_state(ctypes.byref(a), _ptr(h_), _stream(dev)), "selscan_fwd_state")
    return out, h_new


# ------------------------------------------------------------ training from a carried state
def _state16(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    """A (B, ED, N) state as the kernels read it: fp32, contiguous, 16-byte aligned."""
    t = _f32(t)
    return t.clone() if (t is not None and t.data_ptr() % 16) else t


class _SelectiveScanStateFn(torch.autograd.Function):
    """selective_scan_fn from a carried state h0 with the final state as a second output, differentiable in both: the
    forward keeps checkpoints that start from h0, the backward seeds its reverse carry with d h_last and returns d h0."""

    @staticmethod
    def forward(ctx, u, delta, A_log, Bm, Cm, D, h0, z, dt_bias, softplus: bool, grad_mode: bool):
        dev = _require_cuda(u, delta, A_log, Bm, Cm, D, h0, z, dt_bias)
        if u.dim() != 3:
            raise ValueError(f"selective_scan_state: u must be (B, L, ED); got {tuple(u.shape)}")
        B, L, ED = u.shape
        N = A_log.shape[1]
        dt = u.dtype
        if dt not in _DT:
            raise TypeError(f"selective_scan_state: unsupported activation dtype {dt}")
        if tuple(delta.shape) != (B, L, ED) or tuple(Bm.shape) != (B, L, N) or tuple(Cm.shape) != (B, L, N) \
                or tuple(A_log.shape) != (ED, N) or tuple(D.shape) != (ED,) or (h0 is not None and tuple(h0.shape) != (B, ED, N)):
            raise ValueError("selective_scan_state: inconsistent shapes")
        u_, delta_, Bm_, Cm_ = (_as(t, dt) for t in (u, delta, Bm, Cm))
        z_ = None if z is None else _as(z, dt)
        A_log_, D_, bias_ = _f32(A_log), _f32(D), _f32(dt_bias)
        h0_ = _state16(h0)
        out = torch.empty((B, L, ED), dtype=dt, device=dev)
        last = torch.empty((B, ED, N), dtype=torch.float32, device=dev)
        need_grad = grad_mode and any(ctx.needs_input_grad)
        l = nat.lib()
        a = nat.SelscanArgs()
        _fill_common(a, u_, delta_, z_, Bm_, Cm_, A_log_, D_, bias_, softplus)
        a.out, a.out_bs, a.out_rs = out.data_ptr(), out.stride(0), out.stride(1)
        a.last_state = last.data_ptr()
        with torch.cuda.device(dev):
            sz = _sizes(B, L, ED, N, dev, _DT[dt])
            nck = sz[0] if need_grad else 0
            ckpt = _bytes(nck, dev)
            ws = _bytes(sz[1], dev)
            a.ckpt, a.ckpt_bytes = (0 if ckpt is None else ckpt.data_ptr()), nck
            a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), sz[1]
            nat.check(l.gfe_selscan_fwd_carry(ctypes.byref(a), _ptr(h0_), _stream(dev)), "selscan_fwd_carry")
        # an unused output arrives in backward as None: an unused h_last runs the backward with dlast = NULL
        ctx.set_materialize_grads(False)
        if need_grad:
            ctx.save_for_backward(u_, delta_, A_log_, Bm_, Cm_, D_, z_, bias_, ckpt)
            ctx.softplus = softplus
            ctx.in_dtypes = tuple(None if t is None else t.dtype for t in (u, delta, A_log, Bm, Cm, D, h0, z, dt_bias))
        return out, last

    @staticmethod
    def backward(ctx, dout, dlast):
        u, delta, A_log, Bm, Cm, D, z, bias, ckpt = ctx.saved_tensors
        dev = u.device
        B, L, ED = u.shape
        N = A_log.shape[1]
        dt = u.dtype
        dout = torch.zeros((B, L, ED), dtype=dt, device=dev) if dout is None else _as(dout, dt)
        dlast = _state16(dlast)
        du = torch.empty((B, L, ED), dtype=dt, device=dev)
        ddelta = torch.empty((B, L, ED), dtype=dt, device=dev)
        dz = None if z is None else torch.empty((B, L, ED), dtype=dt, device=dev)
        dBm = torch.empty((B, L, N), dtype=dt, device=dev)
        dCm = torch.empty((B, L, N), dtype=dt, device=dev)
        dA_log = torch.empty((ED, N), dtype=torch.float32, device=dev)
        dD = torch.empty((ED,), dtype=torch.float32, device=dev)
        dbias = None if bias is None else torch.empty((ED,), dtype=torch.float32, device=dev)
        dh0 = torch.empty((B, ED, N), dtype=torch.float32, device=dev) if ctx.needs_input_grad[6] else None
        l = nat.lib()
        a = nat.SelscanArgs()
        _fill_common(a, u, delta, z, Bm, Cm, A_log, D, bias, ctx.softplus)
        a.ckpt, a.ckpt_bytes = ckpt.data_ptr(), ckpt.numel()
        a.dout, a.dout_bs, a.dout_rs = dout.data_ptr(), dout.stride(0), dout.stride(1)
        a.du, a.du_bs, a.du_rs = du.data_ptr(), du.stride(0), du.stride(1)
        a.ddelta, a.ddelta_bs, a.ddelta_rs = ddelta.data_ptr(), ddelta.stride(0), ddelta.stride(1)
        if dz is not None:
            a.dz, a.dz_bs, a.dz_rs = dz.data_ptr(), dz.stride(0), dz.stride(1)
        a.dBm, a.dB_bs, a.dB_rs = dBm.data_ptr(), dBm.stride(0), dBm.stride(1)
        a.dCm, a.dC_bs, a.dC_rs = dCm.data_ptr(), dCm.stride(0), dCm.stride(1)
        a.dA_log, a.dD = dA_log.data_ptr(), dD.data_ptr()
        a.ddt_bias = 0 if dbias is None else dbias.data_ptr()
        with torch.cuda.device(dev):
            nws = _sizes(B, L, ED, N, dev, _DT[dt])[2]
            ws = _bytes(nws, dev)
            a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), nws
            nat.check(l.gfe_selscan_bwd_carry(ctypes.byref(a), _ptr(dlast), _ptr(dh0), _stream(dev)), "selscan_bwd_carry")
        dts = ctx.in_dtypes

        def cast(g, i):
            return None if (g is None or dts[i] is None) else (g if g.dtype == dts[i] else g.to(dts[i]))

        return (cast(du, 0), cast(ddelta, 1), cast(dA_log, 2), cast(dBm, 3), cast(dCm, 4), cast(dD, 5), cast(dh0, 6),
                cast(dz, 7), cast(dbias, 8), None, None)


def selective_scan_state(u, delta, A_log, Bm, Cm, D, h0, z=None, dt_bias=None, delta_softplus: bool = True):
    """selective_scan_fn started from a carried state, for training in chunks.  h0: (B, ED, N) or None (zeros); the other
    arguments as for selective_scan_fn.  Returns (out (B, L, ED), h_last (B, ED, N) fp32), both differentiable, h0 included:
    feeding one chunk's h_last (not detached) as the next chunk's h0 gives the gradients of one pass over the whole sequence,
    detaching it gives truncated backpropagation through time.  Under no_grad no checkpoint is allocated.  ``h0`` is not
    modified."""
    return _SelectiveScanStateFn.apply(u, delta, A_log, Bm, Cm, D, h0, z, dt_bias, bool(delta_softplus), torch.is_grad_enabled())


class _CausalConv1dSiluStateFn(torch.autograd.Function):
    """causal_conv1d_silu over cat(inputs, xin) without its first K-1 rows: the conv from a carried window, differentiable in
    the window too."""

    @staticmethod
    def forward(ctx, xin, inputs, weight, bias):
        dev = _require_cuda(xin, inputs, weight, bias)
        B, L, ED = xin.shape
        K = weight.shape[-1]
        x_ = _rows(xin.detach())
        in_ = None if inputs is None else inputs.detach().contiguous()
        w_ = weight.detach().float().reshape(ED, K).contiguous()
        b_ = _f32(bias)
        u = torch.empty((B, L, ED), dtype=xin.dtype, device=dev)
        l = nat.lib()
        with torch.cuda.device(dev):
            nat.check(l.gfe_conv1d_silu_fwd_state(_ptr(x_), x_.stride(0), x_.stride(1), _ptr(w_), _ptr(b_), _ptr(in_), None,
                                                  _ptr(u), u.stride(0), u.stride(1), B, L, ED, K, _DT[xin.dtype], _stream(dev)),
                      "conv1d_silu_fwd_state")
        ctx.save_for_backward(x_, in_, w_, b_)
        ctx.meta = (weight.shape, weight.dtype, None if bias is None else bias.dtype)
        return u

    @staticmethod
    def backward(ctx, du):
        x_, in_, w_, b_ = ctx.saved_tensors
        dev = x_.device
        B, L, ED = x_.shape
        K = w_.shape[1]
        du = _rows(du.detach().to(x_.dtype))
        dx = torch.empty((B, L, ED), dtype=x_.dtype, device=dev)
        dw = torch.empty((ED, K), dtype=torch.float32, device=dev)
        db = None if b_ is None else torch.empty((ED,), dtype=torch.float32, device=dev)
        din = torch.empty((B, ED, K - 1), dtype=x_.dtype, device=dev) if ctx.needs_input_grad[1] else None
        l = nat.lib()
        with torch.cuda.device(dev):
            nws = l.gfe_conv1d_bwd_workspace_bytes(B, L, ED, K)
            ws = _bytes(nws, dev)
            nat.check(l.gfe_conv1d_silu_bwd_carry(_ptr(x_), x_.stride(0), x_.stride(1), _ptr(w_), _ptr(b_), _ptr(in_), _ptr(du),
                                                  du.stride(0), du.stride(1), _ptr(dx), dx.stride(0), dx.stride(1), _ptr(dw),
                                                  _ptr(db), _ptr(din), B, L, ED, K, _DT[x_.dtype], _ptr(ws), nws, _stream(dev)),
                      "conv1d_silu_bwd_carry")
        wshape, wdt, bdt = ctx.meta
        return dx, din, dw.reshape(wshape).to(wdt), (None if db is None else db.to(bdt))


def causal_conv1d_silu_state(xin: torch.Tensor, inputs: Optional[torch.Tensor], weight: torch.Tensor,
                             bias: Optional[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
    """The causal conv + SiLU continuing a carried window, for training in chunks.  xin: (B, L, ED) (any batch / row strides,
    unit channel stride); inputs: (B, ED, K-1) or None (zeros).  Returns (u (B, L, ED), new_inputs (B, ED, K-1)) as
    conv1d_prefill does, differentiable in xin, inputs, weight and bias.  ``inputs`` is read in xin's dtype; new_inputs, the
    last K-1 rows of cat(inputs, xin) along time, is a torch gather, so its gradient reaches both."""
    _require_cuda(xin, inputs, weight, bias)
    if xin.dim() != 3:
        raise ValueError(f"causal_conv1d_silu_state: x must be (B, L, ED); got {tuple(xin.shape)}")
    B, L, ED = xin.shape
    K = weight.shape[-1]
    if xin.dtype not in _DT:
        raise TypeError(f"causal_conv1d_silu_state: unsupported activation dtype {xin.dtype}")
    if weight.numel() != ED * K or (inputs is not None and tuple(inputs.shape) != (B, ED, K - 1)):
        raise ValueError("causal_conv1d_silu_state: weight must be (ED, 1, K) / (ED, K) and inputs (B, ED, K-1)")
    if inputs is not None:
        inputs = inputs.to(xin.dtype)
    u = _CausalConv1dSiluStateFn.apply(xin, inputs, weight, bias)
    window = inputs if inputs is not None else xin.new_zeros((B, ED, K - 1))
    new_inputs = torch.cat([window, xin[:, max(0, L - (K - 1)):].transpose(1, 2)], dim=2)[:, :, -(K - 1):].contiguous()
    return u, new_inputs


# ------------------------------------------------------------ summaries of a whole range
def _summary_call(fn: str, x, delta, A_log, BC, z, dt_bias, softplus: bool, rev: bool):
    """gfe_selscan_summary_fwd (x = u, BC = Bm) or _bwd (x = dout, BC = Cm): (state (B, ED, N) fp32, sum_delta (B, ED) fp32
    or None)."""
    dev = _require_cuda(x, delta, A_log, BC, z, dt_bias)
    _no_autograd(fn, x, delta, A_log, BC, z, dt_bias)
    if x.dim() != 3:
        raise ValueError(f"{fn}: activations must be (B, L, ED); got {tuple(x.shape)}")
    B, L, ED = x.shape
    N = A_log.shape[1]
    dt = x.dtype
    if dt not in _DT:
        raise TypeError(f"{fn}: unsupported activation dtype {dt}")
    if tuple(delta.shape) != (B, L, ED) or tuple(BC.shape) != (B, L, N) or tuple(A_log.shape) != (ED, N) \
            or (z is not None and tuple(z.shape) != (B, L, ED)):
        raise ValueError(f"{fn}: inconsistent shapes")
    x_, delta_, BC_ = (_as(t, dt) for t in (x, delta, BC))
    z_ = None if z is None else _as(z, dt)
    A_log_, bias_ = _f32(A_log), _f32(dt_bias)
    state = torch.empty((B, ED, N), dtype=torch.float32, device=dev)
    sd = None if rev else torch.empty((B, ED), dtype=torch.float32, device=dev)
    l = nat.lib()
    a = nat.SelscanArgs()
    a.batch, a.seqlen, a.d_inner, a.d_state = B, L, ED, N
    a.dtype = _DT[dt]
    a.flags = nat.GFE_FLAG_DELTA_SOFTPLUS if softplus else 0
    a.delta, a.delta_bs, a.delta_rs = delta_.data_ptr(), delta_.stride(0), delta_.stride(1)
    if rev:
        a.dout, a.dout_bs, a.dout_rs = x_.data_ptr(), x_.stride(0), x_.stride(1)
        a.Cm, a.C_bs, a.C_rs = BC_.data_ptr(), BC_.stride(0), BC_.stride(1)
        if z_ is not None:
            a.z, a.z_bs, a.z_rs = z_.data_ptr(), z_.stride(0), z_.stride(1)
    else:
        a.u, a.u_bs, a.u_rs = x_.data_ptr(), x_.stride(0), x_.stride(1)
        a.Bm, a.B_bs, a.B_rs = BC_.data_ptr(), BC_.stride(0), BC_.stride(1)
    a.A_log = A_log_.data_ptr()
    a.dt_bias = 0 if bias_ is None else bias_.data_ptr()
    with torch.cuda.device(dev):
        nws = l.gfe_selscan_summary_workspace_bytes(B, L, ED, N)
        ws = _bytes(nws, dev)
        a.ws, a.ws_bytes = (0 if ws is None else ws.data_ptr()), nws
        if rev:
            nat.check(l.gfe_selscan_summary_bwd(ctypes.byref(a), _ptr(state), _stream(dev)), "selscan_summary_bwd")
        else:
            nat.check(l.gfe_selscan_summary_fwd(ctypes.byref(a), _ptr(state), _ptr(sd), _stream(dev)), "selscan_summary_fwd")
    return state, sd


def selscan_summary(u, delta, A_log, Bm, dt_bias=None, delta_softplus: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
    """What a range of tokens does to the scan state, for passing state between devices that each hold part of a sequence.
    u, delta: (B, L, ED); Bm: (B, L, N) (any batch / row strides, unit channel stride); A_log: (ED, N).  Returns (h_loc
    (B, ED, N) fp32, sum_delta (B, ED) fp32): the final state of ``selective_scan_fn`` over the L tokens started from zero, and
    the sum over the tokens of the step size (softplus(delta + dt_bias) with ``delta_softplus``, else delta + dt_bias).  The
    state after the range from a state h is exp(A sum_delta) h + h_loc per state, A = -exp(A_log).  Inference only."""
    return _summary_call("selscan_summary", u, delta, A_log, Bm, None, dt_bias, delta_softplus, False)


def selscan_summary_rev(dout, delta, A_log, Cm, z=None, dt_bias=None, delta_softplus: bool = True) -> torch.Tensor:
    """The reverse counterpart of ``selscan_summary``: g_loc (B, ED, N) fp32, the gradient of the state before the range that
    the output gradient ``dout`` (B, L, ED) alone produces -- d h0 of ``selective_scan_state`` with no gradient on its final
    state.  With a final-state gradient dlast it is exp(A sum_delta) dlast + g_loc.  z: the gate, or None.  Inference only."""
    return _summary_call("selscan_summary_rev", dout, delta, A_log, Cm, z, dt_bias, delta_softplus, True)[0]


def ssm_step(u, delta, A_log, Bm, Cm, D, h, z=None, dt_bias=None, delta_softplus: bool = True):
    """One token of the selective scan (mamba.py:375-405).  u, delta, z: (B, ED); Bm, Cm: (B, N); h: (B, ED, N) or None.
    Returns (out, h_new); ``h`` is not modified."""
    dev = _require_cuda(u, delta, A_log, Bm, Cm, D, h, z, dt_bias)
    _no_autograd("ssm_step", u, delta, A_log, Bm, Cm, D, h, z, dt_bias)
    B, ED = u.shape
    N = A_log.shape[1]
    dt = u.dtype
    h = None if h is None else h.detach()

    def row(t):
        if t is None:
            return None
        t = t.detach().to(dt)
        return t if t.stride(-1) == 1 else t.contiguous()

    u_, delta_, z_, Bm_, Cm_ = row(u), row(delta), row(z), row(Bm), row(Cm)
    h_new = torch.zeros((B, ED, N), dtype=torch.float32, device=dev) if h is None else h.float().contiguous().clone()
    out = torch.empty((B, ED), dtype=dt, device=dev)
    A_log_, D_, bias_ = _f32(A_log), _f32(D), _f32(dt_bias)
    l = nat.lib()
    with torch.cuda.device(dev):
        nat.check(l.gfe_ssm_step(_ptr(u_), u_.stride(0), _ptr(delta_), delta_.stride(0), _ptr(z_), 0 if z_ is None else z_.stride(0),
                                 _ptr(Bm_), Bm_.stride(0), _ptr(Cm_), Cm_.stride(0), _ptr(A_log_), _ptr(D_), _ptr(bias_),
                                 _ptr(h_new), _ptr(out), out.stride(0), B, ED, N,
                                 nat.GFE_FLAG_DELTA_SOFTPLUS if delta_softplus else 0, _DT[dt], _stream(dev)), "ssm_step")
    return out, h_new
