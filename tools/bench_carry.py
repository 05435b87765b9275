"""Training from a carried state: what the backward through (h, conv window) costs, and what the fused Mamba.prefill under grad
saves over the differentiable token loop.

usage: python tools/bench_carry.py [--iters K] [--reps R] [--out FILE]
  scan   per layer, forward + backward: ops.selective_scan_state from a non-zero h0 with a loss on out and h_last (so the
         backward takes dlast and returns dh0) against selective_scan_fn (zero start, loss on out), alternated R times: cfg 3
         (B=16, L=4096, ED=1536, bf16, chained kernels, waiting segments) and the production shape (B=2, L=1858, ED=1024,
         fp32, chained kernels, independent segments); gated, dt_bias, softplus.
  model  production config (d_model=512, 6 layers, B=2, fp32, training mode): forward + backward of Mamba.prefill(P) under grad
         (fused) against P differentiable MambaBlock.step calls per layer (the token loop), P in {64, 512}.
  chunk  cfg 4's sequence (B=1, L=65536, d_model=512, 2 layers, fp32): forward + backward in 4096-token chunks with the
         caches passed on (gradients of one pass) and detached (truncated BPTT), against one forward + backward; time and
         peak memory.
Times are CUDA-event means over K calls after a warm-up call; one JSON line per measurement.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gfe_mamba_b200 import Mamba, MambaConfig, ops  # noqa: E402

SHAPES = {"cfg3": (16, 4096, 1536, torch.bfloat16), "prod": (2, 1858, 1024, torch.float32)}
N = 16


def time_ms(fn, iters):
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def scan_rows(iters, reps):
    rows = []
    for name, (B, L, ED, dt) in SHAPES.items():
        g = torch.Generator(device="cuda").manual_seed(0)
        r = lambda *s, sc=1.0: (torch.randn(*s, device="cuda", generator=g) * sc).to(dt).requires_grad_()
        u, delta, z, Bm, Cm = r(B, L, ED), r(B, L, ED, sc=0.5), r(B, L, ED), r(B, L, N), r(B, L, N)
        A_log = torch.log(torch.arange(1, N + 1, device="cuda", dtype=torch.float32)).expand(ED, N).contiguous().requires_grad_()
        D = torch.ones(ED, device="cuda", requires_grad=True)
        bias = torch.full((ED,), -4.0, device="cuda", requires_grad=True)
        h0 = (torch.randn(B, ED, N, device="cuda", generator=g) * 0.5).requires_grad_()
        dout = torch.randn(B, L, ED, device="cuda", generator=g).to(dt)
        W = torch.randn(B, ED, N, device="cuda", generator=g)

        def zero():
            y = ops.selective_scan_fn(u, delta, A_log, Bm, Cm, D, z=z, dt_bias=bias)
            y.backward(dout)

        def carry():
            y, h = ops.selective_scan_state(u, delta, A_log, Bm, Cm, D, h0, z=z, dt_bias=bias)
            torch.autograd.backward((y, h), (dout, W))
        for rep in range(reps):
            for label, fn in (("selective_scan_fn zero start", zero), ("selective_scan_state from h0, dlast + dh0", carry)):
                ms = time_ms(fn, iters)
                rows.append(dict(kind="scan fwd+bwd", shape=name, B=B, L=L, ED=ED, dtype=str(dt).split(".")[-1], fn=label,
                                 rep=rep, ms=round(ms, 4), Mtok_s=round(B * L / ms / 1e3, 2)))
    return rows


def model_rows(iters):
    torch.manual_seed(0)
    m = Mamba(MambaConfig(d_model=512, n_layers=6)).cuda().train()
    B = 2
    x = torch.randn(B, 512, 512, device="cuda")
    rows = []
    for P in (64, 512):
        xp = x[:, :P]

        def fused():
            y, caches = m.prefill(xp)
            (y.square().mean() + sum(h.square().mean() for h, _ in caches)).backward()

        def loop():
            caches = [(None, torch.zeros(B, m.config.d_inner, m.config.d_conv - 1, device="cuda")) for _ in m.layers]
            ys = []
            for s in range(P):
                h = xp[:, s]
                for i, layer in enumerate(m.layers):
                    h, caches[i] = layer.step(h, caches[i])
                ys.append(h)
            (torch.stack(ys, 1).square().mean() + sum(c[0].square().mean() for c in caches)).backward()
        t_f = time_ms(fused, iters)
        t_l = time_ms(loop, max(1, iters // 10))
        rows.append(dict(kind="model fwd+bwd", what="Mamba.prefill under grad vs differentiable step loop", B=B, P=P,
                         fused_ms=round(t_f, 3), step_loop_ms=round(t_l, 3), speedup=round(t_l / t_f, 1)))
    return rows


def chunk_rows(iters):
    torch.manual_seed(0)
    m = Mamba(MambaConfig(d_model=512, n_layers=2)).cuda().train()
    x = torch.randn(1, 65536, 512, device="cuda")
    C = 4096

    def one():
        m(x).square().mean().backward()

    def chunked_tbptt():
        caches = None
        for s0 in range(0, x.shape[1], C):
            y, caches = m.prefill(x[:, s0:s0 + C], caches)
            y.square().mean().backward()
            caches = [(h.detach(), i.detach()) for h, i in caches]

    def chunked_full():
        caches, loss = None, 0
        for s0 in range(0, x.shape[1], C):
            y, caches = m.prefill(x[:, s0:s0 + C], caches)
            loss = loss + y.square().mean()
        loss.backward()

    rows = []
    for label, fn in (("one pass", one), ("4096-token chunks, caches passed on", chunked_full),
                      ("4096-token chunks, caches detached (truncated BPTT)", chunked_tbptt)):
        ms = time_ms(fn, iters)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        rows.append(dict(kind="chunked training", B=1, L=x.shape[1], d_model=512, n_layers=2, what=label, ms=round(ms, 2),
                         peak_MiB=round(peak / 2**20, 1)))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_carry: no CUDA device (this measurement needs a GPU; there is no CPU fallback)")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    rows = ([{"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}] + scan_rows(args.iters, args.reps) + model_rows(args.iters)
            + chunk_rows(max(1, args.iters // 10)))
    text = "\n".join(json.dumps(r) for r in rows) + "\n"
    print(text, end="")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
