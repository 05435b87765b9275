"""Selective scan forward + backward per layer at d_state N in {16, 32, 64}: the fused kernels against the reference's
composition (exp(delta A) and delta B u materialised as (B, L, ED, N) fp32 tensors and run through the pscan kernel, what
MambaBlock does for state sizes the fused kernels are not compiled for).  Reports ms per layer, tokens/s and the peak memory
allocated by one forward + backward; a composition that does not fit is reported as out of memory.

usage: python tools/bench_dstate.py [--iters K] [--out FILE]
Shapes: prod (B=2, L=1858, ED=1024, fp32) and cfg3 (B=16, L=4096, ED=1536, bf16), both gated (z) with dt_bias and softplus.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gfe_mamba_b200 import ops  # noqa: E402

SHAPES = {"prod": (2, 1858, 1024, torch.float32), "cfg3": (16, 4096, 1536, torch.bfloat16)}


def inputs(B, L, ED, N, dt):
    g = torch.Generator(device="cuda").manual_seed(N)
    r = lambda *s, sc=1.0: (torch.randn(*s, device="cuda", generator=g) * sc).to(dt).requires_grad_()
    A_log = torch.log(torch.arange(1, N + 1, device="cuda", dtype=torch.float32)).expand(ED, N).clone().requires_grad_()
    return dict(u=r(B, L, ED), delta=r(B, L, ED, sc=0.5), z=r(B, L, ED), Bm=r(B, L, N), Cm=r(B, L, N), A_log=A_log,
                D=torch.ones(ED, device="cuda", requires_grad=True),
                bias=torch.full((ED,), -4.0, device="cuda", requires_grad=True), dout=r(B, L, ED).detach())


def fused(t):
    y = ops.selective_scan_fn(t["u"], t["delta"], t["A_log"], t["Bm"], t["Cm"], t["D"], z=t["z"], dt_bias=t["bias"])
    y.backward(t["dout"])


def composition(t):
    """MambaBlock._ssm_fused's fallback for other state sizes: softplus, discretise, pscan, C contraction, D skip, gate."""
    delta = F.softplus(t["delta"].float() + t["bias"])
    A = -torch.exp(t["A_log"])
    u = t["u"].float()
    hs = ops.pscan(torch.exp(delta.unsqueeze(-1) * A), (delta.unsqueeze(-1) * t["Bm"].float().unsqueeze(2)) * u.unsqueeze(-1))
    y = (hs @ t["Cm"].float().unsqueeze(-1)).squeeze(3) + t["D"] * u
    y = (y * F.silu(t["z"].float())).to(t["u"].dtype)
    y.backward(t["dout"])


def measure(fn, t, iters):
    """(ms per forward + backward, peak bytes allocated by one forward + backward above the inputs)."""
    for k in ("u", "delta", "z", "Bm", "Cm", "A_log", "D", "bias"):
        t[k].grad = None
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn(t)   # warm-up, and the memory probe
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    fn(t)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn(t)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters, peak


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dstate: no CUDA device (this measurement needs a GPU; there is no CPU fallback)")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    rows = [{"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}]
    print(json.dumps(rows[0]), flush=True)
    for shape, (B, L, ED, dt) in SHAPES.items():
        for N in (16, 32, 64):
            for impl, fn, iters in (("fused", fused, args.iters), ("composition", composition, max(2, args.iters // 4))):
                row = dict(shape=shape, B=B, L=L, ED=ED, N=N, dtype=str(dt).replace("torch.", ""), impl=impl)
                t = None
                try:
                    t = inputs(B, L, ED, N, dt)
                    ms, peak = measure(fn, t, iters)
                    row.update(ms_fwd_bwd=round(ms, 3), tokens_per_s=round(B * L / ms * 1e3), peak_alloc_gb=round(peak / 1e9, 3))
                except torch.cuda.OutOfMemoryError:
                    row.update(result="out of memory")
                del t
                torch.cuda.empty_cache()
                rows.append(row)
                print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(r) for r in rows) + "\n")


if __name__ == "__main__":
    main()
