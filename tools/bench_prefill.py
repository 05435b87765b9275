"""Prefill from a decode cache: what the forward kernels started from a carried state cost, and what Mamba.prefill saves
over decoding a prompt token by token.

usage: python tools/bench_prefill.py [--iters K] [--reps R] [--out FILE]
  scan   per layer, ops.ssm_prefill from a non-zero state against selective_scan_fn (zero start) under no_grad, alternated
         R times: cfg 3 (B=16, L=4096, ED=1536, bf16, chained kernels, waiting segments) and the production shape (B=2,
         L=1858, ED=1024, fp32, chained kernels, independent segments); gated, dt_bias, softplus.
  model  production config (d_model=512, 6 layers, B=2, fp32): Mamba.prefill(P) against P x GraphedDecoder.step, P in
         {64, 512, 1858}; and the 1858-token prompt prefilled in chunks of 256 and 1024 against one prefill.
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
from gfe_mamba_b200.decode import GraphedDecoder  # noqa: E402

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
        r = lambda *s, sc=1.0: (torch.randn(*s, device="cuda", generator=g) * sc).to(dt)
        u, delta, z, Bm, Cm = r(B, L, ED), r(B, L, ED, sc=0.5), r(B, L, ED), r(B, L, N), r(B, L, N)
        A_log = torch.log(torch.arange(1, N + 1, device="cuda", dtype=torch.float32)).expand(ED, N).contiguous()
        D = torch.ones(ED, device="cuda")
        bias = torch.full((ED,), -4.0, device="cuda")
        h0 = torch.randn(B, ED, N, device="cuda", generator=g) * 0.5
        with torch.no_grad():
            fwd = lambda: ops.selective_scan_fn(u, delta, A_log, Bm, Cm, D, z=z, dt_bias=bias, return_last_state=True)
            pre = lambda: ops.ssm_prefill(u, delta, A_log, Bm, Cm, D, h0, z=z, dt_bias=bias)
            for rep in range(reps):
                for label, fn in (("selective_scan_fn", fwd), ("ssm_prefill_from_state", pre)):
                    ms = time_ms(fn, iters)
                    rows.append(dict(kind="scan", shape=name, B=B, L=L, ED=ED, dtype=str(dt).split(".")[-1], fn=label, rep=rep,
                                     ms=round(ms, 4), Mtok_s=round(B * L / ms / 1e3, 2)))
    return rows


def model_rows(iters):
    torch.manual_seed(0)
    m = Mamba(MambaConfig(d_model=512, n_layers=6)).cuda().eval()
    B = 2
    x = torch.randn(B, 1858, 512, device="cuda")
    dec = GraphedDecoder(m, B)
    rows = []
    with torch.no_grad():
        for P in (64, 512, 1858):
            xp = x[:, :P]
            t_pre = time_ms(lambda: m.prefill(xp), iters)

            def loop():
                for s in range(P):
                    dec.step(xp[:, s])
            t_loop = time_ms(loop, max(1, iters // 4))
            rows.append(dict(kind="model", what="prefill vs GraphedDecoder.step loop", B=B, P=P, prefill_ms=round(t_pre, 3),
                             step_loop_ms=round(t_loop, 3), speedup=round(t_loop / t_pre, 1)))
        one = time_ms(lambda: m.prefill(x), iters)
        for chunk in (256, 1024):
            def chunked():
                caches = None
                for s0 in range(0, x.shape[1], chunk):
                    _, caches = m.prefill(x[:, s0:s0 + chunk], caches)
            rows.append(dict(kind="model", what="chunked prefill vs one prefill", B=B, P=x.shape[1], chunk=chunk,
                             chunked_ms=round(time_ms(chunked, iters), 3), one_ms=round(one, 3)))
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_prefill: no CUDA device (this measurement needs a GPU; there is no CPU fallback)")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    rows = [{"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q}] + scan_rows(args.iters, args.reps) + model_rows(args.iters)
    text = "\n".join(json.dumps(r) for r in rows) + "\n"
    print(text, end="")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()
