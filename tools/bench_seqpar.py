"""Sequence parallelism: one long sequence split along time over G GPUs (gfe_mamba_b200.parallel.sequence_sharded_*).

usage: torchrun --nproc-per-node G tools/bench_seqpar.py [--steps K] [--warmup W] [--out FILE]
  scan     cfg 4's scan alone: B=1, L=65536, ED=1024, d_state=16, fp32, gated, dt_bias, softplus; forward + backward of
           sequence_sharded_scan (rank g holds L/G tokens), with the split into summary passes (selscan_summary +
           selscan_summary_rev), collectives (the two all-gathers) and main passes (the scan from the carry and its backward
           from dlast), each timed alone on the same inputs.
  channel  channel_sharded_scan at the same shape in the same run (rank g holds ED/G channels of all L tokens).
  model    a Mamba(d_model=512, n_layers=4) training step at B=1, L=65536 under bf16 autocast, sequence-sharded:
           forward, backward and allreduce_gradients(average=False).
Before timing, every rank checks its rows of the output and of the input gradients, and the summed parameter gradients,
against the same computation over the whole sequence on its own GPU.  Times are CUDA-event means over K steps after W
warm-up steps (the working set exceeds L2 at G <= 2 and not at G = 8: a rank's scan inputs are 4 x 256 MB / G); rank 0
prints one JSON line per measurement with the device name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gfe_mamba_b200 import Mamba, MambaConfig, ops, selective_scan_fn  # noqa: E402
from gfe_mamba_b200 import parallel as par  # noqa: E402

B, L, ED, N = 1, 65536, 1024, 16


def device_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    return r.stdout.strip()


def time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    if dist.is_initialized():
        dist.barrier()
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def rel(a, b):
    return float((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-30))


def scan_inputs(dev):
    g = torch.Generator(device="cpu").manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=g)
    d = dict(u=rn(B, L, ED), delta=0.5 * rn(B, L, ED), z=rn(B, L, ED), Bm=rn(B, L, N), Cm=rn(B, L, N), dout=rn(B, L, ED),
             A_log=torch.log(torch.arange(1, N + 1).float()).repeat(ED, 1) + 0.1 * rn(ED, N), D=1 + 0.1 * rn(ED), bias=-4 + rn(ED))
    return {k: v.to(dev) for k, v in d.items()}


def scan_bench(d, rank, world, args, out):
    names = ("u", "delta", "z", "Bm", "Cm")
    loc = {k: par.shard_sequence(d[k], rank, world).contiguous().requires_grad_() for k in names}
    prm = {k: torch.nn.Parameter(d[k].clone()) for k in ("A_log", "D", "bias")}
    dout = par.shard_sequence(d["dout"], rank, world).contiguous()

    def step():
        for t in list(loc.values()) + list(prm.values()):
            t.grad = None
        y = par.sequence_sharded_scan(loc["u"], loc["delta"], prm["A_log"], loc["Bm"], loc["Cm"], prm["D"], z=loc["z"],
                                      dt_bias=prm["bias"])
        y.backward(dout)
        return y

    # parity against the whole sequence on this GPU
    full = {k: d[k].clone().requires_grad_() for k in names}
    pf = {k: torch.nn.Parameter(d[k].clone()) for k in ("A_log", "D", "bias")}
    ref = selective_scan_fn(full["u"], full["delta"], pf["A_log"], full["Bm"], full["Cm"], pf["D"], z=full["z"], dt_bias=pf["bias"])
    ref.backward(d["dout"])
    y = step()
    par.allreduce_gradients(list(prm.values()), average=False)
    lo, hi = par.shard_range(L, rank, world)
    errs = {"out": rel(y, ref[:, lo:hi])}
    errs.update({k: rel(loc[k].grad, full[k].grad[:, lo:hi]) for k in names})
    errs.update({k: rel(prm[k].grad, pf[k].grad) for k in prm})
    del full, pf, ref
    ok = max(errs.values()) < 1e-4
    res = dict(bench="scan", world=world, parity_ok=ok, parity_max_rel=max(errs.values()))
    if not ok:
        out(dict(res, errs=errs))
        raise SystemExit(f"rank {rank}: parity failed {errs}")
    res["ms_per_step"] = time_ms(step, args.steps, args.warmup)

    # the parts, each alone
    with torch.no_grad():
        res["summary_ms"] = time_ms(lambda: (ops.selscan_summary(loc["u"], loc["delta"], prm["A_log"], loc["Bm"], dt_bias=prm["bias"]),
                                             ops.selscan_summary_rev(dout, loc["delta"], prm["A_log"], loc["Cm"], z=loc["z"],
                                                                     dt_bias=prm["bias"])), args.steps, args.warmup)
        if world > 1:
            pk = torch.zeros(B * ED * (N + 1), device=dout.device)
            g = torch.zeros(B * ED * N, device=dout.device)
            res["collective_ms"] = time_ms(lambda: (par._all_gather(pk, world, None), par._all_gather(g, world, None)),
                                           args.steps, args.warmup)
        else:
            res["collective_ms"] = 0.0
    h_in = torch.zeros(B, ED, N, device=dout.device)
    dlast = torch.zeros(B, ED, N, device=dout.device)

    def main_pass():
        for t in list(loc.values()) + list(prm.values()):
            t.grad = None
        y, h_last = ops.selective_scan_state(loc["u"], loc["delta"], prm["A_log"], loc["Bm"], loc["Cm"], prm["D"], h_in,
                                             z=loc["z"], dt_bias=prm["bias"])
        torch.autograd.backward([y, h_last], [dout, dlast])
    res["main_ms"] = time_ms(main_pass, args.steps, args.warmup)
    return res


def channel_bench(d, rank, world, args):
    sh = lambda t, dim=-1: par.shard_channels(t, rank, world, dim=dim).contiguous().clone().requires_grad_()
    u, delta, z = sh(d["u"]), sh(d["delta"]), sh(d["z"])
    A_log, D, bias = sh(d["A_log"], 0), sh(d["D"], 0), sh(d["bias"], 0)
    Bm, Cm = d["Bm"].clone().requires_grad_(), d["Cm"].clone().requires_grad_()
    dout = par.shard_channels(d["dout"], rank, world).contiguous()

    def step():
        for t in (u, delta, z, A_log, D, bias, Bm, Cm):
            t.grad = None
        y = par.channel_sharded_scan(selective_scan_fn, u, delta, A_log, Bm, Cm, D, z=z, dt_bias=bias)
        y.backward(dout)
    return dict(bench="channel", world=world, ms_per_step=time_ms(step, args.steps, args.warmup))


def model_bench(rank, world, args, dev):
    torch.manual_seed(0)
    m = Mamba(MambaConfig(d_model=512, n_layers=4)).to(dev)
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.randn(1, L, 512, generator=g).to(dev)
    lo, hi = par.shard_range(L, rank, world)
    xl = par.shard_sequence(x, rank, world).contiguous()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        y_ref = m(x)[:, lo:hi].float()
        y = par.sequence_sharded_forward(m, xl).float()
    err = rel(y, y_ref)
    del y_ref
    ok = err < 2e-2
    res = dict(bench="model", world=world, d_model=512, n_layers=4, L=L, dtype="bf16 autocast", parity_ok=ok, parity_max_rel=err)
    if not ok:
        raise SystemExit(f"rank {rank}: model parity failed {err}")

    def step():
        m.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = par.sequence_sharded_forward(m, xl)
        (y.float().square().sum() / L).backward()
        par.allreduce_gradients(m.parameters(), average=False)
    res["ms_per_step"] = time_ms(step, max(1, args.steps // 4), max(1, args.warmup))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    info = device_info()

    def out(r):
        if rank == 0:
            line = json.dumps(dict(r, device=info))
            print(line, flush=True)
            if args.out:
                with open(args.out, "a") as f:
                    f.write(line + "\n")
    try:
        d = scan_inputs(dev)
        out(scan_bench(d, rank, world, args, out))
        out(channel_bench(d, rank, world, args))
        del d
        torch.cuda.empty_cache()
        out(model_bench(rank, world, args, dev))
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
