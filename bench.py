#!/usr/bin/env python
"""bench.py -- selective-scan fwd+bwd throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one fused selective-scan forward + backward (the hot path of cross_atten/mamba.py:227-286 with
softplus, D skip and SiLU gate) over one batch of synthetic tensors of the named workload, through the public
API (gfe_mamba_b200.selective_scan_fn -> ctypes -> C ABI).  Default workload: BASELINE.json configs[2]
("cfg3": B=16 per GPU, L=4096, d_model=768 -> ED=1536, N=16, bf16), the shape the metric and the >=60 %-of-HBM
target are quoted on.  Weak scaling: every rank processes its own batch (batch sharding, no data-path
collective); for N > 1 the A_log/D/dt_bias gradients are all-reduced over NCCL each step, as in training.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definition of every field.

--dump-outputs DIR: after the timed steps, rank 0 writes what its last timed step returned -- out and the gradients of
every input and parameter (under N GPUs the all-reduced sums the step receives) -- as DIR/<name>.npy in float32.  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (B per GPU, L, d_model, dtype)        ED = 2 * d_model, N = 16
    "cfg1": (8, 64, 128, "f32"),
    "cfg2": (32, 256, 256, "f32"),
    "cfg3": (16, 4096, 768, "bf16"),
    "cfg4": (1, 65536, 512, "f32"),
    "cfg5": (256, 1024, 512, "f32"),
    "prod": (2, 1858, 512, "f32"),
}
N_STATE = 16


def algorithmic_bytes(B, L, ED, s):
    """SURVEY 8d: fwd reads u, delta, z (3 ED) + B, C (2 N), writes out (ED); bwd reads u, delta, z, dout (4 ED) +
    B, C (2 N), writes du, ddelta, dz (3 ED) + dB, dC (2 N).  Per token, activation size s bytes."""
    fwd = (4 * ED + 2 * N_STATE) * s
    bwd = (7 * ED + 4 * N_STATE) * s
    return B * L * fwd, B * L * bwd


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


KERNEL_SOURCES = ("selscan_v4_fwd.cu", "selscan_chain_bwd.cu", "selscan_chain_host.cu", "selscan_shared.cuh", "selscan.cu",
                  "selscan_seg.cu", "common.cuh")


def kernel_source_hash():
    """Fingerprint of the scan-kernel sources; tools/ncu_traffic.py stores it with every capture so that a capture taken
    from other kernels than the ones being benchmarked is recognised as stale instead of being quoted."""
    import hashlib
    h = hashlib.sha256()
    for name in KERNEL_SOURCES:
        try:
            with open(os.path.join(ROOT, "gfe_mamba_b200", "csrc", name), "rb") as f:
                h.update(f.read())
        except OSError:
            h.update(name.encode())
    return h.hexdigest()[:16]


def measured_traffic(workload, kernel, B):
    """(bytes, note): dram__bytes_read.sum + dram__bytes_write.sum of one launch of `kernel`, from the committed
    `ncu --set full` capture of this workload (profiles/traffic.json, written by tools/ncu_traffic.py).  None when no capture
    exists for it or when the capture was taken from different kernel sources (stale)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            rec = json.load(f)[workload]
    except Exception:
        return None, "no ncu capture for this workload"
    if rec.get("batch_per_gpu") != B:
        return None, "capture is for another batch size"
    if rec.get("source_hash") != kernel_source_hash():
        print(f"bench.py: WARNING profiles/traffic.json[{workload}] was captured from other kernel sources "
              f"({rec.get('source_hash')} != {kernel_source_hash()}): not quoted; re-run tools/gpu_check.sh", file=sys.stderr)
        return None, "stale capture (kernel sources changed since); ignored"
    try:
        return int(rec["kernels"][kernel]), rec.get("source", "")
    except Exception:
        return None, "kernel not in the capture"


OUTPUT_NAMES = ("out", "du", "ddelta", "dz", "dB", "dC", "dA_log", "dD", "ddt_bias")
DUMP_SAMPLE = 1 << 20   # elements kept of a larger output: nine float32 arrays of at most 4 MiB each, under 64 MB in all


def step_outputs(out, grads, flat, by_channels):
    """{name: tensor} of what one step hands its caller.  Under N GPUs the all-reduced sums in `flat` stand for the rank's
    own dB, dC (channel sharding) or parameter gradients (batch sharding)."""
    grads = list(grads)
    if flat is not None:
        i = slice(3, 5) if by_channels else slice(5, None)
        grads[i] = [p.view_as(g) for p, g in zip(flat.split([g.numel() for g in grads[i]]), grads[i])]
    return dict(zip(OUTPUT_NAMES, [out] + grads))


def dump_outputs(path, arrays):
    """Writes every array as path/<name>.npy in float32.  An array of more than DUMP_SAMPLE elements is reduced to its
    elements at DUMP_SAMPLE distinct flat indices drawn by numpy.random.default_rng(0), in increasing order: the same
    indices in every run of the same shape."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach()
        if a.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(a.numel(), DUMP_SAMPLE, replace=False))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(path, name + ".npy"), a.float().cpu().numpy())


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)   # the sampler never outlives the benchmark, even one that fails before stop()
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx = max(mx, float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------- reference arm
def cpu_reference(B, L, ED, steps, warmup, budget_s):
    """The reference's CPU algorithm for this path -- MambaBlock.selective_scan with the Blelloch pscan and its
    custom backward, all (B,L,ED,N) tensors materialised (oracle/gfe_oracle.c: orc_selscan_ref_fwd/bwd, the port of
    mamba.py:265-286 + pscan.py:37-224) -- on the host cores, on a bounded sample: one batch row, full ED, a
    power-of-two number of tokens chosen so that steps+warmup samples fit the time budget."""
    import numpy as np
    from oracle import oracle as orc
    cores = os.cpu_count() or 1
    orc.set_num_threads(cores)
    rng = np.random.default_rng(1234)

    def make(Ls):
        f = lambda *s: rng.standard_normal(s).astype(np.float32)
        x, dy = f(1, Ls, ED), f(1, Ls, ED)
        delta = np.log1p(np.exp(0.5 * f(1, Ls, ED) - 4.0)).astype(np.float32)
        A = -np.exp(np.log(np.arange(1, N_STATE + 1, dtype=np.float32))[None].repeat(ED, 0) + 0.1 * f(ED, N_STATE))
        return x, delta, A.astype(np.float32), f(1, Ls, N_STATE), f(1, Ls, N_STATE), (1 + 0.1 * f(ED)).astype(np.float32), dy

    def one(args):
        t0 = time.perf_counter()
        orc.selscan_ref_fwd(*args[:6])
        orc.selscan_ref_bwd(*args)
        return time.perf_counter() - t0

    Ls = min(L, 256)
    t = one(make(Ls))                                     # calibration
    per_tok = t / Ls
    want = budget_s / max(1, steps + warmup) / per_tok
    while Ls * 2 <= min(L, want):
        Ls *= 2
    args = make(Ls)
    for _ in range(warmup):
        one(args)
    times = [one(args) for _ in range(steps)]
    dt = sum(times) / len(times)
    return {"tokens_per_s": Ls / dt, "ms_per_step": dt * 1e3, "cores": orc.num_threads(), "sample_tokens": Ls,
            "sample": f"B=1 of {B}, L={Ls} of {L} (power of two, reference pads to npo2 anyway), full ED={ED}, fp32, "
                      f"fwd+bwd, {steps} timed samples; tokens/s is flat in B and L (BASELINE.md section 2)"}


# ------------------------------------------------------------------------- multi-GPU correctness, visible in the JSON line
def sharded_parity_check(dist, dev, rank, world, by_channels):
    """Before timing, every rank runs ITS shard of one small shared problem through the same code path the timed loop uses
    (batch rows, or ED channels with the dB/dC all-reduce); the shards are gathered and rank 0 compares them with the whole
    problem computed on one GPU.  Returns {"mode", "max_rel_err", "tol", "ok"} (max-normalised error over out and every
    gradient); raises on failure so that a wrong multi-GPU number is never printed."""
    import torch
    from gfe_mamba_b200 import selective_scan_fn
    from gfe_mamba_b200.parallel import channel_sharded_scan, shard_batch, shard_channels
    Bp, Lp, EDp = 2 * world, 200, 64 * world
    g = torch.Generator(device=dev).manual_seed(99)          # same seed on every rank: one shared problem
    rn = lambda *s: torch.randn(*s, device=dev, generator=g)
    full = dict(u=rn(Bp, Lp, EDp), delta=rn(Bp, Lp, EDp) * 0.5, z=rn(Bp, Lp, EDp), Bm=rn(Bp, Lp, N_STATE), Cm=rn(Bp, Lp, N_STATE),
                dout=rn(Bp, Lp, EDp))
    A_log = torch.log(torch.arange(1, N_STATE + 1, device=dev).float()).repeat(EDp, 1) + 0.1 * rn(EDp, N_STATE)
    Dp = 1 + 0.1 * rn(EDp)
    bias = rn(EDp) * 0.3 - 3.0

    def run(u, delta, z, Bm, Cm, dout, A, D, b, sharded):
        lv = [t.clone().requires_grad_() for t in (u, delta, z, Bm, Cm, A, D, b)]
        if sharded and by_channels:
            out = channel_sharded_scan(selective_scan_fn, lv[0], lv[1], lv[5], lv[3], lv[4], lv[6], z=lv[2], dt_bias=lv[7])
        else:
            out = selective_scan_fn(lv[0], lv[1], lv[5], lv[3], lv[4], lv[6], z=lv[2], dt_bias=lv[7])
        grads = torch.autograd.grad(out, lv, dout)
        return [out.detach()] + [x.detach() for x in grads]

    if by_channels:
        ch = lambda t: shard_channels(t, rank, world).contiguous()
        mine = run(ch(full["u"]), ch(full["delta"]), ch(full["z"]), full["Bm"], full["Cm"], ch(full["dout"]),
                   shard_channels(A_log, rank, world, dim=0).contiguous(), ch(Dp), ch(bias), True)
        cat_dim = {0: 2, 1: 2, 2: 2, 3: 2, 4: None, 5: None, 6: 0, 7: 0, 8: 0}       # dB/dC are already all-reduced
    else:
        sb = lambda t: shard_batch(t, rank, world).contiguous()
        mine = run(sb(full["u"]), sb(full["delta"]), sb(full["z"]), sb(full["Bm"]), sb(full["Cm"]), sb(full["dout"]), A_log, Dp, bias, True)
        for t in mine[6:]:                                                           # parameter gradients: summed over ranks
            dist.all_reduce(t)
        cat_dim = {0: 0, 1: 0, 2: 0, 3: 0, 4: 0, 5: 0, 6: None, 7: None, 8: None}
    gathered = []
    for i, t in enumerate(mine):
        if cat_dim[i] is None:
            gathered.append(t)
        else:
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t.contiguous())
            gathered.append(torch.cat(parts, dim=cat_dim[i]))
    res = None
    if rank == 0:
        want = run(full["u"], full["delta"], full["z"], full["Bm"], full["Cm"], full["dout"], A_log, Dp, bias, False)
        err = max(float((a.detach().float() - b.detach().float()).abs().max() / b.detach().float().abs().max().clamp_min(1e-30)) for a, b in zip(gathered, want))
        res = {"mode": "channels" if by_channels else "batch", "shape": [Bp, Lp, EDp], "max_rel_err": err, "tol": 1e-4, "ok": err < 1e-4}
    flag = torch.tensor([1 if (res is None or res["ok"]) else 0], device=dev)
    dist.broadcast(flag, 0)
    if int(flag.item()) != 1:
        raise SystemExit(f"bench.py: sharded result differs from the single-GPU result: {res}")
    return res


# ------------------------------------------------------------------------------------------------ main
def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner at init), so the
    real stdout is set aside for the JSON line and file descriptor 1 is pointed at stderr for everything else."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    out_stream = _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default=None, choices=[None, "f32", "bf16", "f16"])
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--e2e-rows", type=int, default=0, help="batch rows per pipeline chunk of the e2e leg (0 = B/8)")
    ap.add_argument("--batch", type=int, default=0, help="override the workload's per-GPU batch (A/B measurements)")
    ap.add_argument("--shard", default="batch", choices=["batch", "channels"],
                    help="N > 1: batch = every rank its own B rows (weak scaling); channels = ONE batch, rank g owns ED/N channels, "
                         "dB/dC all-reduced every step (strong scaling; BASELINE config 4)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not bind the process to the GPU's NUMA node for the e2e leg")
    ap.add_argument("--cpu-budget-s", type=float, default=25.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32; seeded sample of a large output)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    B, L, d_model, dts = WORKLOADS[args.workload]
    B = args.batch or B
    dts = args.dtype or dts
    ED_full = 2 * d_model
    by_channels = args.shard == "channels" and world > 1
    if by_channels and ED_full % (32 * world) != 0:
        raise SystemExit(f"bench.py: ED={ED_full} does not split into {world} channel shards of a multiple of 32")
    ED = ED_full // world if by_channels else ED_full      # channels THIS rank scans
    s_bytes = 4 if dts == "f32" else 2
    cfg = {"workload": f"{args.workload}: fused selective scan fwd+bwd, B={B}/GPU, L={L}, d_model={d_model}, ED={ED}, N={N_STATE}",
           "batch_per_gpu": B, "seq_len": L, "d_inner": ED, "d_state": N_STATE,
           "sharding": (f"channels x{world} (ED/{world} = {ED} per GPU, one batch, dB/dC all-reduced)" if by_channels
                        else f"batch x{world}" if world > 1 else "single GPU"),
           "l2_policy": "inputs larger than L2" if 4 * B * L * ED * s_bytes > 2 * 126e6 else "rotating input sets + L2 flush"}
    warmup = max(args.warmup, 3)

    if args.impl == "reference":
        if rank != 0:
            return
        r = cpu_reference(B, L, ED, args.steps, warmup, budget_s=150.0)
        line = {"impl": "reference", "metric": "selective-scan fwd+bwd tokens/s", "value": r["tokens_per_s"], "unit": "tokens/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": cfg,
                "cpu_baseline": {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": r["tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line), file=out_stream, flush=True)
        return

    import torch
    import torch.distributed as dist
    from gfe_mamba_b200 import selective_scan_fn
    from gfe_mamba_b200 import _native

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    _native.lib()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[dts]

    # ---- synthetic inputs (SURVEY 8d), resident in HBM; small workloads rotate over several sets + flush L2
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    gen_shared = torch.Generator(device=dev).manual_seed(4321)   # B and C are replicated under channel sharding
    per_set = (4 * B * L * ED + 2 * B * L * N_STATE) * s_bytes
    nsets = 1 if per_set > 2 * 126e6 else min(8, int(4 * 126e6 // per_set) + 2)

    def make_set():
        rn = lambda *s: torch.randn(*s, device=dev, generator=gen)
        rs = (lambda *s: torch.randn(*s, device=dev, generator=gen_shared)) if by_channels else rn
        return dict(u=rn(B, L, ED).to(dt).requires_grad_(), delta=(rn(B, L, ED) * 0.5).to(dt).requires_grad_(),
                    z=rn(B, L, ED).to(dt).requires_grad_(), Bm=rs(B, L, N_STATE).to(dt).requires_grad_(),
                    Cm=rs(B, L, N_STATE).to(dt).requires_grad_(), dout=rn(B, L, ED).to(dt))

    sets = [make_set() for _ in range(nsets)]
    A_log = (torch.log(torch.arange(1, N_STATE + 1, device=dev).float()).repeat(ED, 1) + 0.1 * torch.randn(ED, N_STATE, device=dev, generator=gen)).requires_grad_()
    D = (1 + 0.1 * torch.randn(ED, device=dev, generator=gen)).requires_grad_()
    dtv = torch.exp(torch.rand(ED, device=dev, generator=gen) * (torch.log(torch.tensor(0.1)) - torch.log(torch.tensor(0.001))) + torch.log(torch.tensor(0.001))).clamp(min=1e-4)
    bias = (dtv + torch.log(-torch.expm1(-dtv))).requires_grad_()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if nsets > 1 else None

    def step(i):
        d = sets[i % nsets]
        out = selective_scan_fn(d["u"], d["delta"], A_log, d["Bm"], d["Cm"], D, z=d["z"], dt_bias=bias)
        grads = torch.autograd.grad(out, (d["u"], d["delta"], d["z"], d["Bm"], d["Cm"], A_log, D, bias), d["dout"])
        flat = None
        if by_channels:   # channel sharding: dB, dC sum over every rank's channels (2 B L N values); parameters are local
            flat = torch.cat([grads[3].reshape(-1), grads[4].reshape(-1)]).float()
            dist.all_reduce(flat)
        elif world > 1:   # data-parallel training: all-reduce the (tiny) parameter gradients
            flat = torch.cat([g.reshape(-1) for g in grads[5:]])
            dist.all_reduce(flat)
        return out, grads, flat

    last = []   # what the last timed step returned; earlier steps' results are released at once, as in the warm-up

    def timed_step(i):
        r = step(i)
        if i == args.steps - 1:
            last.append(r)

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    parity = sharded_parity_check(dist, dev, rank, world, by_channels) if world > 1 else None

    for i in range(warmup):
        step(i)
    sync_all()

    # ---- timed region: K steps, CUDA events, per-kernel device timing from the library, clocks sampled
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    _native.timing_enable(True)
    _native.timing_collect()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    if flush is None:
        e0.record()
        for i in range(args.steps):
            timed_step(i)
        e1.record()
        sync_all()
        elapsed_ms = e0.elapsed_time(e1)
    else:   # small workload: flush L2 between steps, time each step separately
        elapsed_ms = 0.0
        for i in range(args.steps):
            flush.fill_(i & 0xFF)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            timed_step(i)
            b.record()
            torch.cuda.synchronize(dev)
            elapsed_ms += a.elapsed_time(b)
        sync_all()
    kern = _native.timing_collect()
    _native.timing_enable(False)
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    # the step's collective alone (nothing to overlap with), reported next to the step: dB|dC under channel sharding, the
    # parameter-gradient bucket under batch sharding
    allreduce_ms = None
    if world > 1:
        n_el = 2 * B * L * N_STATE if by_channels else ED * N_STATE + 2 * ED
        buf = torch.zeros(n_el, device=dev, dtype=torch.float32)
        for _ in range(3):
            dist.all_reduce(buf)
        sync_all()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(20):
            dist.all_reduce(buf)
        a1.record()
        sync_all()
        t = torch.tensor([a0.elapsed_time(a1) / 20], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        allreduce_ms = {"ms": round(float(t.item()), 4), "bytes": 4 * n_el, "what": "dB|dC (fp32)" if by_channels else "A_log, D, dt_bias gradients (fp32)"}
    tokens_per_s = (1 if by_channels else world) * B * L / (ms_per_step * 1e-3)   # channel sharding: ONE batch of tokens

    # ---- roofline of the dominant kernel + every kernel's share
    peak, peak_src = measured_peaks()
    fwd_b, bwd_b = algorithmic_bytes(B, L, ED, s_bytes)
    kern_list, total_kernel_ms = [], sum(v[0] for v in kern.values())
    for name, (ms, cnt) in sorted(kern.items(), key=lambda kv: -kv[1][0]):
        alg = {"selscan_fwd": fwd_b, "selscan_bwd": bwd_b}.get(name)
        avg = ms / cnt
        kern_list.append({"kernel": name, "launches": int(cnt), "avg_ms": round(avg, 4), "share": round(ms / total_kernel_ms, 4),
                          "algorithmic_GBps": None if alg is None else round(alg / (avg * 1e-3) / 1e9, 1)})
    dom = kern_list[0]
    dom_alg = {"selscan_fwd": fwd_b, "selscan_bwd": bwd_b}.get(dom["kernel"], fwd_b + bwd_b)
    achieved = dom_alg / (dom["avg_ms"] * 1e-3) / 1e9
    traffic, traffic_note = measured_traffic(args.workload, dom["kernel"], B)
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_note, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": dom_alg,
                "step_achieved": round((fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9, 1),
                "step_frac": round((fwd_b + bwd_b) / (ms_per_step * 1e-3) / 1e9 / peak, 4),
                "note": "selective scan at N=16 is bound by MUFU + FP32 operand delivery on B200, not by HBM (DESIGN.md section 4)"}
    gpu_launches = int(sum(v[1] for v in kern.values()))

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_outputs(*last[0], by_channels))
    last.clear()

    # ---- e2e: the same step through the public host-buffer API (gfe_mamba_b200.host_pipeline.HostScanPipeline): pinned HOST
    #      inputs -> H2D, fused fwd+bwd, D2H of out and every activation gradient into pinned HOST outputs, all inside the
    #      timed region; the pipeline overlaps the three over row chunks of the batch.
    from gfe_mamba_b200.host_pipeline import HostScanPipeline, bind_host_to_gpu_node
    orig_affinity = os.sched_getaffinity(0)
    numa_cpus = bind_host_to_gpu_node(dev) if not args.no_numa_bind else None   # pinned buffers below land on the GPU's node
    d0 = sets[0]
    host_in = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in d0.items()}
    for k, v in d0.items():
        host_in[k].copy_(v.detach())
    host_out = {k: torch.empty((B, L, N_STATE if k in ("dBm", "dCm") else ED), dtype=dt).pin_memory()
                for k in ("out", "du", "ddelta", "dz", "dBm", "dCm")}
    del sets, d0
    torch.cuda.empty_cache()
    pipe = HostScanPipeline(B, L, ED, N_STATE, dt, dev, rows_per_chunk=args.e2e_rows or None, has_z=True)

    def e2e_step():
        g = pipe.run(host_in, A_log.detach(), D.detach(), bias.detach(), host_out)
        torch.cuda.current_stream().synchronize()
        return g

    e2e_step()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    sync_all()
    e2e_s = (time.perf_counter() - t0) / args.e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": (1 if by_channels else world) * B * L / e2e_s, "unit": "tokens/s", "h2d_bytes_per_step": pipe.h2d_bytes, "d2h_bytes_per_step": pipe.d2h_bytes,
           "ms_per_step": round(e2e_s * 1e3, 3), "steps": args.e2e_steps, "rows_per_chunk": pipe.rows, "host_cpus": numa_cpus,
           "api": "gfe_mamba_b200.host_pipeline.HostScanPipeline.run (pinned host in/out, H2D | fwd+bwd | D2H overlapped over row chunks)"}

    os.sched_setaffinity(0, orig_affinity)   # the CPU baseline below uses every host core again

    # ---- CPU baseline beside the GPU number (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_reference(B, L, ED, steps=2, warmup=1, budget_s=args.cpu_budget_s)
        cpu = {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}

    if rank == 0:
        line = {"metric": "selective-scan fwd+bwd tokens/s", "value": tokens_per_s, "unit": "tokens/s", "n_gpus": world,
                "steps": args.steps, "warmup": warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
                "scaling": "strong" if by_channels else "weak", "vs_baseline": None, "dtype": dts, "data": "synthetic", "config": cfg,
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": gpu_launches, "clocks": clocks,
                "kernels": kern_list}
        if parity is not None:
            line["parity_check"] = parity
        if allreduce_ms is not None:
            line["allreduce"] = allreduce_ms
        print(json.dumps(line), file=out_stream, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True   # the benchmark leaves the tree as the build left it (it may be read-only)
    main()
