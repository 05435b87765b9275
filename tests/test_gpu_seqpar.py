"""Sequence sharding on the GPU.

* The summary entry points (ops.selscan_summary / selscan_summary_rev) against fp64 references: h_loc against the final state
  of a scan from zero, sum_delta against sum softplus(delta + b), g_loc against the d h0 of selective_scan_state's backward
  with no final-state gradient and against its fp64 closed form.  Both kernel families (the chained one serves d_state 16 with
  ED % 32 == 0, the generic one everything else), every N x dtype x gate x step-size flag, strided B / C slices of x_proj's
  output, small B * ED (L split) and large, L from 1 to past one segment, and long-memory channels per channel.
* Ranks emulated in one process: a sequence cut into P uneven pieces, each run as a rank would (summary, combine, scan from
  the carry; reverse summary, reverse combine, backward from dlast), against one pass over the whole sequence.  The same for
  the conv window.
* Two GPUs (NCCL, skipped below two): sequence_sharded_scan and sequence_sharded_forward against one GPU; one rank (no
  process group) runs Mamba.forward's kernels.
"""
import copy
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gfe_mamba_b200 import Mamba, MambaConfig, ops
from gfe_mamba_b200 import parallel as par

pytestmark = pytest.mark.gpu
DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


def _chained(N, ED):
    return N == 16 and ED % 32 == 0


def _inputs(B, L, ED, N, dtype, seed, gate=True, bias=True, softplus=True, strided=False, bias_range=None):
    g = torch.Generator(device="cpu").manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g)
    R = 8
    d = dict(u=rn(B, L, ED), z=rn(B, L, ED) if gate else None, dout=rn(B, L, ED),
             A_log=torch.log(torch.arange(1, N + 1).float()).repeat(ED, 1) + 0.1 * rn(ED, N))
    d["delta"] = 0.5 * rn(B, L, ED) if softplus else 0.02 + 0.1 * torch.rand(B, L, ED, generator=g)
    if bias_range is not None:
        d["bias"] = torch.linspace(*bias_range, ED)
    else:
        d["bias"] = (-4 + rn(ED)) if (bias and softplus) else (0.01 * torch.rand(ED, generator=g) if bias else None)
    if strided:   # B and C as slices of one (B, L, R + 2N) tensor, like x_proj's output
        dbc = rn(B, L, R + 2 * N).cuda().to(dtype)
        d["Bm"], d["Cm"] = dbc[..., R:R + N], dbc[..., R + N:]
    else:
        d["Bm"], d["Cm"] = rn(B, L, N), rn(B, L, N)
    out = {}
    for k, v in d.items():
        if v is None or k in ("A_log", "bias"):
            out[k] = None if v is None else v.cuda()
        else:
            out[k] = v.cuda().to(dtype)
    return out


def _step(d, softplus):
    x = d["delta"].double() + (0 if d["bias"] is None else d["bias"].double())
    return torch.nn.functional.softplus(x) if softplus else x


def _ref_summaries(d, softplus):
    """fp64: h_loc = sum_t exp(A sum_{s>t} dl_s) dl_t u_t B_t; g_loc = sum_t exp(A sum_{s<=t} dl_s) C_t dy_t."""
    dl = _step(d, softplus)                                       # (B, L, ED)
    A = -torch.exp(d["A_log"].double())                           # (ED, N)
    incl = torch.cumsum(dl, 1)
    after = incl[:, -1:] - incl                                   # sum over s > t
    h = torch.einsum("bten,bte,btn->ben", torch.exp(after.unsqueeze(-1) * A), dl * d["u"].double(), d["Bm"].double())
    dy = d["dout"].double()
    if d["z"] is not None:
        z = d["z"].double()
        dy = dy * z * torch.sigmoid(z)
    g = torch.einsum("bten,bte,btn->ben", torch.exp(incl.unsqueeze(-1) * A), dy, d["Cm"].double())
    return h, dl.sum(1), g


def _kernel_dh0(d, softplus):
    leaves = {k: d[k].detach().clone().requires_grad_() for k in ("u", "delta")}
    h0 = torch.zeros(d["u"].shape[0], d["u"].shape[2], d["A_log"].shape[1], device="cuda", requires_grad=True)
    D = torch.ones(d["u"].shape[2], device="cuda")
    out, _ = ops.selective_scan_state(leaves["u"], leaves["delta"], d["A_log"], d["Bm"], d["Cm"], D, h0, z=d["z"],
                                      dt_bias=d["bias"], delta_softplus=softplus)
    out.backward(d["dout"])
    return h0.grad


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _per_channel(got, want, axis):
    g, w = got.double().movedim(axis, 0).flatten(1), want.double().movedim(axis, 0).flatten(1)
    return ((g - w).abs().amax(1) / w.abs().amax(1).clamp_min(1e-30)).max().item()


def _check_summaries(d, softplus, tol=1e-4):
    h_loc, sd = ops.selscan_summary(d["u"], d["delta"], d["A_log"], d["Bm"], dt_bias=d["bias"], delta_softplus=softplus)
    g_loc = ops.selscan_summary_rev(d["dout"], d["delta"], d["A_log"], d["Cm"], z=d["z"], dt_bias=d["bias"],
                                    delta_softplus=softplus)
    h_ref, sd_ref, g_ref = _ref_summaries(d, softplus)
    errs = dict(h_loc=_rel(h_loc, h_ref), sum_delta=_rel(sd, sd_ref), g_loc=_rel(g_loc, g_ref),
                g_loc_vs_dh0=_rel(g_loc, _kernel_dh0(d, softplus)))
    assert max(errs.values()) < tol, errs
    return h_loc, sd, g_loc


@pytest.mark.parametrize("N", [16, 32, 64])
@pytest.mark.parametrize("dt", ["f32", "bf16", "f16"])
@pytest.mark.parametrize("gate", [True, False])
@pytest.mark.parametrize("flag", ["softplus_bias", "plain"])
def test_summaries_match_fp64(N, dt, gate, flag):
    sp = flag == "softplus_bias"
    d = _inputs(1, 2100, 256, N, DT[dt], seed=N + len(dt), gate=gate, bias=sp, softplus=sp)
    _check_summaries(d, sp)


@pytest.mark.parametrize("N,ED", [(16, 256), (16, 80), (32, 256), (64, 96)])
@pytest.mark.parametrize("L", [1, 15, 129, 2100])
def test_summaries_shapes_and_lengths(N, ED, L):
    """Both families (N = 16 with ED % 32 == 0 chained, the rest generic), L from one token to many segments."""
    _check_summaries(_inputs(2, L, ED, N, torch.float32, seed=L + ED), True)


@pytest.mark.parametrize("N,ED", [(16, 1536), (32, 1536)])
def test_summaries_large_batch_no_split(N, ED):
    """B * ED large enough that the main passes do not split L."""
    _check_summaries(_inputs(8, 300, ED, N, torch.bfloat16, seed=5), True)


@pytest.mark.parametrize("N,ED", [(16, 256), (32, 256), (16, 80)])
@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_summaries_strided_bc(N, ED, dt):
    d = _inputs(2, 700, ED, N, DT[dt], seed=3, strided=True)
    assert d["Bm"].stride(1) != N
    _check_summaries(d, True)


@pytest.mark.parametrize("N,ED", [(16, 256), (32, 128), (64, 64)])
def test_summaries_long_memory_per_channel(N, ED):
    """dt_bias in [-16, -4] across channels: step sizes down to ~1e-7; errors per channel, fp32."""
    d = _inputs(1, 3000, ED, N, torch.float32, seed=11, bias_range=(-16.0, -4.0))
    h_loc, sd = ops.selscan_summary(d["u"], d["delta"], d["A_log"], d["Bm"], dt_bias=d["bias"])
    g_loc = ops.selscan_summary_rev(d["dout"], d["delta"], d["A_log"], d["Cm"], z=d["z"], dt_bias=d["bias"])
    h_ref, sd_ref, g_ref = _ref_summaries(d, True)
    errs = dict(h_loc=_per_channel(h_loc, h_ref, 1), sum_delta=_per_channel(sd, sd_ref, 1), g_loc=_per_channel(g_loc, g_ref, 1))
    assert max(errs.values()) < 1e-3, errs


def test_summary_argument_errors():
    d = _inputs(1, 64, 256, 16, torch.float32, seed=1)
    with pytest.raises(RuntimeError, match="inference-only"):
        ops.selscan_summary(d["u"].requires_grad_(), d["delta"], d["A_log"], d["Bm"])
    with pytest.raises(ValueError):
        ops.selscan_summary(d["u"].detach(), d["delta"], d["A_log"], d["Cm"][:, :10])
    with pytest.raises(RuntimeError, match="d_state"):
        ops.selscan_summary(d["u"].detach(), d["delta"], d["A_log"][:, :8].contiguous(), d["Bm"][..., :8])


# ------------------------------------------------------------------------------------ ranks emulated in one process
def _cuts(L, P):
    g = np.random.default_rng(P)
    w = g.uniform(0.5, 1.5, P)
    edges = np.round(np.cumsum(w) / w.sum() * L).astype(int)
    return [0] + [int(e) for e in edges[:-1]] + [L]


@pytest.mark.parametrize("P", [2, 3, 8])
@pytest.mark.parametrize("N,ED", [(16, 256), (32, 96)])
@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_emulated_ranks_scan(P, N, ED, dt):
    B, L = 2, 1500
    d = _inputs(B, L, ED, N, DT[dt], seed=P * 7 + N)
    names = ("u", "delta", "z", "Bm", "Cm")
    full = {k: d[k].clone().requires_grad_() for k in names}
    par_ = {k: torch.nn.Parameter(v.clone()) for k, v in (("A_log", d["A_log"]), ("D", 1 + 0.1 * d["A_log"][:, 0]), ("bias", d["bias"]))}
    ref = ops.selective_scan_fn(full["u"], full["delta"], par_["A_log"], full["Bm"], full["Cm"], par_["D"], z=full["z"],
                                dt_bias=par_["bias"])
    ref.backward(d["dout"])
    ref_g = {k: v.grad.clone() for k, v in list(full.items()) + list(par_.items())}
    for v in list(full.values()) + list(par_.values()):
        v.grad = None
    cuts = _cuts(L, P)
    pieces = [{k: full[k][:, lo:hi] for k in names} | {"dout": d["dout"][:, lo:hi]} for lo, hi in zip(cuts, cuts[1:])]
    with torch.no_grad():
        s = [ops.selscan_summary(p["u"], p["delta"], par_["A_log"], p["Bm"], dt_bias=par_["bias"]) for p in pieces]
        h_all, sd_all = torch.stack([x[0] for x in s]), torch.stack([x[1] for x in s])
        g_all = torch.stack([ops.selscan_summary_rev(p["dout"], p["delta"], par_["A_log"], p["Cm"], z=p["z"], dt_bias=par_["bias"])
                             for p in pieces])
    outs = []
    for r, p in enumerate(pieces):
        h_in = par.sequence_carry_in(h_all, sd_all, par_["A_log"], r) if r > 0 else None
        out, h_last = ops.selective_scan_state(p["u"], p["delta"], par_["A_log"], p["Bm"], p["Cm"], par_["D"], h_in, z=p["z"],
                                               dt_bias=par_["bias"])
        dlast = par.sequence_dlast(g_all, sd_all, par_["A_log"], r)
        torch.autograd.backward([out, h_last], [p["dout"], dlast])
        outs.append(out.detach())
    tol = 1e-4 if dt == "f32" else 2e-2
    errs = {"out": _rel(torch.cat(outs, 1), ref)}
    errs.update({k: _rel(v.grad, ref_g[k]) for k, v in list(full.items()) + list(par_.items())})
    assert max(errs.values()) < tol, errs


@pytest.mark.parametrize("P", [2, 3, 8])
@pytest.mark.parametrize("K", [2, 4])
@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_emulated_ranks_conv(P, K, dt):
    B, L, ED = 2, 600, 128
    g = torch.Generator(device="cpu").manual_seed(P + K)
    xin = torch.randn(B, L, ED, generator=g).cuda().to(DT[dt]).requires_grad_()
    w = torch.nn.Parameter(0.5 * torch.randn(ED, 1, K, generator=g).cuda())
    b = torch.nn.Parameter(0.1 * torch.randn(ED, generator=g).cuda())
    du = torch.randn(B, L, ED, generator=g).cuda().to(DT[dt])
    ref = ops.causal_conv1d_silu(xin, w, b)
    ref.backward(du)
    ref_g = [t.grad.clone() for t in (xin, w, b)]
    for t in (xin, w, b):
        t.grad = None
    cuts = _cuts(L, P)
    outs = []
    for lo, hi in zip(cuts, cuts[1:]):
        window = xin[:, lo - (K - 1):lo].transpose(1, 2) if lo > 0 else None   # the previous rank's last K-1 rows
        u, _ = ops.causal_conv1d_silu_state(xin[:, lo:hi], window, w, b)
        u.backward(du[:, lo:hi])
        outs.append(u.detach())
    tol = 1e-4 if dt == "f32" else 2e-2
    errs = dict(u=_rel(torch.cat(outs, 1), ref), dx=_rel(xin.grad, ref_g[0]), dw=_rel(w.grad, ref_g[1]), db=_rel(b.grad, ref_g[2]))
    assert max(errs.values()) < tol, errs


def test_world_one_is_mamba_forward():
    torch.manual_seed(0)
    for cfg in (MambaConfig(d_model=64, n_layers=2), MambaConfig(d_model=64, n_layers=2, d_state=32, d_conv=3)):
        m = Mamba(cfg).cuda()
        x = torch.randn(2, 300, 64, device="cuda")
        y_ref = m(x)
        y_ref.square().sum().backward()
        g_ref = {n: p.grad.clone() for n, p in m.named_parameters()}
        m.zero_grad(set_to_none=True)
        y = par.sequence_sharded_forward(m, x)
        y.square().sum().backward()
        assert _rel(y, y_ref) < 1e-6
        for n, p in m.named_parameters():
            assert _rel(p.grad, g_ref[n]) < 1e-5, n


def test_unsupported_config_raises():
    m = Mamba(MambaConfig(d_model=32, n_layers=1, d_state=8)).cuda()
    with pytest.raises(ValueError):
        par.sequence_sharded_forward(m, torch.randn(1, 16, 32, device="cuda"))


# ------------------------------------------------------------------------------------------------ two GPUs
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, mode):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        if mode.startswith("scan"):
            _scan_case(rank, world, dev, mode)
        else:
            _model_case(rank, world, dev, mode)
    finally:
        dist.destroy_process_group()


def _scan_case(rank, world, dev, mode):
    dt = torch.bfloat16 if "bf16" in mode else torch.float32
    with_h0 = "h0" in mode
    B, L, ED, N = 2, 1000, 256, 16
    torch.cuda.set_device(dev)
    d = _inputs(B, L, ED, N, dt, seed=21)
    names = ("u", "delta", "z", "Bm", "Cm")
    h0 = (0.3 * torch.randn(B, ED, N, generator=torch.Generator().manual_seed(2))).cuda() if with_h0 else None

    def params():
        return {k: torch.nn.Parameter(v.clone()) for k, v in (("A_log", d["A_log"]), ("D", 1 + 0.1 * d["A_log"][:, 0]),
                                                               ("bias", d["bias"]))}
    full = {k: d[k].clone().requires_grad_() for k in names}
    pf = params()
    h0f = None if h0 is None else h0.clone().requires_grad_()
    ref, _ = ops.selective_scan_state(full["u"], full["delta"], pf["A_log"], full["Bm"], full["Cm"], pf["D"], h0f, z=full["z"],
                                      dt_bias=pf["bias"])
    ref.backward(d["dout"])
    lo, hi = par.shard_range(L, rank, world)
    loc = {k: par.shard_sequence(d[k], rank, world).clone().requires_grad_() for k in names}
    pl = params()
    h0l = None if h0 is None else h0.clone().requires_grad_()
    out = par.sequence_sharded_scan(loc["u"], loc["delta"], pl["A_log"], loc["Bm"], loc["Cm"], pl["D"], z=loc["z"],
                                    dt_bias=pl["bias"], h0=h0l)
    out.backward(par.shard_sequence(d["dout"], rank, world))
    par.allreduce_gradients(list(pl.values()), average=False)
    tol = 1e-4 if dt == torch.float32 else 2e-2
    errs = {"out": _rel(out, ref[:, lo:hi])}
    errs.update({k: _rel(loc[k].grad, full[k].grad[:, lo:hi]) for k in names})
    errs.update({k: _rel(pl[k].grad, pf[k].grad) for k in pl})
    if with_h0:
        if rank == 0:
            errs["h0"] = _rel(h0l.grad, h0f.grad)
        else:
            assert h0l.grad is None
    assert max(errs.values()) < tol, (rank, mode, errs)


def _model_case(rank, world, dev, mode):
    cfg = MambaConfig(d_model=64, n_layers=2, d_state=32 if "d32" in mode else 16)
    torch.manual_seed(0)
    m = Mamba(cfg).to(dev)
    ref_m = copy.deepcopy(m)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 777, 64, generator=g).to(dev)
    wt = torch.randn(2, 777, 64, generator=g).to(dev)
    y_ref = ref_m(x)
    (y_ref * wt).sum().backward()
    lo, hi = par.shard_range(777, rank, world)
    y = par.sequence_sharded_forward(m, par.shard_sequence(x, rank, world))
    (y * par.shard_sequence(wt, rank, world)).sum().backward()
    par.allreduce_gradients(m.parameters(), average=False)
    errs = {"y": _rel(y, y_ref[:, lo:hi])}
    errs.update({n: _rel(p.grad, q.grad) for (n, p), q in zip(m.named_parameters(), ref_m.parameters())})
    assert max(errs.values()) < 1e-4, (rank, mode, errs)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("mode", ["scan_f32", "scan_f32_h0", "scan_bf16", "scan_bf16_h0", "model_d16", "model_d32"])
def test_two_gpu_sequence_sharding_matches_single_gpu(mode):
    mp.spawn(_worker, args=(2, _free_port(), mode), nprocs=2, join=True)
