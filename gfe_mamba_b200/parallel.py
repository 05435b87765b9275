"""Multi-GPU plumbing for the selective-scan path: one process per GPU, torch.distributed (NCCL on GPUs,
gloo in the CPU unit tests).  The recurrence is independent per (batch row, channel), so the data path never
needs a collective; only gradients are exchanged (SURVEY 8e):

  batch sharding    each rank runs its own B/G sequences; after backward ONE flat-bucket all-reduce sums the
                    parameter gradients (A_log, D, conv1d, dt_proj, x_proj, in_proj, out_proj, norm).
  channel sharding  (one long sequence, BASELINE config 4) rank g owns channels [g*ED/G, (g+1)*ED/G) of
                    u, delta, z, A_log, D, dt_bias and out; B and C are shared, so their gradients -- sums over
                    ALL channels -- are all-reduced in backward (2 * B * L * N values).
  sequence sharding (one long sequence, a whole Mamba model) rank g owns tokens [lo, hi) of every row; only the conv
                    window (K-1 rows) and the scan state cross a rank boundary.  Each rank summarises its range
                    (ops.selscan_summary), one all-gather shares the summaries, and every rank combines those of the
                    ranks before it into its carry-in; backward does the same in reverse from the output gradient.
                    Parameter gradients are per-rank partial sums: allreduce_gradients(..., average=False).

The reference has no distributed code on this path (classify_mamba.py:69-73 is commented out); this module is
what its Accelerate/DDP use elsewhere (main_gan_vit.py:31,54) would provide.
"""
from __future__ import annotations

from typing import Callable, Iterable, List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import ops


def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced [lo, hi) slice of ``total`` items for ``rank`` (first ``total % world`` ranks get one more)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_batch(x: torch.Tensor, rank: int, world: int) -> torch.Tensor:
    """Rows of dim 0 owned by ``rank`` under batch sharding."""
    lo, hi = shard_range(x.shape[0], rank, world)
    return x[lo:hi]


def shard_channels(t: torch.Tensor, rank: int, world: int, dim: int = -1, multiple: int = 32) -> torch.Tensor:
    """Channel slice owned by ``rank`` under ED sharding.  ED / world must be a multiple of ``multiple`` (32 keeps every
    rank on the fast kernels: one warp serves 32 adjacent channels)."""
    ED = t.shape[dim]
    if ED % (world * multiple) != 0:
        raise ValueError(f"ED={ED} is not divisible into {world} shards of a multiple of {multiple} channels")
    per = ED // world
    return t.narrow(dim, rank * per, per)


def allreduce_gradients(params: Iterable[torch.nn.Parameter], group: Optional[dist.ProcessGroup] = None,
                        average: bool = True, bucket_bytes: int = 256 << 20) -> int:
    """Sum (or average) the gradients of ``params`` over the group with as few collectives as possible: gradients are
    packed into flat fp32 buckets (one bucket covers a whole Mamba stack), all-reduced, and unpacked in place.
    Parameters without a gradient contribute zeros so that every rank issues identical collectives.
    Returns the number of all-reduce calls issued."""
    params = [p for p in params if p.requires_grad]
    if not params or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return 0
    world = dist.get_world_size(group)
    calls, i = 0, 0
    while i < len(params):
        bucket: List[torch.nn.Parameter] = []
        size = 0
        while i < len(params) and (not bucket or (size + params[i].numel()) * 4 <= bucket_bytes):
            bucket.append(params[i])
            size += params[i].numel()
            i += 1
        dev = bucket[0].device
        flat = torch.zeros(size, dtype=torch.float32, device=dev)
        off = 0
        for p in bucket:
            if p.grad is not None:
                flat[off:off + p.numel()].copy_(p.grad.reshape(-1))
            off += p.numel()
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        calls += 1
        if average:
            flat.div_(world)
        off = 0
        for p in bucket:
            g = flat[off:off + p.numel()].view_as(p).to(p.dtype)
            if p.grad is None:
                p.grad = g.clone()
            else:
                p.grad.copy_(g)
            off += p.numel()
    return calls


class _AllReduceGrad(torch.autograd.Function):
    """Identity in forward; sums the incoming gradient over the group in backward (for tensors replicated across
    ranks whose consumers are sharded: B and C under channel sharding)."""

    @staticmethod
    def forward(ctx, x, group):
        ctx.group = group
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        if dist.is_initialized() and dist.get_world_size(ctx.group) > 1:
            g = g.clone()
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=ctx.group)
        return g, None


def channel_sharded_scan(scan_fn: Callable, u, delta, A_log, Bm, Cm, D, z=None, dt_bias=None,
                         group: Optional[dist.ProcessGroup] = None, **kw):
    """Run ``scan_fn`` (gfe_mamba_b200.selective_scan_fn) on THIS rank's channel shard.

    ``u, delta, z`` are already the local shards (B, L, ED/G); ``A_log, D, dt_bias`` the local rows; ``Bm, Cm`` are the
    full, replicated (B, L, N) tensors.  The output is the local (B, L, ED/G) shard.  In backward the gradients of
    Bm and Cm are all-reduced (they sum over every rank's channels); nothing else is exchanged.  For a whole model on one
    long sequence see sequence_sharded_scan / sequence_sharded_forward below: they split time instead of channels, and their
    parameter gradients are per-rank partial sums that the caller sums over the group."""
    Bm = _AllReduceGrad.apply(Bm, group)
    Cm = _AllReduceGrad.apply(Cm, group)
    return scan_fn(u, delta, A_log, Bm, Cm, D, z=z, dt_bias=dt_bias, **kw)


# ------------------------------------------------------------------------------------------ sequence sharding
def shard_sequence(x: torch.Tensor, rank: int, world: int, dim: int = 1) -> torch.Tensor:
    """Tokens of ``rank`` under sequence sharding: the contiguous slice ``shard_range`` gives along ``dim`` (a view)."""
    lo, hi = shard_range(x.shape[dim], rank, world)
    return x.narrow(dim, lo, hi - lo)


def _rank_world(group) -> Tuple[int, int]:
    if not dist.is_initialized():
        return 0, 1
    return dist.get_rank(group), dist.get_world_size(group)


def _all_gather(t: torch.Tensor, world: int, group) -> torch.Tensor:
    """(world, *t.shape): every rank's ``t`` in group order, one collective."""
    out = torch.empty((world,) + tuple(t.shape), dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(out, t.contiguous(), group=group)
    return out


def _decay(A_log: torch.Tensor, sum_delta: torch.Tensor) -> torch.Tensor:
    """exp(A sum_delta) per (b, c, n) with A = -exp(A_log): (..., B, ED) sums -> (..., B, ED, N) fp32."""
    return torch.exp(-torch.exp(A_log.detach().float()) * sum_delta.unsqueeze(-1))


def sequence_carry_in(h_loc: torch.Tensor, sum_delta: torch.Tensor, A_log: torch.Tensor, rank: int) -> torch.Tensor:
    """The scan state entering ``rank``'s range from the gathered summaries h_loc (W, B, ED, N) and sum_delta (W, B, ED) of
    every rank: carry = exp(A sum_delta[r]) carry + h_loc[r] over the ranks r < rank from zero, in fp32."""
    carry = torch.zeros_like(h_loc[0], dtype=torch.float32)
    for r in range(rank):
        carry = _decay(A_log, sum_delta[r]) * carry + h_loc[r]
    return carry


def sequence_dlast(g_loc: torch.Tensor, sum_delta: torch.Tensor, A_log: torch.Tensor, rank: int) -> torch.Tensor:
    """The gradient of the scan state leaving ``rank``'s range, from the gathered reverse summaries g_loc (W, B, ED, N) and the
    forward sum_delta (W, B, ED): dlast = sum over s > rank of (prod over rank < q < s of exp(A sum_delta[q])) g_loc[s],
    computed as carry = exp(A sum_delta[s]) carry + g_loc[s] from the last rank down to rank + 1, in fp32."""
    carry = torch.zeros_like(g_loc[0], dtype=torch.float32)
    for s in range(g_loc.shape[0] - 1, rank, -1):
        carry = _decay(A_log, sum_delta[s]) * carry + g_loc[s]
    return carry


class _SequenceScanGrad(torch.autograd.Function):
    """Identity on (out, h_last) of this rank's scan in forward.  In backward it turns the output gradient into the gradient
    of h_last: this rank's reverse summary, one all-gather, and the reverse combine over the later ranks.  So the scan's own
    backward (gfe_selscan_bwd_carry) runs once, seeded with what every later rank's tokens contribute."""

    @staticmethod
    def forward(ctx, out, h_last, saved):
        ctx.saved = saved
        return out.view_as(out)

    @staticmethod
    def backward(ctx, dout):
        delta, A_log, Cm, z, dt_bias, softplus, sum_delta, rank, world, group = ctx.saved
        g_loc = ops.selscan_summary_rev(dout, delta, A_log, Cm, z=z, dt_bias=dt_bias, delta_softplus=softplus)
        g_all = _all_gather(g_loc, world, group)
        dlast = sequence_dlast(g_all, sum_delta, A_log, rank) if rank < world - 1 else None
        return dout, dlast, None


def sequence_sharded_scan(u, delta, A_log, Bm, Cm, D, z=None, dt_bias=None, delta_softplus: bool = True,
                          h0: Optional[torch.Tensor] = None, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """``selective_scan_fn`` over one sequence split along time: each rank holds tokens [lo, hi) of every row of u, delta, z
    (B, L_r, ED) and Bm, Cm (B, L_r, N), ranks in group order, and gets its rows of the output.  Parameters are replicated.

    Forward: this rank's summary (ops.selscan_summary), ONE all-gather of (h_loc, sum_delta), the combine over the earlier
    ranks (sequence_carry_in), then the scan from that carry (ops.selective_scan_state; checkpoints only under grad).
    Backward: the reverse summary of the output gradient, one all-gather, the reverse combine over the later ranks
    (sequence_dlast), then the scan's backward from that final-state gradient.  No rank waits on another's scan.

    h0 (B, ED, N): the state before the first token, significant on rank 0 only (its gradient is returned there).  Gradients
    of u, delta, z, Bm, Cm are this rank's rows; those of A_log, D, dt_bias are this rank's partial sums, which the caller sums
    over the group (allreduce_gradients(..., average=False) or train.LayerGradSync).  With one rank this is
    selective_scan_state from h0."""
    rank, world = _rank_world(group)
    if world == 1:
        return ops.selective_scan_state(u, delta, A_log, Bm, Cm, D, h0, z=z, dt_bias=dt_bias, delta_softplus=delta_softplus)[0]
    with torch.no_grad():
        h_loc, sd = ops.selscan_summary(u, delta, A_log, Bm, dt_bias=dt_bias, delta_softplus=delta_softplus)
        if rank == 0 and h0 is not None:   # rank 0's range as seen by the others starts from h0
            h_loc = _decay(A_log, sd) * h0.detach().float() + h_loc
        Bsz, ED, N = h_loc.shape
        packed = _all_gather(torch.cat([h_loc.reshape(-1), sd.reshape(-1)]), world, group)
        h_all = packed[:, :Bsz * ED * N].view(world, Bsz, ED, N)
        sd_all = packed[:, Bsz * ED * N:].view(world, Bsz, ED)
        h_in = sequence_carry_in(h_all, sd_all, A_log, rank) if rank > 0 else None
    if rank == 0:
        h_in = h0
    out, h_last = ops.selective_scan_state(u, delta, A_log, Bm, Cm, D, h_in, z=z, dt_bias=dt_bias, delta_softplus=delta_softplus)
    if out.requires_grad:
        saved = (delta.detach(), A_log.detach(), Cm.detach(), None if z is None else z.detach(),
                 None if dt_bias is None else dt_bias.detach(), delta_softplus, sd_all, rank, world, group)
        out = _SequenceScanGrad.apply(out, h_last, saved)
    return out


class _PreviousWindow(torch.autograd.Function):
    """The conv window of this rank: the last K-1 rows of the previous rank's input, as (B, ED, K-1) (zeros on rank 0), from
    one all-gather of every rank's tail.  Backward sends the window's gradient back the same way: the rows this rank's tail
    contributed to the next rank's window."""

    @staticmethod
    def forward(ctx, tail, rank, world, group):
        ctx.meta = (rank, world, group)
        tails = _all_gather(tail.detach(), world, group)                     # (W, B, K-1, ED)
        prev = tails[rank - 1] if rank > 0 else torch.zeros_like(tail)
        return prev.transpose(1, 2).contiguous()

    @staticmethod
    def backward(ctx, dwin):
        rank, world, group = ctx.meta
        dwins = _all_gather(dwin.transpose(1, 2), world, group)               # (W, B, K-1, ED)
        dtail = dwins[rank + 1] if rank < world - 1 else torch.zeros_like(dwins[0])
        return dtail, None, None, None


def sequence_sharded_conv1d_silu(xin: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor],
                                 inputs: Optional[torch.Tensor] = None,
                                 group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """``causal_conv1d_silu`` over one sequence split along time: xin (B, L_r, ED) holds this rank's tokens, ranks in group
    order; returns this rank's rows of u.  Each rank's window is the previous rank's last K-1 rows of xin (one all-gather of
    the tails); on rank 0 it is ``inputs`` (B, ED, K-1) or zeros.  Backward returns the window's gradient to the previous
    rank, which adds it to the gradient of its last K-1 rows.  Every rank must hold at least K-1 tokens (ValueError
    otherwise)."""
    rank, world = _rank_world(group)
    K = weight.shape[-1]
    L = xin.shape[1]
    if world > 1 and L < K - 1:
        raise ValueError(f"sequence_sharded_conv1d_silu: rank {rank} holds {L} tokens, fewer than the conv window's K-1 = {K - 1}")
    ops._require_cuda(xin, weight, bias, inputs)
    if world == 1:
        return ops.causal_conv1d_silu_state(xin, inputs, weight, bias)[0]
    window = _PreviousWindow.apply(xin[:, L - (K - 1):], rank, world, group)
    if rank == 0 and inputs is not None:
        window = window + inputs.to(window.dtype)
    return ops.causal_conv1d_silu_state(xin, window, weight, bias)[0]


def _sequence_sharded_mixer(block, x: torch.Tensor, group) -> torch.Tensor:
    """MambaBlock.forward on this rank's tokens: in_proj, the sharded conv, x_proj / dt_proj (inner layernorms included), the
    sharded scan with the gate fused, out_proj."""
    xz = block.in_proj(x)
    xin, z = xz.chunk(2, dim=-1)
    u = sequence_sharded_conv1d_silu(xin, block.conv1d.weight, block.conv1d.bias, group=group)
    delta, Bm, Cm = block._project(u)
    y = sequence_sharded_scan(u, delta, block.A_log, Bm, Cm, block.D, z=z, dt_bias=block.dt_proj.bias, delta_softplus=True,
                              group=group)
    return block.out_proj(y)


def sequence_sharded_forward(model, x_local: torch.Tensor, group: Optional[dist.ProcessGroup] = None) -> torch.Tensor:
    """This rank's rows of ``model(x_full)`` for a ``Mamba`` model whose input sequence is split along time: x_local (B, L_r, D)
    holds tokens [lo, hi) of every row (``shard_sequence``), ranks in group order.  Differentiable; the gradients of the
    parameters are this rank's partial sums, to be summed over the group with allreduce_gradients(..., average=False).

    The token-wise parts (projections, add + RMSNorm) run locally; per layer the conv window and the scan state cross the rank
    boundaries (sequence_sharded_conv1d_silu, sequence_sharded_scan): four all-gathers per layer and training step, issued
    in the same order on every rank.  Every rank must hold at least d_conv - 1 tokens.  The configuration must be one the
    from-state kernels serve (d_state in ops.FUSED_D_STATES, 2 <= d_conv <= 4): anything else raises ValueError."""
    from .mamba import _fusable_norm
    cfg = model.config
    if cfg.d_state not in ops.FUSED_D_STATES or not 2 <= cfg.d_conv <= 4:
        raise ValueError(f"sequence_sharded_forward: d_state={cfg.d_state}, d_conv={cfg.d_conv} outside the from-state kernels "
                         f"(d_state in {ops.FUSED_D_STATES}, d_conv in 2..4)")
    ops._require_cuda(x_local)
    rank, world = _rank_world(group)
    if world > 1 and len(model.layers) > 0:   # every rank learns every rank's length, so that all raise together
        lens = _all_gather(torch.tensor([x_local.shape[1]], device=x_local.device), world, group).flatten().tolist()
        if min(lens) < cfg.d_conv - 1:
            raise ValueError(f"sequence_sharded_forward: rank lengths {lens}; every rank needs at least d_conv - 1 = "
                             f"{cfg.d_conv - 1} tokens")
    if len(model.layers) == 0:
        return x_local
    if not _fusable_norm(x_local, cfg):
        x = x_local
        for layer in model.layers:
            x = _sequence_sharded_mixer(layer.mixer, layer.norm(x), group) + x
        return x
    resid, branch = x_local, None
    for layer in model.layers:
        resid, normed = ops.add_rmsnorm(resid, branch, layer.norm.weight, layer.norm.eps)
        branch = _sequence_sharded_mixer(layer.mixer, normed, group)
    return branch + resid


def parameter_gradient_names(model: torch.nn.Module) -> Sequence[str]:
    """Names of the parameters whose gradients the batch-sharded step all-reduces (everything trainable)."""
    return [n for n, p in model.named_parameters() if p.requires_grad]
