"""Sequence sharding without a GPU: the summary entry points of the C ABI (declared, exported, bound, sized), the rank
combines of gfe_mamba_b200.parallel against a direct fp64 loop, shard_sequence, and the sharded functions' refusals on a
gloo world of two (CPU tensors: there is no CPU fallback; a rank too short for the conv window)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gfe_mamba_b200 import _native as nat
from gfe_mamba_b200 import parallel as par

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("gfe_selscan_summary_workspace_bytes", "gfe_selscan_summary_fwd", "gfe_selscan_summary_bwd")


def test_summary_symbols_declared_exported_bound():
    header = open(os.path.join(ROOT, "include", "gfe_mamba_b200.h")).read()
    lib = nat.lib()
    for name in NEW:
        assert f" {name}(" in header, name
        assert name in nat.SIGNATURES, name
        assert getattr(lib, name) is not None


def test_summary_workspace_without_gpu():
    ws = nat.lib().gfe_selscan_summary_workspace_bytes
    for N in (16, 32, 64):
        for (B, L, ED) in ((1, 1, 256), (1, 65536, 1024), (8, 300, 1536), (2, 75, 80)):
            n = ws(B, L, ED, N)
            # at least one segment's local state and sum of step sizes per (b, c)
            assert n >= B * ED * (N + 1) * 4, (B, L, ED, N, n)
    assert ws(1, 100, 256, 24) == 0 and ws(0, 100, 256, 16) == 0 and ws(1, 0, 256, 16) == 0 and ws(1, 100, -1, 16) == 0


def _summaries(W, B, ED, N, seed):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(W, B, ED, N, generator=g)
    sd = torch.rand(W, B, ED, generator=g) * 3
    A_log = torch.randn(ED, N, generator=g) * 0.5
    return h, sd, A_log


@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_rank_combines_match_fp64_loop(W):
    B, ED, N = 2, 5, 4
    h, sd, A_log = _summaries(W, B, ED, N, seed=W)
    A = -np.exp(A_log.double().numpy())
    hn, sdn = h.double().numpy(), sd.double().numpy()
    for r in range(W):
        want = np.zeros((B, ED, N))
        for q in range(r):
            want = np.exp(A[None] * sdn[q][..., None]) * want + hn[q]
        got = par.sequence_carry_in(h, sd, A_log, r)
        assert got.dtype == torch.float32 and np.abs(got.double().numpy() - want).max() <= 1e-5 * max(1.0, np.abs(want).max())
        # dlast_r = sum_{s > r} (prod_{r < q < s} exp(A sd_q)) g_s
        want = np.zeros((B, ED, N))
        for s in range(r + 1, W):
            P = np.ones((B, ED, N))
            for q in range(r + 1, s):
                P = P * np.exp(A[None] * sdn[q][..., None])
            want = want + P * hn[s]
        got = par.sequence_dlast(h, sd, A_log, r)
        assert np.abs(got.double().numpy() - want).max() <= 1e-5 * max(1.0, np.abs(want).max())


def test_shard_sequence_boundaries():
    x = torch.arange(2 * 17 * 3).view(2, 17, 3)
    for world in (1, 2, 3, 8):
        parts = [par.shard_sequence(x, r, world) for r in range(world)]
        assert torch.equal(torch.cat(parts, 1), x)
        assert max(p.shape[1] for p in parts) - min(p.shape[1] for p in parts) <= 1
        assert all(p.data_ptr() == x[:, par.shard_range(17, r, world)[0]:].data_ptr() for r, p in enumerate(parts))   # views
    assert par.shard_sequence(x.transpose(0, 1), 1, 2, dim=0).shape == (8, 2, 3)
    with pytest.raises(ValueError):
        par.shard_sequence(x, 2, 2)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _entry(rank, world, port):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from gfe_mamba_b200 import Mamba, MambaConfig
        B, L, ED, N, K = 1, 8, 64, 16, 4
        t = lambda *s: torch.randn(*s)
        with pytest.raises(RuntimeError, match="CUDA"):
            par.sequence_sharded_scan(t(B, L, ED), t(B, L, ED), t(ED, N), t(B, L, N), t(B, L, N), t(ED))
        with pytest.raises(RuntimeError, match="CUDA"):
            par.sequence_sharded_conv1d_silu(t(B, L, ED), t(ED, 1, K), t(ED))
        with pytest.raises(ValueError, match="K-1"):
            par.sequence_sharded_conv1d_silu(t(B, K - 2, ED), t(ED, 1, K), t(ED))
        with pytest.raises(RuntimeError, match="CUDA"):
            par.sequence_sharded_forward(Mamba(MambaConfig(d_model=32, n_layers=1)), t(B, L, 32))
        with pytest.raises(ValueError, match="d_state"):
            par.sequence_sharded_forward(Mamba(MambaConfig(d_model=32, n_layers=1, d_state=24)), t(B, L, 32))
        with pytest.raises(ValueError, match="d_conv"):
            par.sequence_sharded_forward(Mamba(MambaConfig(d_model=32, n_layers=1, d_conv=5)), t(B, L, 32))
    finally:
        dist.destroy_process_group()


def test_sharded_functions_refuse_cpu_and_short_ranks_gloo():
    mp.spawn(_entry, args=(2, _free_port()), nprocs=2, join=True)
