"""CPU-only checks of the d_state envelope: the size queries of the C ABI follow the generic kernels' layouts for N = 32 and 64,
every other N from 1 to 128 stays unsupported, and the Python routing set (ops.FUSED_D_STATES) is the C ABI's."""
import ctypes

import pytest

SIZES = [(16, 300, 1024), (2, 203, 40), (3, 77, 1000)]   # B * ceil(ED / 32) warps fill the GPU: no L-split, one segment


def _a(v):
    return (v + 255) // 256 * 256


@pytest.mark.parametrize("N", [32, 64])
@pytest.mark.parametrize("B,L,ED", SIZES)
def test_size_queries_follow_the_generic_layout(B, L, ED, N):
    """Checkpoint: fp32 state every 16 steps ([b][chunk][pair][ED]) + y in the activation dtype; forward workspace: none
    without an L-split; backward: one dB|dC row of 2 N floats per warp and token + dA[N] | dD | ddt_bias per channel.
    The chained kernels (ED % 32 == 0) serve d_state = 16 only, so ED = 1024 takes the same layout."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    nseg = 1 if B * -(-ED // 32) * 2 >= 4 * 148 else None   # plan_segments on 148 SMs (a B200, or no device)
    states = B * -(-L // 16) * ED * N * 4
    for dt, el in ((_native.GFE_F32, 4), (_native.GFE_BF16, 2), (_native.GFE_F16, 2)):
        assert lib.gfe_selscan_ckpt_bytes_dt(B, L, ED, N, dt) == states + B * L * ED * el
    assert lib.gfe_selscan_ckpt_bytes(B, L, ED, N) == states + B * L * ED * 4
    if nseg == 1:
        assert lib.gfe_selscan_fwd_workspace_bytes(B, L, ED, N) == 0
        assert lib.gfe_selscan_bwd_workspace_bytes(B, L, ED, N) == _a(-(-ED // 32) * B * L * 2 * N * 4) + _a(B * (N + 2) * ED * 4)


def test_split_workspace_scales_with_n():
    """With an L-split the forward workspace holds N / 2 float2 per (b, segment, channel) + sum(delta): its state part
    doubles from N = 32 to N = 64, and both exceed N = 16's generic layout at ED % 32 != 0."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    B, L, ED = 1, 2100, 40
    w = {N: lib.gfe_selscan_fwd_workspace_bytes(B, L, ED, N) for N in (16, 32, 64)}
    assert 0 < w[16] < w[32] < w[64]
    assert w[64] - w[32] >= w[32] - w[16] > 0   # align(seg_h) grows with N, align(seg_sd) does not


def test_unsupported_d_state_stays_unsupported():
    """Every N in 1..128 outside {16, 32, 64}: the size queries return 0, the scan and the decode step refuse with
    GFE_ERR_UNSUPPORTED before any launch, with 'd_state' in the message."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    fake = ctypes.c_void_p(256)
    for N in range(1, 129):
        if N in (16, 32, 64):
            continue
        for B, L, ED in SIZES:
            assert lib.gfe_selscan_ckpt_bytes(B, L, ED, N) == 0, N
            assert lib.gfe_selscan_ckpt_bytes_dt(B, L, ED, N, _native.GFE_BF16) == 0, N
            assert lib.gfe_selscan_fwd_workspace_bytes(B, L, ED, N) == 0, N
            assert lib.gfe_selscan_bwd_workspace_bytes(B, L, ED, N) == 0, N
        a = _native.SelscanArgs()
        a.batch, a.seqlen, a.d_inner, a.d_state = 1, 8, 32, N
        assert lib.gfe_selscan_fwd(ctypes.byref(a), None) == -3 and b"d_state" in lib.gfe_last_error_string(), N
        assert lib.gfe_selscan_bwd(ctypes.byref(a), None) == -3 and b"d_state" in lib.gfe_last_error_string(), N
        rc = lib.gfe_ssm_step(fake, 0, fake, 0, None, 0, fake, 0, fake, 0, fake, fake, None, fake, fake, 0, 1, 32, N, 0,
                              _native.GFE_F32, None)
        assert rc == -3 and b"d_state" in lib.gfe_last_error_string(), N


def test_python_set_matches_the_c_abi():
    from gfe_mamba_b200 import _native, ops
    lib = _native.lib()
    assert set(ops.FUSED_D_STATES) == {N for N in range(1, 129) if lib.gfe_selscan_ckpt_bytes(2, 64, 40, N) > 0}


def test_block_routing_follows_the_set():
    """MambaBlock takes the one-node inner path for every fused d_state and the composition otherwise (decided on shapes
    only, so a stand-in object plays in_proj's output)."""
    import torch
    from gfe_mamba_b200 import MambaBlock, MambaConfig, ops

    class _Cuda:   # what _inner_fusable reads of the tensor
        is_cuda, dtype = True, torch.float32

        def __init__(self, ed):
            self.shape = (1, 1, 2 * ed)

        def dim(self):
            return 3
    for N in (4, 8, 16, 32, 48, 64, 128):
        blk = MambaBlock(MambaConfig(d_model=16, n_layers=1, d_state=N))
        assert blk._inner_fusable(_Cuda(blk.config.d_inner)) == (N in ops.FUSED_D_STATES), N
