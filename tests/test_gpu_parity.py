"""GPU parity: the sm_100a kernels, called through the public API (ctypes -> C ABI), against the CPU oracle and
the reference-generated golden fixtures.  Run with ``pytest -m gpu`` on a B200.

Tolerances (BASELINE.json north_star): fp32 max-normalised error <= 1e-4, bf16 <= 2e-2, on outputs and gradients.
"""
import os

import numpy as np
import pytest
import torch

from oracle import oracle as orc

pytestmark = pytest.mark.gpu

TOL = {torch.float32: 1e-4, torch.bfloat16: 2e-2, torch.float16: 5e-3}


def relerr(a, b):
    a = a.detach().float().cpu().numpy().astype(np.float64) if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = b.detach().float().cpu().numpy().astype(np.float64) if torch.is_tensor(b) else np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.isfinite(a).all(), "non-finite values from the CUDA path"
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def cuda(a, dtype=torch.float32, grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dtype)
    return t.requires_grad_() if grad else t


def _load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name + ".npz")))


def make_scan_inputs(B, L, ED, N=16, seed=0, dt_scale=0.5):
    """Synthetic inputs of SURVEY 8d: dt_bias as mamba.py:150-155, A_log = log(1..N) + jitter, D = 1 + jitter."""
    r = np.random.default_rng(seed)
    u = r.standard_normal((B, L, ED)).astype(np.float32)
    draw = (r.standard_normal((B, L, ED)) * dt_scale).astype(np.float32)
    z = r.standard_normal((B, L, ED)).astype(np.float32)
    Bm = r.standard_normal((B, L, N)).astype(np.float32)
    Cm = r.standard_normal((B, L, N)).astype(np.float32)
    A_log = (np.log(np.arange(1, N + 1, dtype=np.float32))[None].repeat(ED, 0) + 0.1 * r.standard_normal((ED, N))).astype(np.float32)
    D = (1.0 + 0.1 * r.standard_normal(ED)).astype(np.float32)
    dt = np.exp(r.uniform(np.log(1e-3), np.log(1e-1), ED)).clip(min=1e-4)
    bias = (dt + np.log(-np.expm1(-dt))).astype(np.float32)
    dout = r.standard_normal((B, L, ED)).astype(np.float32)
    return dict(u=u, draw=draw, z=z, Bm=Bm, Cm=Cm, A_log=A_log, D=D, bias=bias, dout=dout)


def run_fused(d, dtype, use_z=True, use_bias=True, softplus=True):
    from gfe_mamba_b200 import selective_scan_fn
    u, draw = cuda(d["u"], dtype, True), cuda(d["draw"], dtype, True)
    z = cuda(d["z"], dtype, True) if use_z else None
    Bm, Cm = cuda(d["Bm"], dtype, True), cuda(d["Cm"], dtype, True)
    A_log, D = cuda(d["A_log"], grad=True), cuda(d["D"], grad=True)
    bias = cuda(d["bias"], grad=True) if use_bias else None
    out = selective_scan_fn(u, draw, A_log, Bm, Cm, D, z=z, dt_bias=bias, delta_softplus=softplus)
    out.backward(cuda(d["dout"], dtype))
    torch.cuda.synchronize()
    g = dict(out=out, du=u.grad, ddelta=draw.grad, dz=None if z is None else z.grad, dB=Bm.grad, dC=Cm.grad,
             dA_log=A_log.grad, dD=D.grad, ddt_bias=None if bias is None else bias.grad)
    return g


def oracle_fused(d, dtype, use_z=True, use_bias=True, softplus=True):
    """fp64 sequential oracle on the inputs as the kernel sees them (rounded to ``dtype``)."""
    def rnd(a):
        return torch.from_numpy(a).to(dtype).float().numpy()
    u, draw, z, Bm, Cm, dout = (rnd(d[k]) for k in ("u", "draw", "z", "Bm", "Cm", "dout"))
    zz = z if use_z else None
    bias = d["bias"] if use_bias else None
    out = orc.selscan_seq_fwd(u, draw, d["A_log"], Bm, Cm, d["D"], z=zz, dt_bias=bias, softplus=softplus)
    g = orc.selscan_seq_bwd(u, draw, d["A_log"], Bm, Cm, d["D"], dout, z=zz, dt_bias=bias, softplus=softplus)
    g["out"] = out
    return g


def compare(got, want, tol, keys=("out", "du", "ddelta", "dz", "dB", "dC", "dA_log", "dD", "ddt_bias")):
    errs = {}
    for k in keys:
        if want.get(k) is None:
            assert got.get(k) is None
            continue
        errs[k] = relerr(got[k], want[k])
    bad = {k: v for k, v in errs.items() if not v <= tol}
    assert not bad, f"over tolerance {tol}: {bad} (all: {errs})"
    return errs


# ------------------------------------------------------------------------------------------------- pscan
@pytest.mark.parametrize("L", [1, 2, 3, 4, 5, 8, 37, 64])
def test_pscan_golden(golden_dir, L):
    from cross_atten.pscan import pscan
    g = _load(golden_dir, "pscan_small")
    A, X = cuda(g[f"L{L}_A"], grad=True), cuda(g[f"L{L}_X"], grad=True)
    H = pscan(A, X)
    H.backward(cuda(g[f"L{L}_dH"]))
    assert relerr(H, g[f"L{L}_H"]) < 1e-5
    assert relerr(X.grad, g[f"L{L}_dX"]) < 1e-5
    assert relerr(A.grad, g[f"L{L}_dA"]) < 1e-5


@pytest.mark.parametrize("shape", [(2, 1858, 8, 16), (32, 256, 64, 16), (1, 4096, 4, 16), (3, 100, 5, 3), (2, 777, 7, 1),
                                   (8, 300, 1024, 16), (16, 128, 1024, 16), (2, 1858, 1024, 16)])
def test_pscan_vs_oracle(shape):
    """Random shapes incl. non-power-of-two L, the L-split path (small B*D*N), odd D*N (scalar path), and sizes that select
    each single-pass variant: 1 / 2 / 4 elements per thread with 32 / 16 / 8 steps of loads in flight."""
    from gfe_mamba_b200 import pscan
    r = np.random.default_rng(7)
    A = r.uniform(0.3, 1.0, shape).astype(np.float32)
    X = r.standard_normal(shape).astype(np.float32)
    dH = r.standard_normal(shape).astype(np.float32)
    At, Xt = cuda(A, grad=True), cuda(X, grad=True)
    H = pscan(At, Xt)
    H.backward(cuda(dH))
    H_ref = orc.pscan_fwd(A, X)
    dA_ref, dX_ref = orc.pscan_bwd(A, H_ref, dH)
    assert relerr(H, H_ref) < 1e-4
    assert relerr(Xt.grad, dX_ref) < 1e-4
    assert relerr(At.grad, dA_ref) < 1e-4


def test_pscan_does_not_mutate_inputs_and_is_linear_in_x():
    from gfe_mamba_b200 import pscan
    torch.manual_seed(0)
    A = torch.rand(2, 300, 8, 16, device="cuda") * 0.5 + 0.5
    X1, X2 = torch.randn_like(A), torch.randn_like(A)
    A0, X0 = A.clone(), X1.clone()
    H1, H2 = pscan(A, X1), pscan(A, X2)
    assert torch.equal(A, A0) and torch.equal(X1, X0)
    H12 = pscan(A, 2.0 * X1 - 3.0 * X2)
    assert relerr(H12, 2.0 * H1 - 3.0 * H2) < 1e-5


# --------------------------------------------------------------------------------------- fused selective scan
@pytest.mark.parametrize("B,L,ED", [(2, 1, 32), (1, 5, 40), (2, 16, 64), (2, 17, 32), (3, 37, 96), (2, 64, 33),
                                    (2, 300, 64), (2, 1858, 64),
                                    (1, 2100, 40), (2, 1858, 1000)])   # ED % 32 != 0 with few warps: generic kernels split L
def test_selscan_fp32_vs_oracle(B, L, ED):
    d = make_scan_inputs(B, L, ED, seed=B * 1000 + L)
    compare(run_fused(d, torch.float32), oracle_fused(d, torch.float32), TOL[torch.float32])


@pytest.mark.parametrize("use_z,use_bias,softplus", [(False, True, True), (True, False, True), (True, True, False),
                                                     (False, False, False)])
def test_selscan_variants(use_z, use_bias, softplus):
    d = make_scan_inputs(2, 75, 64, seed=5)
    if not softplus:   # delta must then already be positive
        d["draw"] = np.abs(d["draw"]) * 0.2 + 1e-3
        d["bias"] = np.abs(d["bias"]) * 0.01
    compare(run_fused(d, torch.float32, use_z, use_bias, softplus),
            oracle_fused(d, torch.float32, use_z, use_bias, softplus), TOL[torch.float32])


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_selscan_half_precision(dtype):
    """16-bit activations, fp32 state/params: oracle = fp64 math on the rounded inputs (SURVEY 8d)."""
    d = make_scan_inputs(2, 512, 128, seed=11)
    compare(run_fused(d, dtype), oracle_fused(d, dtype), TOL[dtype])


# ---- the chained kernels (selscan_v4_fwd.cu / selscan_chain_bwd.cu), serving ED % 32 == 0; their L-segments wait on each
# ---- other when B * ED / 32 >= 296 warps ------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,L,ED", [(24, 203, 512),    # ragged L (not a multiple of 8 / 16), one segment
                                    (20, 1000, 512),   # every chain has a CTA of its own: one unit per chain, ragged tail
                                    (40, 400, 1024),   # more chains (640) than resident CTAs: three chained L-segments
                                    (10, 1170, 4096),  # same, 64-channel blocks on both sides, ragged last segment
                                    (24, 203, 480),    # ED % 64 == 32: 32-channel blocks on both sides
                                    (40, 16, 256), (40, 1, 256), (40, 9, 256)])   # shorter than one chunk
def test_selscan_chained_fp32_vs_oracle(B, L, ED):
    d = make_scan_inputs(B, L, ED, seed=B + L + ED)
    compare(run_fused(d, torch.float32), oracle_fused(d, torch.float32), TOL[torch.float32])


@pytest.mark.parametrize("use_z,use_bias,softplus", [(False, True, True), (True, False, True), (True, True, False),
                                                     (False, False, False)])
def test_selscan_chained_variants(use_z, use_bias, softplus):
    d = make_scan_inputs(20, 300, 512, seed=6)
    if not softplus:
        d["draw"] = np.abs(d["draw"]) * 0.2 + 1e-3
        d["bias"] = np.abs(d["bias"]) * 0.01
    compare(run_fused(d, torch.float32, use_z, use_bias, softplus),
            oracle_fused(d, torch.float32, use_z, use_bias, softplus), TOL[torch.float32])


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_selscan_chained_half_precision(dtype):
    d = make_scan_inputs(20, 523, 512, seed=12)
    compare(run_fused(d, dtype), oracle_fused(d, dtype), TOL[dtype])


def test_selscan_chained_strided_views_and_inference():
    """Chained kernels on in-place views (u|z halves of one tensor, B/C slices of x_proj's output) and without checkpoints
    (no grad): same output as with them."""
    from gfe_mamba_b200 import selective_scan_fn
    B, L, ED, N, R = 20, 200, 512, 16, 32
    d = make_scan_inputs(B, L, ED, seed=22)
    xz = torch.cat([cuda(d["u"]), cuda(d["z"])], dim=-1)
    dbc = torch.cat([torch.zeros(B, L, R, device="cuda"), cuda(d["Bm"]), cuda(d["Cm"])], dim=-1)
    u, z = xz[..., :ED], xz[..., ED:]
    Bm, Cm = dbc[..., R:R + N], dbc[..., R + N:]
    A_log, D, bias = cuda(d["A_log"]), cuda(d["D"]), cuda(d["bias"])
    with torch.no_grad():
        out = selective_scan_fn(u, cuda(d["draw"]), A_log, Bm, Cm, D, z=z, dt_bias=bias)
    want = orc.selscan_seq_fwd(d["u"], d["draw"], d["A_log"], d["Bm"], d["Cm"], d["D"], z=d["z"], dt_bias=d["bias"])
    assert relerr(out, want) < TOL[torch.float32]
    got = run_fused(d, torch.float32)
    assert relerr(out, got["out"]) < 1e-6


def test_selscan_l_split_path():
    """Few channels, long L -> the chained kernels run independent L-segments whose carries come from the summary and
    combine passes."""
    d = make_scan_inputs(1, 4096, 64, seed=3)
    compare(run_fused(d, torch.float32), oracle_fused(d, torch.float32), TOL[torch.float32])
    d = make_scan_inputs(2, 1858, 32, seed=4)   # production-like L, ragged last chunk, split
    compare(run_fused(d, torch.float32), oracle_fused(d, torch.float32), TOL[torch.float32])


@pytest.mark.parametrize("use_z,use_bias,softplus,dtype", [(True, True, True, torch.float32), (False, True, True, torch.float32),
                                                           (True, False, False, torch.float32), (True, True, True, torch.bfloat16),
                                                           (False, False, True, torch.float16)])
def test_selscan_independent_segments_variants(use_z, use_bias, softplus, dtype):
    """Independent L-segments (summary + combine + main pass on the chained kernels): 32-channel blocks (ED % 64 == 32), ragged
    last segment, every flag combination of the reverse summary (dy = dout silu(z) | dout)."""
    d = make_scan_inputs(1, 2100, 96, seed=7)
    if not softplus:
        d["draw"] = np.abs(d["draw"]) * 0.2 + 1e-3
        d["bias"] = np.abs(d["bias"]) * 0.01
    compare(run_fused(d, dtype, use_z, use_bias, softplus), oracle_fused(d, dtype, use_z, use_bias, softplus), TOL[dtype])


def test_selscan_independent_segments_unaligned_views():
    """The same path on views that rule out 16-byte cp.async pieces (B/C slices at a 4-element offset of a wider tensor)."""
    from gfe_mamba_b200 import selective_scan_fn
    B, L, ED, N, R = 1, 1500, 64, 16, 4
    d = make_scan_inputs(B, L, ED, seed=23)
    xz = cuda(np.concatenate([d["u"], d["z"]], -1), grad=True)
    dbc = cuda(np.concatenate([np.zeros((B, L, R + 1), np.float32), d["Bm"], d["Cm"]], -1), grad=True)
    u, z = xz.chunk(2, dim=-1)
    _, Bm, Cm = torch.split(dbc, [R + 1, N, N], dim=-1)
    draw = cuda(d["draw"], grad=True)
    A_log, D, bias = cuda(d["A_log"], grad=True), cuda(d["D"], grad=True), cuda(d["bias"], grad=True)
    out = selective_scan_fn(u, draw, A_log, Bm, Cm, D, z=z, dt_bias=bias)
    out.backward(cuda(d["dout"]))
    want = oracle_fused(d, torch.float32)
    tol = TOL[torch.float32]
    assert relerr(out, want["out"]) < tol
    assert relerr(xz.grad[..., :ED], want["du"]) < tol and relerr(xz.grad[..., ED:], want["dz"]) < tol
    assert relerr(draw.grad, want["ddelta"]) < tol
    assert relerr(dbc.grad[..., R + 1:R + 1 + N], want["dB"]) < tol and relerr(dbc.grad[..., R + 1 + N:], want["dC"]) < tol
    assert relerr(A_log.grad, want["dA_log"]) < tol and relerr(bias.grad, want["ddt_bias"]) < tol


def test_selscan_strided_views():
    """u/z as the halves of one (B, L, 2ED) tensor, B/C as slices of (B, L, R+2N): consumed in place."""
    from gfe_mamba_b200 import selective_scan_fn
    B, L, ED, N, R = 2, 130, 64, 16, 4
    d = make_scan_inputs(B, L, ED, seed=21)
    xz = cuda(np.concatenate([d["u"], d["z"]], -1), grad=True)
    dbc = cuda(np.concatenate([np.zeros((B, L, R), np.float32), d["Bm"], d["Cm"]], -1), grad=True)
    u, z = xz.chunk(2, dim=-1)
    _, Bm, Cm = torch.split(dbc, [R, N, N], dim=-1)
    draw = cuda(d["draw"], grad=True)
    A_log, D, bias = cuda(d["A_log"], grad=True), cuda(d["D"], grad=True), cuda(d["bias"], grad=True)
    out = selective_scan_fn(u, draw, A_log, Bm, Cm, D, z=z, dt_bias=bias)
    out.backward(cuda(d["dout"]))
    want = oracle_fused(d, torch.float32)
    tol = TOL[torch.float32]
    assert relerr(out, want["out"]) < tol
    assert relerr(xz.grad[..., :ED], want["du"]) < tol and relerr(xz.grad[..., ED:], want["dz"]) < tol
    assert relerr(dbc.grad[..., R:R + N], want["dB"]) < tol and relerr(dbc.grad[..., R + N:], want["dC"]) < tol
    assert relerr(A_log.grad, want["dA_log"]) < tol and relerr(bias.grad, want["ddt_bias"]) < tol


def test_selscan_golden_reference_api(golden_dir):
    """MambaBlock.selective_scan(x, delta, A, B, C, D) against the reference's own pscan-based result + autograd."""
    from cross_atten.mamba import MambaBlock, MambaConfig
    g = _load(golden_dir, "selscan_small")
    for tag, D_model in (("L37", 4), ("L64", 8)):
        blk = MambaBlock(MambaConfig(d_model=D_model, n_layers=1)).cuda()
        t = {k: cuda(g[f"{tag}_{k}"], grad=True) for k in ("x", "delta", "A", "B", "C", "D")}
        y = blk.selective_scan(t["x"], t["delta"], t["A"], t["B"], t["C"], t["D"])
        y.backward(cuda(g[f"{tag}_dy"]))
        assert relerr(y, g[f"{tag}_y"]) < 1e-4
        assert relerr(blk.selective_scan_seq(t["x"], t["delta"], t["A"], t["B"], t["C"], t["D"]), g[f"{tag}_y_seq"]) < 1e-4
        for k, gk in (("x", "dx"), ("delta", "ddelta"), ("A", "dA"), ("B", "dB"), ("C", "dC"), ("D", "dD")):
            assert relerr(t[k].grad, g[f"{tag}_{gk}"]) < 1e-4, (tag, k)


def test_selscan_other_state_size_uses_pscan_kernel():
    """d_state != 16 runs the reference's composition on top of the CUDA pscan kernel (no CPU path)."""
    from gfe_mamba_b200 import MambaBlock, MambaConfig
    torch.manual_seed(1)
    blk = MambaBlock(MambaConfig(d_model=8, n_layers=1, d_state=4)).cuda()
    x = torch.randn(2, 21, 8, device="cuda")
    y = blk(x)
    p = {k: v.detach().cpu().numpy() for k, v in blk.state_dict().items()}
    assert relerr(y, orc.block_forward(p, x.cpu().numpy(), 4, blk.config.dt_rank)) < 1e-4


# ------------------------------------------------------------------------------------------ conv1d + SiLU
@pytest.mark.parametrize("B,L,ED,K", [(2, 1, 32, 4), (2, 3, 40, 4), (2, 64, 64, 4), (3, 130, 96, 4), (2, 257, 33, 3), (1, 70, 64, 2)])
def test_conv1d_silu(B, L, ED, K):
    from gfe_mamba_b200 import causal_conv1d_silu
    r = np.random.default_rng(L)
    xz = r.standard_normal((B, L, 2 * ED)).astype(np.float32)
    w = (r.standard_normal((ED, 1, K)) * 0.5).astype(np.float32)
    b = (r.standard_normal(ED) * 0.1).astype(np.float32)
    du = r.standard_normal((B, L, ED)).astype(np.float32)
    xzt, wt, bt = cuda(xz, grad=True), cuda(w, grad=True), cuda(b, grad=True)
    u = causal_conv1d_silu(xzt[..., :ED], wt, bt)       # strided half, as in MambaBlock.forward
    u.backward(cuda(du))
    xin = np.ascontiguousarray(xz[..., :ED])
    assert relerr(u, orc.conv1d_silu_fwd(xin, w, b)) < 1e-5
    dxin, dw, db = orc.conv1d_silu_bwd(xin, w, b, du)
    assert relerr(xzt.grad[..., :ED], dxin) < 1e-4 and float(xzt.grad[..., ED:].abs().max()) == 0.0
    assert relerr(wt.grad, dw) < 1e-4 and relerr(bt.grad, db) < 1e-4


@pytest.mark.parametrize("dtype,K", [(torch.bfloat16, 4), (torch.float16, 3)])
def test_conv1d_silu_half_precision(dtype, K):
    """16-bit activations (four channels per lane, packed FP32 math): oracle on the rounded inputs, ragged L and a second tile."""
    from gfe_mamba_b200 import causal_conv1d_silu
    B, L, ED = 2, 203, 128
    r = np.random.default_rng(9)
    rnd = lambda a: torch.from_numpy(a).to(dtype).float().numpy()
    xz = rnd(r.standard_normal((B, L, 2 * ED)).astype(np.float32))
    w = (r.standard_normal((ED, 1, K)) * 0.5).astype(np.float32)
    b = (r.standard_normal(ED) * 0.1).astype(np.float32)
    du = rnd(r.standard_normal((B, L, ED)).astype(np.float32))
    xzt = torch.from_numpy(xz).to(dtype).cuda().requires_grad_()
    wt, bt = cuda(w, grad=True), cuda(b, grad=True)
    u = causal_conv1d_silu(xzt[..., :ED], wt, bt)
    u.backward(torch.from_numpy(du).to(dtype).cuda())
    xin = np.ascontiguousarray(xz[..., :ED])
    tol = TOL[dtype]
    assert relerr(u, orc.conv1d_silu_fwd(xin, w, b)) < tol
    dxin, dw, db = orc.conv1d_silu_bwd(xin, w, b, du)
    assert relerr(xzt.grad[..., :ED], dxin) < tol
    assert relerr(wt.grad, dw) < 1e-3 and relerr(bt.grad, db) < 1e-3   # fp32 accumulation of exactly representable inputs


def test_conv1d_matches_torch_conv1d():
    """Same op as the reference module: nn.Conv1d(groups=ED, padding=K-1)(x^T)[:, :, :L]^T then silu (mamba.py:208-212)."""
    from gfe_mamba_b200 import causal_conv1d_silu
    torch.manual_seed(0)
    B, L, ED, K = 2, 100, 64, 4
    conv = torch.nn.Conv1d(ED, ED, K, groups=ED, padding=K - 1).cuda()
    x = torch.randn(B, L, ED, device="cuda")
    want = torch.nn.functional.silu(conv(x.transpose(1, 2))[:, :, :L].transpose(1, 2))
    assert relerr(causal_conv1d_silu(x, conv.weight, conv.bias), want) < 1e-5


# --------------------------------------------------------------------------------------------- block level
def _load_block(golden_dir):
    from cross_atten.mamba import MambaBlock, MambaConfig
    g = _load(golden_dir, "block_small")
    d_model, d_state, expand, d_conv, dt_rank, B, L = (int(v) for v in g["meta"])
    blk = MambaBlock(MambaConfig(d_model=d_model, n_layers=1, d_state=d_state, expand_factor=expand, d_conv=d_conv))
    blk.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")}, strict=True)
    return blk.cuda(), g


def test_block_golden_forward_backward(golden_dir):
    blk, g = _load_block(golden_dir)
    x = cuda(g["x"], grad=True)
    y = blk(x)
    y.backward(cuda(g["dy"]))
    assert relerr(y, g["y"]) < 1e-4
    assert relerr(x.grad, g["dx"]) < 1e-4
    for k, p in blk.named_parameters():
        assert relerr(p.grad, g[f"grad.{k}"]) < 1e-4, k


def test_block_golden_step(golden_dir):
    blk, g = _load_block(golden_dir)
    B, L = g["x"].shape[:2]
    x = cuda(g["x"])
    cache = (None, torch.zeros(B, blk.config.d_inner, blk.config.d_conv - 1, device="cuda"))
    ys = []
    for t in range(L):
        yt, cache = blk.step(x[:, t], cache)
        ys.append(yt)
    assert relerr(torch.stack(ys, 1), g["y_step"]) < 1e-4
    assert relerr(cache[0], g["h_last"]) < 1e-4 and relerr(cache[1], g["inputs_last"]) < 1e-5


def test_mamba_cfg1_golden(mamba_cfg1):
    """BASELINE config 1: Mamba(d_model=128, n_layers=2), B=8, L=64, fp32, forward + backward."""
    from cross_atten.mamba import Mamba, MambaConfig
    g = mamba_cfg1
    d_model, n_layers = int(g["meta"][0]), int(g["meta"][1])
    model = Mamba(MambaConfig(d_model=d_model, n_layers=n_layers))
    model.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("sd.")}, strict=True)
    model.cuda()
    x = cuda(g["x"], grad=True)
    y = model(x)
    y.backward(cuda(g["dy"]))
    assert relerr(y, g["y"]) < 1e-4
    assert relerr(x.grad, g["dx"]) < 1e-4
    grads = dict(model.named_parameters())
    for k in (k for k in g if k.startswith("grad.")):
        assert relerr(grads[k[5:]].grad, g[k]) < 1e-4, k


def test_block_bf16_autocast_close_to_fp32(golden_dir):
    blk, g = _load_block(golden_dir)
    x = cuda(g["x"])
    with torch.autocast("cuda", dtype=torch.bfloat16):
        y = blk(x)
    assert relerr(y, g["y"]) < 2e-2


def test_inner_layernorms_and_use_cuda_flag():
    """jamba.py uses inner_layernorms=True; mamba_transformer.py:65 passes use_cuda=True."""
    from cross_atten.mamba import MambaBlock, MambaConfig
    torch.manual_seed(2)
    cfg = MambaConfig(d_model=32, n_layers=1, inner_layernorms=True, use_cuda=True)
    blk = MambaBlock(cfg).cuda()
    assert cfg.use_cuda is True
    x = torch.randn(2, 50, 32, device="cuda", requires_grad=True)
    y = blk(x)
    y.sum().backward()
    assert torch.isfinite(y).all() and torch.isfinite(x.grad).all()
    assert all(p.grad is not None for p in blk.parameters())


# ------------------------------------------------------------------------------------------- full-size checks
def test_cfg2_shape_vs_oracle():
    """BASELINE config 2 scan shape: B=32, L=256, ED=512, fp32, fwd+bwd."""
    d = make_scan_inputs(32, 256, 512, seed=1236)
    compare(run_fused(d, torch.float32), oracle_fused(d, torch.float32), TOL[torch.float32])


def test_cfg3_full_size_properties_bf16():
    """BASELINE config 3 (B=16, L=4096, ED=1536, bf16) at full size: oracle on one batch row + size-independent
    properties (causality / prefix invariance, batch independence, linearity in u)."""
    from gfe_mamba_b200 import selective_scan_fn
    B, L, ED, N = 16, 4096, 1536, 16
    torch.manual_seed(1237)
    dev = "cuda"
    dt = torch.bfloat16
    u = torch.randn(B, L, ED, device=dev).to(dt)
    draw = (torch.randn(B, L, ED, device=dev) * 0.5).to(dt)
    z = torch.randn(B, L, ED, device=dev).to(dt)
    Bm, Cm = torch.randn(B, L, N, device=dev).to(dt), torch.randn(B, L, N, device=dev).to(dt)
    d0 = make_scan_inputs(1, 1, ED, seed=1237)
    A_log, D, bias = cuda(d0["A_log"]), cuda(d0["D"]), cuda(d0["bias"])
    out = selective_scan_fn(u, draw, A_log, Bm, Cm, D, z=z, dt_bias=bias)
    # (1) oracle on batch row 3, first 1024 steps (causal => comparable)
    sl = slice(3, 4)
    want = orc.selscan_seq_fwd(*(t[sl, :1024].float().cpu().numpy() for t in (u, draw)), d0["A_log"],
                               Bm[sl, :1024].float().cpu().numpy(), Cm[sl, :1024].float().cpu().numpy(), d0["D"],
                               z=z[sl, :1024].float().cpu().numpy(), dt_bias=d0["bias"])
    assert relerr(out[sl, :1024], want) < 2e-2
    # (2) prefix invariance + batch independence: rows 0..1, first 2048 steps, computed alone
    out2 = selective_scan_fn(u[:2, :2048], draw[:2, :2048], A_log, Bm[:2, :2048], Cm[:2, :2048], D, z=z[:2, :2048], dt_bias=bias)
    assert relerr(out2, out[:2, :2048]) < 1e-2
    # (3) linearity in u (fp32 accumulate, bf16 output rounding only)
    out_s = selective_scan_fn((u * 2).to(dt), draw, A_log, Bm, Cm, D, z=z, dt_bias=bias)
    assert relerr(out_s, out.float() * 2) < 1e-2


def _full_size_case(B, L, ED, dt, seed):
    N = 16
    torch.manual_seed(seed)
    dev = "cuda"
    t = dict(u=torch.randn(B, L, ED, device=dev).to(dt), draw=(torch.randn(B, L, ED, device=dev) * 0.5).to(dt),
             z=torch.randn(B, L, ED, device=dev).to(dt), Bm=torch.randn(B, L, N, device=dev).to(dt),
             Cm=torch.randn(B, L, N, device=dev).to(dt), dout=torch.randn(B, L, ED, device=dev).to(dt))
    d0 = make_scan_inputs(1, 1, ED, seed=seed)
    return t, d0


def _fwd_bwd(t, d0, rows=slice(None), scale=1.0):
    from gfe_mamba_b200 import selective_scan_fn
    leaves = {k: t[k][rows].detach().clone().requires_grad_() for k in ("u", "draw", "z", "Bm", "Cm")}
    par = {k: cuda(d0[k], grad=True) for k in ("A_log", "D", "bias")}
    out = selective_scan_fn(leaves["u"], leaves["draw"], par["A_log"], leaves["Bm"], leaves["Cm"], par["D"], z=leaves["z"],
                            dt_bias=par["bias"])
    out.backward((t["dout"][rows].float() * scale).to(out.dtype))
    g = {k: v.grad for k, v in leaves.items()}
    g.update({k: v.grad for k, v in par.items()})
    return out.detach(), g


@pytest.mark.parametrize("name,B,L,ED,dt,tol", [("cfg3", 16, 4096, 1536, torch.bfloat16, 2e-2),
                                                ("cfg5", 256, 1024, 1024, torch.float32, 1e-4),
                                                ("cfg4", 1, 65536, 1024, torch.float32, 1e-4)])
def test_full_size_backward_properties(name, B, L, ED, dt, tol):
    """BASELINE configs 3, 5 and 4 at FULL size, forward + backward, through size-independent properties:
    (1) one batch row computed alone (another kernel variant: the L-split pair) gives the same row of every activation
    gradient; (2) that row agrees with the fp64 oracle; (3) the gradients are linear in dout; (4) dD, which has the closed
    form sum dout * silu(z) * u, matches a plain torch reduction over the whole batch."""
    t, d0 = _full_size_case(B, L, ED, dt, seed=4242)
    out, g = _fwd_bwd(t, d0)
    r = min(5, B - 1)
    Lo = min(L, 4096)                                   # the oracle leg is bounded (cfg4: prefix of the output only)
    if B > 1:
        out1, g1 = _fwd_bwd(t, d0, rows=slice(r, r + 1))
        assert relerr(out1, out[r:r + 1]) < tol
        for k in ("u", "draw", "z", "Bm", "Cm"):
            assert relerr(g1[k], g[k][r:r + 1]) < tol, (name, k)
    rnd = lambda x: x[r:r + 1].float().cpu().numpy()
    if L <= 4096:
        want = oracle_fused(dict(u=rnd(t["u"]), draw=rnd(t["draw"]), z=rnd(t["z"]), Bm=rnd(t["Bm"]), Cm=rnd(t["Cm"]),
                                 dout=rnd(t["dout"]), A_log=d0["A_log"], D=d0["D"], bias=d0["bias"]), torch.float32)
        assert relerr(out[r:r + 1], want["out"]) < tol
        for k, kk in (("u", "du"), ("draw", "ddelta"), ("z", "dz"), ("Bm", "dB"), ("Cm", "dC")):
            assert relerr(g[k][r:r + 1], want[kk]) < (tol if B == 1 else 2 * tol), (name, k)   # dB/dC rows are per batch row
    else:   # causal prefix of the forward output against the oracle
        pre = lambda x: x[:, :Lo].float().cpu().numpy()
        want = orc.selscan_seq_fwd(pre(t["u"]), pre(t["draw"]), d0["A_log"], pre(t["Bm"]), pre(t["Cm"]), d0["D"], z=pre(t["z"]),
                                   dt_bias=d0["bias"])
        assert relerr(out[:, :Lo], want) < tol
    _, g2 = _fwd_bwd(t, d0, scale=2.0)
    for k in ("u", "draw", "z", "Bm", "Cm", "A_log", "D", "bias"):
        assert relerr(g2[k], g[k].float() * 2) < max(tol, 1e-3) , (name, k)
    zf, uf, df = t["z"].float(), t["u"].float(), t["dout"].float()
    dD_ref = (df * (zf * torch.sigmoid(zf)) * uf).sum(dim=(0, 1))
    assert relerr(g["D"], dD_ref) < max(tol, 1e-3), name


@pytest.mark.parametrize("rows", [1, 2, 5])
def test_host_pipeline_matches_oracle_and_direct_call(rows):
    """Host-buffer entry point (pinned host in/out, H2D | fwd+bwd | D2H overlapped over row chunks): same numbers as the
    oracle and, row for row, as the device-tensor call (the chunk's batch size may select another kernel variant, so the
    comparison is to tolerance, not bitwise); parameter gradients are summed over the chunks."""
    from gfe_mamba_b200.host_pipeline import HostScanPipeline
    B, L, ED, N = 5, 70, 64, 16
    d = make_scan_inputs(B, L, ED, seed=77)
    host_in = {k: torch.from_numpy(d[s]).pin_memory() for k, s in
               (("u", "u"), ("delta", "draw"), ("z", "z"), ("Bm", "Bm"), ("Cm", "Cm"), ("dout", "dout"))}
    host_out = {k: torch.empty((B, L, N if k in ("dBm", "dCm") else ED)).pin_memory() for k in ("out", "du", "ddelta", "dz", "dBm", "dCm")}
    A_log, D, bias = cuda(d["A_log"]), cuda(d["D"]), cuda(d["bias"])
    pipe = HostScanPipeline(B, L, ED, N, torch.float32, torch.device("cuda"), rows_per_chunk=rows)
    for _ in range(2):   # second run reuses the double buffers
        dA_log, dD, dbias = pipe.run(host_in, A_log, D, bias, host_out)
        torch.cuda.synchronize()
    got = dict(out=host_out["out"], du=host_out["du"], ddelta=host_out["ddelta"], dz=host_out["dz"], dB=host_out["dBm"],
               dC=host_out["dCm"], dA_log=dA_log, dD=dD, ddt_bias=dbias)
    compare(got, oracle_fused(d, torch.float32), TOL[torch.float32])
    direct = run_fused(d, torch.float32)
    for k in ("out", "du", "ddelta", "dz", "dB", "dC"):
        assert relerr(got[k], direct[k]) < 1e-5, k
    assert pipe.h2d_bytes == 4 * (4 * B * L * ED + 2 * B * L * N) and pipe.d2h_bytes == 4 * (4 * B * L * ED + 2 * B * L * N)


# ------------------------------------------------------------------------------- residual add + RMSNorm (SURVEY 8f rank 1)
@pytest.mark.parametrize("rows,D,dtype", [(7, 128, torch.float32), (300, 768, torch.float32), (1000, 256, torch.bfloat16),
                                          (33, 1024, torch.float32), (65, 2048, torch.bfloat16), (5, 512, torch.float16),
                                          (1, 4, torch.float32),
                                          (70, 4096, torch.float32), (19, 8192, torch.bfloat16), (600, 1028, torch.float32)])   # wider than the register-resident row: two-pass kernels
@pytest.mark.parametrize("with_add", [True, False])
def test_add_rmsnorm_vs_torch(rows, D, dtype, with_add):
    """resid = x + a; y = x * rsqrt(mean(x^2) + eps) * w exactly as cross_atten/mamba.py:103 and :408-418, forward and backward
    (dx, da, dw), against the same expression in torch fp64 on the inputs as the kernel sees them."""
    from gfe_mamba_b200 import add_rmsnorm
    g = torch.Generator(device="cpu").manual_seed(rows * 7 + D)
    x = torch.randn(rows, D, generator=g).to(dtype).cuda().requires_grad_()
    a = torch.randn(rows, D, generator=g).to(dtype).cuda().requires_grad_() if with_add else None
    w = (1 + 0.1 * torch.randn(D, generator=g)).cuda().requires_grad_()
    dres, dy = torch.randn(rows, D, generator=g).to(dtype).cuda(), torch.randn(rows, D, generator=g).to(dtype).cuda()
    resid, y = add_rmsnorm(x, a, w, 1e-5)
    (resid.float() * dres.float()).sum().add((y.float() * dy.float()).sum()).backward()
    xd = x.detach().double().requires_grad_()
    ad = a.detach().double().requires_grad_() if with_add else None
    wd = w.detach().double().requires_grad_()
    rd = (xd + ad).detach().to(dtype).double() + ((xd + ad) - (xd + ad).detach()) if with_add else xd   # value rounded to dtype, gradient of the sum
    yd = rd * torch.rsqrt(rd.pow(2).mean(-1, keepdim=True) + 1e-5) * wd
    ((rd * dres.double()).sum() + (yd * dy.double()).sum()).backward()
    tol = TOL[dtype]
    assert relerr(resid, rd.detach()) < tol and relerr(y, yd.detach()) < tol
    assert relerr(x.grad, xd.grad) < tol and relerr(w.grad, wd.grad) < tol
    if with_add:
        assert relerr(a.grad, ad.grad) < tol


@pytest.mark.parametrize("rows,D,io", [(300, 512, torch.bfloat16), (37, 768, torch.float16), (5, 4, torch.bfloat16),
                                       (40, 4096, torch.bfloat16)])   # the last one: two-pass kernels
@pytest.mark.parametrize("with_add", [True, False])
def test_add_rmsnorm_mixed_dtypes(rows, D, io, with_add):
    """fp32 residual stream with a 16-bit branch (the stack under autocast): resid = x + a in fp32, y in the branch dtype;
    backward dx in fp32 and da in the branch dtype from the same pass.  Against torch fp64 on the inputs as the kernel sees them."""
    from gfe_mamba_b200 import add_rmsnorm
    g = torch.Generator(device="cpu").manual_seed(rows + D)
    x = torch.randn(rows, D, generator=g).cuda().requires_grad_()
    a = torch.randn(rows, D, generator=g).to(io).cuda().requires_grad_() if with_add else None
    w = (1 + 0.1 * torch.randn(D, generator=g)).cuda().requires_grad_()
    dres, dy = torch.randn(rows, D, generator=g).cuda(), torch.randn(rows, D, generator=g).to(io).cuda()
    resid, y = add_rmsnorm(x, a, w, 1e-5, out_dtype=io)
    assert resid.dtype == torch.float32 and y.dtype == io
    (resid * dres).sum().add((y.float() * dy.float()).sum()).backward()
    xd = x.detach().double().requires_grad_()
    ad = a.detach().double().requires_grad_() if with_add else None
    wd = w.detach().double().requires_grad_()
    rd = (xd + ad).detach().float().double() + ((xd + ad) - (xd + ad).detach()) if with_add else xd
    yd = rd * torch.rsqrt(rd.pow(2).mean(-1, keepdim=True) + 1e-5) * wd
    ((rd * dres.double()).sum() + (yd * dy.double()).sum()).backward()
    assert relerr(resid, rd.detach()) < 1e-6 and relerr(y, yd.detach()) < TOL[io]
    assert relerr(x.grad, xd.grad) < 1e-5 and relerr(w.grad, wd.grad) < 1e-4
    if with_add:
        assert a.grad.dtype == io and relerr(a.grad, ad.grad) < TOL[io]
        assert torch.equal(a.grad, x.grad.to(io))            # the same values, rounded once


def test_add_rmsnorm_picks_the_autocast_dtype():
    """Under CUDA autocast an fp32 stream hands the next mixer its input in the autocast dtype (no cast kernel), and only then."""
    from gfe_mamba_b200 import add_rmsnorm
    x = torch.randn(8, 64, device="cuda")
    w = torch.ones(64, device="cuda")
    assert add_rmsnorm(x, None, w)[1].dtype == torch.float32
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert add_rmsnorm(x, None, w)[1].dtype == torch.bfloat16
        assert add_rmsnorm(x, x.bfloat16(), w)[1].dtype == torch.bfloat16
        assert add_rmsnorm(x, x, w)[1].dtype == torch.float32          # an fp32 branch is not rounded behind the caller's back
        assert add_rmsnorm(x.bfloat16(), None, w)[1].dtype == torch.bfloat16


def test_mamba_stack_fused_norm_matches_layerwise():
    """Mamba.forward with the residual adds fused into the next RMSNorm == the reference's layer-by-layer formulation."""
    from gfe_mamba_b200 import Mamba, MambaConfig
    torch.manual_seed(3)
    model = Mamba(MambaConfig(d_model=64, n_layers=3)).cuda()
    x = torch.randn(2, 50, 64, device="cuda", requires_grad=True)
    y = model(x)
    y.square().mean().backward()
    gx = x.grad.clone()
    gp = {n: p.grad.clone() for n, p in model.named_parameters()}
    model.zero_grad(); x.grad = None
    h = x
    for layer in model.layers:          # ResidualBlock.forward: mixer(norm(x)) + x with the torch RMSNorm module
        h = layer(h)
    h.square().mean().backward()
    assert relerr(y, h) < 1e-5 and relerr(gx, x.grad) < 1e-4
    for n, p in model.named_parameters():
        assert relerr(gp[n], p.grad) < 1e-4, n


def test_graphed_decoder_matches_step_loop():
    """CUDA-graph decode (gfe_mamba_b200.decode.GraphedDecoder) == Mamba.step token by token == Mamba.forward."""
    from gfe_mamba_b200 import Mamba, MambaConfig
    from gfe_mamba_b200.decode import GraphedDecoder
    torch.manual_seed(11)
    cfg = MambaConfig(d_model=64, n_layers=3)
    model = Mamba(cfg).cuda().eval()
    B, T = 4, 12
    x = torch.randn(B, T, cfg.d_model, device="cuda")
    with torch.no_grad():
        want = model(x)
        caches = [(None, torch.zeros(B, cfg.d_inner, cfg.d_conv - 1, device="cuda")) for _ in range(cfg.n_layers)]
        eager = []
        for t in range(T):
            yt, caches = model.step(x[:, t], caches)
            eager.append(yt)
        dec = GraphedDecoder(model, B)
        graphed = [dec.step(x[:, t]).clone() for t in range(T)]
    for t in range(T):
        assert relerr(graphed[t], eager[t]) < 1e-6, t
        assert relerr(graphed[t], want[:, t]) < 1e-4, t


def test_error_behaviour():
    from gfe_mamba_b200 import selective_scan_fn, pscan
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pscan(torch.rand(1, 4, 2, 2), torch.rand(1, 4, 2, 2))
    d = make_scan_inputs(1, 8, 32)
    with pytest.raises(ValueError):
        selective_scan_fn(cuda(d["u"]), cuda(d["draw"])[:, :4], cuda(d["A_log"]), cuda(d["Bm"]), cuda(d["Cm"]), cuda(d["D"]))
