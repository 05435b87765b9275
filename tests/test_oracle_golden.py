"""Pins the CPU oracle (oracle/) against fixtures produced by the unmodified reference
(tests/golden/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest

from oracle import oracle as orc


def _load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name + ".npz")))


def relerr(a, b):
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max() / max(np.abs(b).max(), 1e-30))


@pytest.mark.parametrize("L", [1, 2, 3, 4, 5, 8, 37, 64])
def test_pscan_bit_exact(golden_dir, L):
    """The Blelloch restatement follows pscan.py op for op -> bit-identical fp32 results."""
    g = _load(golden_dir, "pscan_small")
    H = orc.pscan_fwd(g[f"L{L}_A"], g[f"L{L}_X"])
    assert np.array_equal(H, g[f"L{L}_H"]), relerr(H, g[f"L{L}_H"])
    dA, dX = orc.pscan_bwd(g[f"L{L}_A"], g[f"L{L}_H"], g[f"L{L}_dH"])
    assert np.array_equal(dX, g[f"L{L}_dX"]), relerr(dX, g[f"L{L}_dX"])
    assert np.array_equal(dA, g[f"L{L}_dA"]), relerr(dA, g[f"L{L}_dA"])


@pytest.mark.parametrize("L", [1, 2, 3, 5, 37, 64])
def test_pscan_vs_fp64_sequential(golden_dir, L):
    g = _load(golden_dir, "pscan_small")
    H64 = orc.pscan_seq64(g[f"L{L}_A"], g[f"L{L}_X"])
    assert relerr(g[f"L{L}_H"], H64) < 1e-6


def test_npo2():
    for L, want in [(1, 1), (2, 2), (3, 4), (4, 4), (5, 8), (37, 64), (64, 64), (1858, 2048), (4096, 4096), (65536, 65536)]:
        assert orc.npo2(L) == want


@pytest.mark.parametrize("tag", ["L37", "L64"])
def test_selscan_ref_style(golden_dir, tag):
    """Materialising restatement of MambaBlock.selective_scan; expf differs from torch's vectorised exp by <= 1 ulp."""
    g = _load(golden_dir, "selscan_small")
    a = [g[f"{tag}_{k}"] for k in ("x", "delta", "A", "B", "C", "D")]
    y = orc.selscan_ref_fwd(*a)
    assert relerr(y, g[f"{tag}_y"]) < 2e-6
    assert relerr(y, g[f"{tag}_y_seq"]) < 2e-6
    gr = orc.selscan_ref_bwd(*a, g[f"{tag}_dy"])
    for k in ("dx", "ddelta", "dA", "dB", "dC", "dD"):
        assert relerr(gr[k], g[f"{tag}_{k}"]) < 5e-6, k


@pytest.mark.parametrize("tag", ["L37", "L64"])
def test_selscan_seq_fused(golden_dir, tag):
    """fp64 sequential fused form == reference selective_scan / selective_scan_seq (no softplus, no gate)."""
    g = _load(golden_dir, "selscan_small")
    A_log = np.log(-g[f"{tag}_A"])
    y = orc.selscan_seq_fwd(g[f"{tag}_x"], g[f"{tag}_delta"], A_log, g[f"{tag}_B"], g[f"{tag}_C"], g[f"{tag}_D"],
                            softplus=False)
    assert relerr(y, g[f"{tag}_y"]) < 2e-6
    gr = orc.selscan_seq_bwd(g[f"{tag}_x"], g[f"{tag}_delta"], A_log, g[f"{tag}_B"], g[f"{tag}_C"], g[f"{tag}_D"],
                             g[f"{tag}_dy"], softplus=False)
    assert relerr(gr["du"], g[f"{tag}_dx"]) < 5e-6
    assert relerr(gr["ddelta"], g[f"{tag}_ddelta"]) < 5e-6
    assert relerr(gr["dB"], g[f"{tag}_dB"]) < 5e-6
    assert relerr(gr["dC"], g[f"{tag}_dC"]) < 5e-6
    assert relerr(gr["dD"], g[f"{tag}_dD"]) < 5e-6
    # reference differentiates w.r.t. A; the fused form w.r.t. A_log: dA_log = dA * A
    assert relerr(gr["dA_log"], g[f"{tag}_dA"] * g[f"{tag}_A"]) < 5e-6


def _block_params(g):
    return {k[3:]: v for k, v in g.items() if k.startswith("sd.")}


def test_block_forward(golden_dir):
    g = _load(golden_dir, "block_small")
    d_model, d_state, _, _, dt_rank, _, _ = (int(v) for v in g["meta"])
    y = orc.block_forward(_block_params(g), g["x"], d_state, dt_rank)
    assert relerr(y, g["y"]) < 5e-6


def test_block_step_matches_forward(golden_dir):
    """Reference redundancy (ii) of SURVEY 4: step() replay == forward()."""
    g = _load(golden_dir, "block_small")
    assert relerr(g["y_step"], g["y"]) < 5e-6


def test_block_fused_grads(golden_dir):
    """Fused-op backward (softplus + bias + gate inside) against the reference's autograd through the block."""
    g = _load(golden_dir, "block_small")
    p = _block_params(g)
    d_model, d_state, _, d_conv, dt_rank, B, L = (int(v) for v in g["meta"])
    ED = p["A_log"].shape[0]
    x = g["x"]
    xz = x @ p["in_proj.weight"].T
    xin, z = np.ascontiguousarray(xz[..., :ED]), np.ascontiguousarray(xz[..., ED:])
    u = orc.conv1d_silu_fwd(xin, p["conv1d.weight"], p["conv1d.bias"])
    dbc = u @ p["x_proj.weight"].T
    dt, Bm, Cm = dbc[..., :dt_rank], dbc[..., dt_rank:dt_rank + d_state], dbc[..., dt_rank + d_state:]
    draw = dt @ p["dt_proj.weight"].T
    dgate = g["dy"] @ p["out_proj.weight"]                                  # d(out_proj input)
    gr = orc.selscan_seq_bwd(u, draw, p["A_log"], Bm, Cm, p["D"], dgate, z=z, dt_bias=p["dt_proj.bias"])
    assert relerr(gr["dA_log"], g["grad.A_log"]) < 1e-5
    assert relerr(gr["dD"], g["grad.D"]) < 1e-5
    assert relerr(gr["ddt_bias"], g["grad.dt_proj.bias"]) < 1e-5
    # chain the rest by hand: x_proj / dt_proj / conv / in_proj
    ddt = gr["ddelta"] @ p["dt_proj.weight"]
    ddbc = np.concatenate([ddt, gr["dB"], gr["dC"]], -1)
    assert relerr(np.einsum("blr,blc->rc", ddbc, u), g["grad.x_proj.weight"]) < 1e-5
    assert relerr(np.einsum("ble,blr->er", gr["ddelta"], dt), g["grad.dt_proj.weight"]) < 1e-5
    du_total = gr["du"] + ddbc @ p["x_proj.weight"]
    dxin, dw, db = orc.conv1d_silu_bwd(xin, p["conv1d.weight"], p["conv1d.bias"], du_total)
    assert relerr(dw, g["grad.conv1d.weight"]) < 1e-5
    assert relerr(db, g["grad.conv1d.bias"]) < 1e-5
    dxz = np.concatenate([dxin, gr["dz"]], -1)
    assert relerr(dxz @ p["in_proj.weight"], g["dx"]) < 1e-5
    assert relerr(np.einsum("blo,bli->oi", dxz, x), g["grad.in_proj.weight"]) < 1e-5


def test_ssm_step(golden_dir):
    g = _load(golden_dir, "block_small")
    p = _block_params(g)
    _, d_state, _, d_conv, dt_rank, B, L = (int(v) for v in g["meta"])
    ED = p["A_log"].shape[0]
    h, inputs = None, np.zeros((B, ED, d_conv - 1), np.float32)
    w = p["conv1d.weight"].reshape(ED, d_conv)
    for t in range(L):
        xz = g["x"][:, t] @ p["in_proj.weight"].T
        xin, z = xz[:, :ED], xz[:, ED:]
        win = np.concatenate([inputs, xin[:, :, None]], 2)                  # mamba.py:357-358
        v = (win * w[None]).sum(-1) + p["conv1d.bias"]
        u = orc._silu(v)
        dbc = u @ p["x_proj.weight"].T
        dt, Bm, Cm = dbc[:, :dt_rank], dbc[:, dt_rank:dt_rank + d_state], dbc[:, dt_rank + d_state:]
        delta = orc._softplus(dt @ p["dt_proj.weight"].T + p["dt_proj.bias"])
        y, h = orc.ssm_step(u, delta, p["A_log"], Bm, Cm, p["D"], h)
        out = (y * orc._silu(z)) @ p["out_proj.weight"].T
        assert relerr(out, g["y_step"][:, t]) < 1e-5
        inputs = win[:, :, 1:]
    assert relerr(h, g["h_last"]) < 1e-5
    assert relerr(inputs, g["inputs_last"]) < 1e-6


def test_mamba_cfg1_forward(mamba_cfg1):
    """BASELINE config 1 end to end (2 layers, RMSNorm + residual)."""
    g = mamba_cfg1
    d_model, n_layers, d_state, _, _, dt_rank, _, _ = (int(v) for v in g["meta"])
    sd = {k[3:]: v for k, v in g.items() if k.startswith("sd.")}
    y = orc.mamba_forward(sd, g["x"], n_layers, d_state, dt_rank)
    assert relerr(y, g["y"]) < 1e-5
