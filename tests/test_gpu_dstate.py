"""d_state = 32 and 64 on the fused kernels: the generic selective-scan kernels, the decode kernel and every layer above them.

Like test_gpu_kernel_matrix.py, each case first proves which path it reached: the library's launch registry must show the
generic selscan kernels (summary passes exactly when plan_segments splits L) and no pscan kernel, i.e. not the reference's
(B, L, ED, N) composition.  Results are then compared with the fp64 oracle on the rounded inputs, or, for the modules, with
the op-by-op composition that other state sizes take.
Tolerances: max-normalised per tensor, fp32 1e-4, 16-bit 2e-2; per channel 1e-3 in fp32 for small step sizes.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as orc

pytestmark = pytest.mark.gpu

NS = [32, 64]
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
TOL = {torch.float32: 1e-4, torch.bfloat16: 2e-2, torch.float16: 2e-2}
R_UNALIGNED = 5   # B and C as slices of a (B, L, R + 2N) tensor starting 5 elements into each row


# ------------------------------------------------------------------------------------------------- helpers
def relerr(a, b):
    a = a.detach().float().cpu().numpy().astype(np.float64) if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = b.detach().float().cpu().numpy().astype(np.float64) if torch.is_tensor(b) else np.asarray(b, np.float64)
    assert a.shape == b.shape, (a.shape, b.shape)
    assert np.isfinite(a).all(), "non-finite values from the CUDA path"
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def compare(got, want, tol, keys=("out", "du", "ddelta", "dz", "dB", "dC", "dA_log", "dD", "ddt_bias")):
    errs = {}
    for k in keys:
        if want.get(k) is None:
            assert got.get(k) is None, k
            continue
        errs[k] = relerr(got[k], want[k])
    bad = {k: v for k, v in errs.items() if not v <= tol}
    assert not bad, f"over tolerance {tol}: {bad} (all: {errs})"
    return errs


def scan_inputs(B, L, ED, N, seed):
    """SURVEY 8d's synthetic inputs: A_log = log(1..N) + jitter, dt_bias as mamba.py:150-155."""
    r = np.random.default_rng(seed)
    f = lambda *s: r.standard_normal(s).astype(np.float32)
    dt = np.exp(r.uniform(np.log(1e-3), np.log(1e-1), ED)).clip(min=1e-4)
    return dict(u=f(B, L, ED), draw=0.5 * f(B, L, ED), z=f(B, L, ED), Bm=f(B, L, N), Cm=f(B, L, N),
                A_log=(np.log(np.arange(1, N + 1, dtype=np.float32))[None].repeat(ED, 0) + 0.1 * f(ED, N)).astype(np.float32),
                D=(1.0 + 0.1 * f(ED)).astype(np.float32), bias=(dt + np.log(-np.expm1(-dt))).astype(np.float32),
                dout=f(B, L, ED))


def launches(fn):
    """Run fn() with the library's launch registry on; returns (fn's result, {kernel name: launches})."""
    from gfe_mamba_b200 import _native
    _native.timing_collect()
    _native.timing_enable(True)
    try:
        res = fn()
        torch.cuda.synchronize()
        got = {k: n for k, (_, n) in _native.timing_collect().items()}
    finally:
        _native.timing_enable(False)
        _native.timing_collect()
    return res, got


def split_along_l(B, L, ED):
    """plan_segments (api.cu): the generic kernels split L when B * ceil(ED / 32) warps fill less than half the schedulers."""
    smsp = 4 * torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    nwarps = B * -(-ED // 32)
    if nwarps * 2 >= smsp:
        return False
    S = max(1, min(-(-2 * smsp // nwarps), L // 128, 256))
    seg_len = max(16, -(-(-(-L // S)) // 16) * 16)
    return -(-L // seg_len) > 1


def assert_generic(B, L, ED, got, grad=True, split=None):
    """The generic kernels ran (for every ED, also multiples of 32), with summaries iff L is split, and nothing else."""
    s = split_along_l(B, L, ED)
    if split is not None:
        assert s == split, f"the launch plan of {(B, L, ED)} does not give this schedule"
    want = {"selscan_fwd": 1}
    if s:
        want["selscan_fwd_summary"] = 1
    if grad:
        want.update(selscan_bwd=1, selscan_bwd_finalize_bc=1, selscan_bwd_finalize_par=1)
        if s:
            want["selscan_bwd_summary"] = 1
    assert got == want, f"launched {got}, expected {want}"


def _np(x):
    return None if x is None else x.detach().float().cpu().numpy()


def prep(d, dtype, *, use_z=True, use_bias=True, softplus=True, R=None, strided=False):
    """Device leaves.  R: B and C are slices [R, R+N), [R+N, R+2N) of one tensor.  strided: u and z are the two halves of
    one (B, L, 2 ED) tensor (in_proj's output)."""
    B, L, ED = d["u"].shape
    N = d["Bm"].shape[-1]
    leaf = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dtype).requires_grad_()
    t = dict(draw=leaf(d["draw"]), uz=None, bc=None)
    if strided:
        t["uz"] = leaf(np.concatenate([d["u"], d["z"]], -1))
        t["u"], t["z"] = t["uz"][..., :ED], (t["uz"][..., ED:] if use_z else None)
    else:
        t["u"], t["z"] = leaf(d["u"]), (leaf(d["z"]) if use_z else None)
    if R is None:
        t["Bm"], t["Cm"] = leaf(d["Bm"]), leaf(d["Cm"])
    else:
        t["bc"] = leaf(np.concatenate([np.zeros((B, L, R), np.float32), d["Bm"], d["Cm"]], -1))
        t["Bm"], t["Cm"] = t["bc"][..., R:R + N], t["bc"][..., R + N:]
    f32 = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda().requires_grad_()
    t["A_log"], t["D"] = f32(d["A_log"]), f32(d["D"])
    t["bias"] = f32(d["bias"]) if use_bias else None
    t["dout"] = torch.from_numpy(d["dout"]).to("cuda", dtype)
    t["softplus"] = softplus
    t["N"], t["ED"] = N, ED
    return t


def run(t, grad=True, last=False):
    from gfe_mamba_b200 import selective_scan_fn
    with torch.set_grad_enabled(grad):
        res = selective_scan_fn(t["u"], t["draw"], t["A_log"], t["Bm"], t["Cm"], t["D"], z=t["z"], dt_bias=t["bias"],
                                delta_softplus=t["softplus"], return_last_state=last)
    out, hl = res if last else (res, None)
    g = dict(out=out.detach(), last=hl)
    if grad:
        out.backward(t["dout"])
        N, ED = t["N"], t["ED"]
        if t["uz"] is not None:
            du, dz = t["uz"].grad[..., :ED], (t["uz"].grad[..., ED:] if t["z"] is not None else None)
        else:
            du, dz = t["u"].grad, (None if t["z"] is None else t["z"].grad)
        if t["bc"] is not None:
            R = t["bc"].shape[-1] - 2 * N
            dB, dC = t["bc"].grad[..., R:R + N], t["bc"].grad[..., R + N:]
        else:
            dB, dC = t["Bm"].grad, t["Cm"].grad
        g.update(du=du, ddelta=t["draw"].grad, dz=dz, dB=dB, dC=dC, dA_log=t["A_log"].grad, dD=t["D"].grad,
                 ddt_bias=None if t["bias"] is None else t["bias"].grad)
    return g


def oracle(t, grad=True, last=False):
    """fp64 oracle on the values the kernels read (the rounded leaves)."""
    a = {k: _np(t[k]) for k in ("u", "draw", "z", "Bm", "Cm", "A_log", "D", "bias")}
    res = orc.selscan_seq_fwd(a["u"], a["draw"], a["A_log"], a["Bm"], a["Cm"], a["D"], z=a["z"], dt_bias=a["bias"],
                              softplus=t["softplus"], return_last_state=last)
    out, hl = res if last else (res, None)
    g = dict(out=out, last=hl)
    if grad:
        g.update(orc.selscan_seq_bwd(a["u"], a["draw"], a["A_log"], a["Bm"], a["Cm"], a["D"], _np(t["dout"]), z=a["z"],
                                     dt_bias=a["bias"], softplus=t["softplus"]))
    return g


def positive_delta(d):
    """delta_softplus=False: delta + dt_bias must already be a step size."""
    d = dict(d)
    d["draw"] = np.abs(d["draw"]) * 0.2 + 1e-3
    d["bias"] = np.abs(d["bias"]) * 0.01
    return d


# ------------------------------------------------------------------------------------------------- the scan matrix
# ED not a multiple of 32 (partial last warp) and a multiple of 32 (which at d_state = 16 would take the chained kernels)
SHAPES = {("ED40", False): (2, 203, 40), ("ED1000", False): (2, 203, 1000), ("ED64", False): (8, 203, 64),
          ("ED40", True): (1, 2100, 40), ("ED1000", True): (1, 1858, 1000), ("ED64", True): (1, 2100, 64)}


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("gate", [True, False], ids=["z", "noz"])
@pytest.mark.parametrize("shape,split", list(SHAPES), ids=[f"{s}-{'split' if p else 'nosplit'}" for s, p in SHAPES])
@pytest.mark.parametrize("N", NS)
def test_scan_matrix(N, shape, split, gate, dt):
    """selscan_{fwd,bwd}_kernel<T, HAS_Z, N> (+ both summary passes with the L-split): every output and gradient."""
    dtype = DTYPES[dt]
    B, L, ED = SHAPES[(shape, split)]
    t = prep(scan_inputs(B, L, ED, N, seed=N + ED + L + gate), dtype, use_z=gate)
    got, n = launches(lambda: run(t))
    assert_generic(B, L, ED, n, split=split)
    compare(got, oracle(t), TOL[dtype])


@pytest.mark.parametrize("sched", ["nosplit", "split"])
@pytest.mark.parametrize("dt,use_bias,softplus", [("f32", False, True), ("bf16", True, False), ("f16", False, False)])
@pytest.mark.parametrize("N", NS)
def test_flags_and_views(N, dt, use_bias, softplus, sched):
    """dt_bias=None, delta_softplus=False, u / z as strided halves of one tensor and B / C as slices at an unaligned offset,
    all consumed in place."""
    dtype = DTYPES[dt]
    B, L, ED = SHAPES[("ED64", sched == "split")]
    d = scan_inputs(B, L, ED, N, seed=7 * N + B)
    if not softplus:
        d = positive_delta(d)
    t = prep(d, dtype, use_bias=use_bias, softplus=softplus, R=R_UNALIGNED, strided=True)
    assert t["u"].stride(1) == 2 * ED and t["Bm"].stride(1) == R_UNALIGNED + 2 * N
    got, n = launches(lambda: run(t))
    assert_generic(B, L, ED, n, split=sched == "split")
    compare(got, oracle(t), TOL[dtype])


# ------------------------------------------------------------------------------------------------- final state, decode
PATHS = {"nosplit": (2, 203, 40), "split": (1, 2100, 64)}


def per_channel_err(got, want, axis):
    g = np.moveaxis(np.asarray(_np(got) if torch.is_tensor(got) else got, np.float64), axis, 0)
    w = np.moveaxis(np.asarray(want, np.float64), axis, 0)
    assert g.shape == w.shape and np.isfinite(g).all()
    g, w = g.reshape(g.shape[0], -1), w.reshape(w.shape[0], -1)
    return np.abs(g - w).max(1) / np.maximum(np.abs(w).max(1), 1e-30)


@pytest.mark.parametrize("grad", [True, False], ids=["grad", "nograd"])
@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("N", NS)
def test_last_state(N, path, dt, grad):
    dtype = DTYPES[dt]
    B, L, ED = PATHS[path]
    t = prep(scan_inputs(B, L, ED, N, seed=L + ED + N + grad), dtype)
    got, n = launches(lambda: run(t, grad=grad, last=True))
    assert_generic(B, L, ED, n, grad=grad, split=path == "split")
    want = oracle(t, grad=grad, last=True)
    assert got["last"].shape == (B, ED, N) and got["last"].dtype == torch.float32
    assert relerr(got["last"], want["last"]) < (1e-4 if dtype == torch.float32 else 1e-3)
    compare(got, want, TOL[dtype], keys=("out", "du", "ddelta", "dz", "dB", "dC", "dA_log", "dD", "ddt_bias") if grad else ("out",))


def decode_from(t, hl, L, T):
    from gfe_mamba_b200 import ops
    outs, h = [], hl
    with torch.no_grad():
        for s in range(L, L + T):
            y, h = ops.ssm_step(t["u"][:, s], t["draw"][:, s], t["A_log"], t["Bm"][:, s], t["Cm"][:, s], t["D"], h,
                                z=None if t["z"] is None else t["z"][:, s], dt_bias=t["bias"], delta_softplus=t["softplus"])
            outs.append(y)
    return torch.stack(outs, 1), h


def slice_l(d, L):
    return {k: (v[:, :L] if k in ("u", "draw", "z", "Bm", "Cm", "dout") else v) for k, v in d.items()}


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("N", NS)
def test_prefill_then_decode(N, path):
    """Scan L tokens with return_last_state, continue T tokens with ssm_step: one scan over L + T tokens."""
    B, L, ED = PATHS[path]
    T = 6
    d = scan_inputs(B, L + T, ED, N, seed=3 * L + ED + N)
    t = prep(d, torch.float32)
    pre, n = launches(lambda: run(prep(slice_l(d, L), torch.float32), grad=False, last=True))
    assert_generic(B, L, ED, n, grad=False, split=path == "split")
    (ys, h), n = launches(lambda: decode_from(t, pre["last"], L, T))
    assert n == {"ssm_step": T}
    full = oracle(t, grad=False, last=True)
    assert relerr(ys, full["out"][:, L:]) < 1e-4 and relerr(h, full["last"]) < 1e-4
    whole = run(t, grad=False, last=True)
    assert relerr(ys, whole["out"][:, L:]) < 1e-4 and relerr(h, whole["last"]) < 1e-4


@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("N", NS)
def test_small_step_sizes_per_channel(N, path):
    """dt_bias over [-16, -4] across channels: per-channel errors of last_state, dA_log and the decode continuation."""
    B, L, ED = PATHS[path]
    T = 6
    d = scan_inputs(B, L + T, ED, N, seed=17 + ED + N)
    d["bias"] = np.linspace(-16.0, -4.0, ED).astype(np.float32)
    t_pre = prep(slice_l(d, L), torch.float32)
    got, n = launches(lambda: run(t_pre, grad=True, last=True))
    assert_generic(B, L, ED, n, split=path == "split")
    want = oracle(t_pre, grad=True, last=True)
    t = prep(d, torch.float32)
    ys, h = decode_from(t, got["last"], L, T)
    full = oracle(t, grad=False, last=True)
    errs = dict(last_state=per_channel_err(got["last"], want["last"], 1), dA_log=per_channel_err(got["dA_log"], want["dA_log"], 0),
                decode_out=per_channel_err(ys, full["out"][:, L:], 2), decode_h=per_channel_err(h, full["last"], 1))
    worst = {k: float(e.max()) for k, e in errs.items()}
    assert all(v < 1e-3 for v in worst.values()), worst


def _ssm_step_ref(u, delta, A_log, Bm, Cm, D, h, z, bias, softplus):
    dl = delta.astype(np.float64) + (0.0 if bias is None else bias.astype(np.float64))
    if softplus:
        dl = np.where(dl > 20.0, dl, np.log1p(np.exp(np.minimum(dl, 20.0))))
    y, h_new = orc.ssm_step(u, dl.astype(np.float32), A_log, Bm, Cm, D, h)
    y = y.astype(np.float64)
    return (y if z is None else y * (z / (1.0 + np.exp(-z.astype(np.float64))))), h_new


@pytest.mark.parametrize("h0", ["state", "none"])
@pytest.mark.parametrize("gate", [True, False], ids=["z", "noz"])
@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("N", NS)
def test_decode_kernel(N, dt, gate, h0):
    """ssm_step_kernel<T, N> over a few tokens: z as the strided half of in_proj's output, B / C as slices of x_proj's
    output, ED = 200 (a partial 128-channel block); h=None is a zero state; inputs are left unmodified."""
    from gfe_mamba_b200 import ops
    dtype = DTYPES[dt]
    Bsz, ED, T, R = 3, 200, 4, R_UNALIGNED
    r = np.random.default_rng(N + 10 * gate)
    dev = lambda a, dtp=dtype: torch.from_numpy(np.ascontiguousarray(a, np.float32)).to("cuda", dtp)
    p = scan_inputs(1, 1, ED, N, seed=N)
    uz = dev(r.standard_normal((T, Bsz, 2 * ED)))
    delta = dev(r.standard_normal((T, Bsz, ED)) * 0.5)
    dbc = dev(r.standard_normal((T, Bsz, R + 2 * N)))
    A_log, D, bias = dev(p["A_log"], torch.float32), dev(p["D"], torch.float32), dev(p["bias"], torch.float32)
    h = dev(r.standard_normal((Bsz, ED, N)) * 0.5, torch.float32) if h0 == "state" else None
    h_ref = None if h is None else h.cpu().numpy()
    for s in range(T):
        u, z = uz[s, :, :ED], uz[s, :, ED:]
        Bm, Cm = dbc[s, :, R:R + N], dbc[s, :, R + N:]
        before = [v.clone() for v in (uz, delta, dbc) + (() if h is None else (h,))]
        with torch.no_grad():
            (y, h_new), n = launches(lambda: ops.ssm_step(u, delta[s], A_log, Bm, Cm, D, h, z=z if gate else None, dt_bias=bias))
        assert n == {"ssm_step": 1}
        for v, v0 in zip((uz, delta, dbc) + (() if h is None else (h,)), before):
            assert torch.equal(v, v0), "ssm_step modified its input"
        y_ref, h_ref = _ssm_step_ref(_np(u), _np(delta[s]), p["A_log"], _np(Bm), _np(Cm), p["D"], h_ref, _np(z) if gate else None,
                                     p["bias"], True)
        assert h_new.shape == (Bsz, ED, N) and y.dtype == dtype
        assert relerr(y, y_ref) < TOL[dtype], s
        assert relerr(h_new, h_ref) < 1e-4, s
        h = h_new


# ------------------------------------------------------------------------------------------------- modules
def _composition(monkeypatch):
    """MambaBlock's routing with only d_state = 16 fused: d_state = 32 / 64 take the reference's composition (pscan)."""
    from gfe_mamba_b200 import ops
    monkeypatch.setattr(ops, "FUSED_D_STATES", (16,))


def _block(N, d_model=40, seed=5):
    from gfe_mamba_b200 import MambaBlock, MambaConfig
    torch.manual_seed(seed)
    blk = MambaBlock(MambaConfig(d_model=d_model, n_layers=1, d_state=N)).cuda()
    with torch.no_grad():
        blk.A_log.add_(0.1 * torch.randn_like(blk.A_log))
        blk.D.add_(0.1 * torch.randn_like(blk.D))
    return blk


def _fwd_bwd(blk, x0, dy, autocast=None):
    blk.zero_grad(set_to_none=True)
    x = x0.clone().requires_grad_()
    with torch.autocast("cuda", dtype=autocast, enabled=autocast is not None):
        y = blk(x)
    y.float().backward(dy)
    return [y.detach().float(), x.grad.float()] + [p.grad.float().clone() for p in blk.parameters()]


@pytest.mark.parametrize("inner", [True, False], ids=["inner-node", "op-by-op"])
@pytest.mark.parametrize("autocast", [None, torch.bfloat16], ids=["f32", "bf16-autocast"])
@pytest.mark.parametrize("N", NS)
def test_block_forward_backward(N, autocast, inner, monkeypatch):
    """MambaBlock forward + backward on the fused kernels (the one-node inner path, or conv + selective_scan_fn when the
    inner path is switched off) against the reference's composition on the pscan kernel."""
    blk = _block(N)
    B, L = 3, 150
    x0 = torch.randn(B, L, 40, device="cuda")
    dy = torch.randn(B, L, 40, device="cuda")
    assert blk._inner_fusable(torch.empty(1, 1, 2 * blk.config.d_inner, device="cuda"))
    if not inner:
        monkeypatch.setattr(blk, "_inner_fusable", lambda xz: False)
    got, n = launches(lambda: _fwd_bwd(blk, x0, dy, autocast))
    assert_generic(B, L, blk.config.d_inner, {k: v for k, v in n.items() if k.startswith(("selscan", "pscan"))})
    assert ("conv1d_silu_fwd" in n) and not any(k.startswith("pscan") for k in n)
    _composition(monkeypatch)
    want, n2 = launches(lambda: _fwd_bwd(blk, x0, dy, autocast))
    assert "pscan_fwd" in n2 and not any(k.startswith("selscan") for k in n2)
    names = ["y", "dx"] + [nm for nm, _ in blk.named_parameters()]
    tol = 1e-4 if autocast is None else 3e-2
    for nm, ga, gb in zip(names, got, want):
        assert relerr(ga, gb) < tol, nm


@pytest.mark.parametrize("N", NS)
def test_block_step_matches_forward(N, monkeypatch):
    """MambaBlock.step on the decode kernels, token by token == forward == the composition's step."""
    blk = _block(N).eval()
    B, T = 2, 10
    x = torch.randn(B, T, 40, device="cuda")
    with torch.no_grad():
        want = blk(x)

        def steps():
            cache, ys = (None, torch.zeros(B, blk.config.d_inner, blk.config.d_conv - 1, device="cuda")), []
            for s in range(T):
                y, cache = blk.step(x[:, s], cache)
                ys.append(y)
            return torch.stack(ys, 1), cache[0]
        (ys, h), n = launches(steps)
        assert n.get("ssm_step") == T and h.shape == (B, blk.config.d_inner, N)
        _composition(monkeypatch)
        ys_ref, h_ref = steps()
    assert relerr(ys, want) < 1e-4
    assert relerr(ys, ys_ref) < 1e-4 and relerr(h, h_ref) < 1e-4


@pytest.mark.parametrize("N", NS)
def test_stack_forward_mean_autocast(N, monkeypatch):
    """Mamba (2 layers) forward_mean under bf16 autocast, forward and backward, against the composition."""
    from gfe_mamba_b200 import Mamba, MambaConfig
    torch.manual_seed(3)
    model = Mamba(MambaConfig(d_model=64, n_layers=2, d_state=N)).cuda()
    x0 = torch.randn(2, 120, 64, device="cuda")

    def go():
        model.zero_grad(set_to_none=True)
        x = x0.clone().requires_grad_()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = model.forward_mean(x)
        y.float().square().sum().backward()
        return [y.detach().float(), x.grad.float()] + [p.grad.float().clone() for p in model.parameters()]
    got, n = launches(go)
    assert n.get("selscan_fwd") == 2 and n.get("selscan_bwd") == 2 and not any(k.startswith("pscan") for k in n)
    _composition(monkeypatch)
    want = go()
    assert got[0].dtype == torch.float32
    for i, (a, b) in enumerate(zip(got, want)):
        assert relerr(a, b) < 3e-2, i


def test_graphed_decoder_dstate32():
    """CUDA-graph decode of an N = 32 stack == Mamba.step token by token == Mamba.forward."""
    from gfe_mamba_b200 import Mamba, MambaConfig
    from gfe_mamba_b200.decode import GraphedDecoder
    torch.manual_seed(11)
    cfg = MambaConfig(d_model=64, n_layers=3, d_state=32)
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


# ------------------------------------------------------------------------------------------------- memory
@pytest.mark.parametrize("N", NS)
def test_memory_stays_near_checkpoint_and_workspace(N):
    """Production shape (B=2, L=1858, ED=1024), fp32: the composition would hold ~9 (B, L, ED, N) fp32 tensors (several GB);
    the fused forward + backward peaks at the checkpoint + workspace the library reports plus the (B, L, ED) activations."""
    from gfe_mamba_b200 import _native as nat
    B, L, ED = 2, 1858, 1024
    composition = 9 * B * L * ED * N * 4
    assert composition > 4e9
    t = prep(scan_inputs(B, L, ED, N, seed=N), torch.float32)
    l = nat.lib()
    ckpt = l.gfe_selscan_ckpt_bytes_dt(B, L, ED, N, nat.GFE_F32)
    ws = max(l.gfe_selscan_fwd_workspace_bytes(B, L, ED, N), l.gfe_selscan_bwd_workspace_bytes(B, L, ED, N))
    assert ckpt > 0
    act = B * L * ED * 4
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    _, n = launches(lambda: run(t))
    peak = torch.cuda.max_memory_allocated() - base
    assert_generic(B, L, ED, n)
    # out, dout copy, du, ddelta, dz (+ small dB, dC, parameter gradients)
    allowed = 2 * (ckpt + ws) + 6 * act
    assert peak <= allowed, (peak, ckpt, ws)
    assert allowed * 10 < composition
