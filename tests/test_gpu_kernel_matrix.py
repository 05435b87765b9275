"""GPU kernel matrix: every compiled variant of the selective-scan, decode and conv kernels against the fp64 oracle.

The parity suite (test_gpu_parity*.py) is organised by shape; this file is organised by the template instantiations the host
code chooses from at run time, and every case first proves which one it reached:
  * chained kernels (ED % 32 == 0): T in {f32, bf16, f16} x gate x 64- / 32-channel blocks x cp.async (CPB = 16) or plain-load
    staging (CPB = 0, B/C as slices of x_proj's output at an unaligned offset) x waiting or independent L-segments;
  * generic kernels (ED % 32 != 0): every dtype, gated or not, with and without the L-split, partial warps;
  * the final state (return_last_state) of every path, and prefill followed by decode from that state;
  * the decode kernels (ssm_step, conv1d_step) directly, every dtype and flag, strided halves, d_conv 2..4;
  * the unpacked 16-bit conv kernels and a conv backward that sums many tile rows;
  * per-channel errors where delta = softplus(x) is tiny (dt_bias down to -16): a max-normalised error cannot see a channel
    whose values are small.
Path assertions read the library's launch registry (_native.timing_*) and mirror the launch plans (plan_segments in api.cu,
chain_cpb / chain_pair_stores in selscan_chain_host.cu, conv_vec in conv1d.cu), so a change of plan that moves a case onto
another kernel fails here instead of silently testing something else.
Tolerances: as test_gpu_parity.TOL (max-normalised per tensor); per-channel 1e-3 in fp32.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from test_gpu_parity import TOL, compare, cuda, make_scan_inputs, relerr

pytestmark = pytest.mark.gpu

N = 16
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
R_UNALIGNED = 5   # dt_rank of d_model = 65..80: B and C start 5 elements into each row of x_proj's output


# ------------------------------------------------------------------------------------------------- path assertions
def launches(fn):
    """Run fn() with the library's launch registry on; returns (fn's result, {kernel name: launches})."""
    from gfe_mamba_b200 import _native
    _native.timing_collect()   # drop whatever an earlier caller left
    _native.timing_enable(True)
    try:
        res = fn()
        torch.cuda.synchronize()
        got = {k: n for k, (_, n) in _native.timing_collect().items()}
    finally:
        _native.timing_enable(False)
        _native.timing_collect()
    return res, got


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def split_along_l(B, L, ED):
    """plan_segments (api.cu): the generic kernels split L, and the chained kernels make their segments independent, when
    B * ceil(ED / 32) warps fill less than half the schedulers."""
    smsp, nwarps = 4 * _sms(), B * -(-ED // 32)
    if nwarps * 2 >= smsp:
        return False
    S = max(1, min(-(-2 * smsp // nwarps), L // 128, 256))
    seg_len = max(16, -(-(-(-L // S)) // 16) * 16)
    return -(-L // seg_len) > 1


def cpb16(dtype, *staged):
    """chain_cpb (selscan_chain_host.cu): 16-byte cp.async staging when every staged base and batch / row stride is a
    multiple of 16 bytes (the outputs and checkpoints this file passes are fresh allocations, hence aligned)."""
    s = torch.empty((), dtype=dtype).element_size()
    return all(t.data_ptr() % 16 == 0 and (t.stride(0) * s) % 16 == 0 and (t.stride(1) * s) % 16 == 0
               for t in staged if t is not None)


def assert_scan_path(path, B, L, ED, got, grad=True):
    """path: 'generic' | 'generic-split' (ED % 32 != 0) or 'waiting' | 'independent' (chained, ED % 32 == 0)."""
    chained = path in ("waiting", "independent")
    split = path in ("generic-split", "independent")
    assert (ED % 32 == 0) == chained, f"{path}: ED={ED} selects the {'chained' if ED % 32 == 0 else 'generic'} kernels"
    assert split_along_l(B, L, ED) == split, f"{path}: the launch plan of {(B, L, ED)} does not give this schedule"
    want = {"selscan_fwd": 1}
    if split:
        want["selscan_fwd_summary"] = 1
    if grad:
        want.update(selscan_bwd=1, selscan_bwd_finalize_bc=1, selscan_bwd_finalize_par=1)
        if split:
            want["selscan_bwd_summary"] = 1
    assert got == want, f"{path}: launched {got}, expected {want}"


# ------------------------------------------------------------------------------------------------- scan runner
def _prep(d, dtype, *, use_z=True, use_bias=True, softplus=True, R=None):
    """Device leaves in ``dtype``; with R, B and C are the slices [R, R+N) and [R+N, R+2N) of one (B, L, R+2N) tensor."""
    B, L, ED = d["u"].shape
    leaf = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to("cuda", dtype).requires_grad_()
    t = dict(u=leaf(d["u"]), draw=leaf(d["draw"]), z=leaf(d["z"]) if use_z else None)
    if R is None:
        t["Bm"], t["Cm"] = leaf(d["Bm"]), leaf(d["Cm"])
        t["bc"] = None
    else:
        bc = np.concatenate([np.zeros((B, L, R), np.float32), d["Bm"], d["Cm"]], -1)
        t["bc"] = leaf(bc)
        t["Bm"], t["Cm"] = t["bc"][..., R:R + N], t["bc"][..., R + N:]
    t["A_log"], t["D"] = cuda(d["A_log"], grad=True), cuda(d["D"], grad=True)
    t["bias"] = cuda(d["bias"], grad=True) if use_bias else None
    t["dout"] = torch.from_numpy(d["dout"]).to("cuda", dtype)
    t["softplus"] = softplus
    return t


def _run(t, grad=True, last=False):
    from gfe_mamba_b200 import selective_scan_fn
    with torch.set_grad_enabled(grad):
        res = selective_scan_fn(t["u"], t["draw"], t["A_log"], t["Bm"], t["Cm"], t["D"], z=t["z"], dt_bias=t["bias"],
                                delta_softplus=t["softplus"], return_last_state=last)
    out, hl = res if last else (res, None)
    g = dict(out=out.detach(), last=hl)
    if grad:
        out.backward(t["dout"])
        R = None if t["bc"] is None else t["bc"].shape[-1] - 2 * N
        dB = t["Bm"].grad if R is None else t["bc"].grad[..., R:R + N]
        dC = t["Cm"].grad if R is None else t["bc"].grad[..., R + N:]
        g.update(du=t["u"].grad, ddelta=t["draw"].grad, dz=None if t["z"] is None else t["z"].grad, dB=dB, dC=dC,
                 dA_log=t["A_log"].grad, dD=t["D"].grad, ddt_bias=None if t["bias"] is None else t["bias"].grad)
    return g


def _np(x):
    return None if x is None else x.detach().float().cpu().numpy()


def _oracle(t, grad=True, last=False):
    """fp64 oracle on the values the kernels read (the rounded leaves)."""
    a = dict(u=_np(t["u"]), draw=_np(t["draw"]), z=_np(t["z"]), Bm=_np(t["Bm"]), Cm=_np(t["Cm"]), A_log=_np(t["A_log"]),
             D=_np(t["D"]), bias=_np(t["bias"]))
    res = orc.selscan_seq_fwd(a["u"], a["draw"], a["A_log"], a["Bm"], a["Cm"], a["D"], z=a["z"], dt_bias=a["bias"],
                              softplus=t["softplus"], return_last_state=last)
    out, hl = res if last else (res, None)
    g = dict(out=out, last=hl)
    if grad:
        g.update(orc.selscan_seq_bwd(a["u"], a["draw"], a["A_log"], a["Bm"], a["Cm"], a["D"], _np(t["dout"]), z=a["z"],
                                     dt_bias=a["bias"], softplus=t["softplus"]))
    return g


def _positive_delta(d):
    """delta_softplus=False: delta + dt_bias must already be a step size."""
    d = dict(d)
    d["draw"] = np.abs(d["draw"]) * 0.2 + 1e-3
    d["bias"] = np.abs(d["bias"]) * 0.01
    return d


# ------------------------------------------------------------------------------------- chained kernels: the matrix
# (B, L, ED) per (schedule, channel-block width); L ragged.  waiting: B * ED / 32 >= 296 warps, two chained segments;
# independent: one row, 15 segments whose carries come from the summary + combine passes.
CHAIN_SHAPES = {("waiting", 64): (20, 267, 512), ("waiting", 32): (24, 267, 480),
                ("independent", 64): (1, 2100, 64), ("independent", 32): (1, 2100, 96)}
CHAIN_MATRIX = [pytest.param(dt, gate, cpc, cpb, sched, id=f"{dt}-{'z' if gate else 'noz'}-cpc{cpc}-cpb{cpb}-{sched}")
                for sched in ("waiting", "independent") for cpc in (64, 32) for cpb in (16, 0) for gate in (True, False)
                for dt in DTYPES]


@pytest.mark.parametrize("dt,gate,cpc,cpb,sched", CHAIN_MATRIX)
def test_chained_matrix(dt, gate, cpc, cpb, sched):
    """selscan_fwd_v4_kernel / selscan_bwd_chain_kernel <T, HAS_Z, CPB, CPC> (+ selscan_seg_summary_kernel, REV both ways, on
    the independent schedule): every output and gradient against the oracle."""
    dtype = DTYPES[dt]
    B, L, ED = CHAIN_SHAPES[(sched, cpc)]
    assert (64 if ED % 64 == 0 else 32) == cpc
    d = make_scan_inputs(B, L, ED, seed=B * 7 + ED + cpb + gate)
    t = _prep(d, dtype, use_z=gate, R=None if cpb == 16 else R_UNALIGNED)
    assert cpb16(dtype, t["u"], t["draw"], t["z"], t["Bm"], t["Cm"], t["dout"]) == (cpb == 16)
    got, n = launches(lambda: _run(t))
    assert_scan_path(sched, B, L, ED, n)
    compare(got, _oracle(t), TOL[dtype])


@pytest.mark.parametrize("sched", ["waiting", "independent"])
@pytest.mark.parametrize("dt,use_bias,softplus", [("f32", False, True), ("bf16", True, False), ("f16", False, False)])
def test_chained_bias_and_softplus_flags(sched, dt, use_bias, softplus):
    """dt_bias=None and delta_softplus=False on both schedules, on the plain-load staging."""
    dtype = DTYPES[dt]
    B, L, ED = CHAIN_SHAPES[(sched, 32)]
    d = make_scan_inputs(B, L, ED, seed=31 + B)
    if not softplus:
        d = _positive_delta(d)
    t = _prep(d, dtype, use_bias=use_bias, softplus=softplus, R=R_UNALIGNED)
    assert not cpb16(dtype, t["Bm"])
    got, n = launches(lambda: _run(t))
    assert_scan_path(sched, B, L, ED, n)
    compare(got, _oracle(t), TOL[dtype])


# ------------------------------------------------------------------------------------------------- generic kernels
# ED % 32 != 0: partial last warp (ED = 40, 80, 1000) and a single partial warp (ED = 20); L < 256 never splits
GENERIC_SHAPES = {(20, False): (2, 203, 20), (40, False): (2, 203, 40), (80, False): (2, 203, 80), (1000, False): (10, 203, 1000),
                  (20, True): (1, 2100, 20), (40, True): (1, 2100, 40), (80, True): (1, 2100, 80), (1000, True): (2, 1858, 1000)}


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("gate", [True, False], ids=["z", "noz"])
@pytest.mark.parametrize("ED,split", list(GENERIC_SHAPES), ids=[f"ED{e}-{'split' if s else 'nosplit'}" for e, s in GENERIC_SHAPES])
def test_generic_matrix(dt, gate, ED, split):
    """selscan_{fwd,bwd}_kernel<T, HAS_Z>, selscan_fwd_summary_kernel<T>, selscan_bwd_summary_kernel<T, HAS_Z>."""
    dtype = DTYPES[dt]
    B, L, ED = GENERIC_SHAPES[(ED, split)]
    d = make_scan_inputs(B, L, ED, seed=ED + L + gate)
    t = _prep(d, dtype, use_z=gate)
    got, n = launches(lambda: _run(t))
    assert_scan_path("generic-split" if split else "generic", B, L, ED, n)
    compare(got, _oracle(t), TOL[dtype])


def test_inner_node_generic_width_bf16():
    """MambaBlock(d_model=40) under bf16 autocast: the one-node inner path on the generic kernels (ED = 80, B/C slices at
    offset dt_rank = 3) against the op-by-op composition of the same kernels."""
    from gfe_mamba_b200 import MambaBlock, MambaConfig
    torch.manual_seed(5)
    blk = MambaBlock(MambaConfig(d_model=40, n_layers=1)).cuda()
    with torch.no_grad():
        blk.A_log.add_(0.1 * torch.randn_like(blk.A_log))
        blk.D.add_(0.1 * torch.randn_like(blk.D))
    x0 = torch.randn(3, 150, 40, device="cuda")
    dy = torch.randn(3, 150, 40, device="cuda")
    assert blk._inner_fusable(torch.empty(1, 1, 2 * blk.config.d_inner, device="cuda"))

    def run(fused):
        blk.zero_grad(set_to_none=True)
        if not fused:
            blk._inner_fusable = lambda xz: False
        elif "_inner_fusable" in blk.__dict__:
            del blk.__dict__["_inner_fusable"]
        x = x0.clone().requires_grad_()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = blk(x)
        y.float().backward(dy)
        return [y.detach().float(), x.grad.float()] + [p.grad.float().clone() for p in blk.parameters()]

    (a, n), b = launches(lambda: run(True)), run(False)
    assert_scan_path("generic", 3, 150, 80, {k: v for k, v in n.items() if k.startswith("selscan")})
    names = ["y", "dx"] + [nm for nm, _ in blk.named_parameters()]
    for nm, ga, gb in zip(names, a, b):
        err = float((ga - gb).abs().max() / gb.abs().max().clamp_min(1e-30))
        assert err < 3e-2, (nm, err)


# ------------------------------------------------------------------------------------------------- final state
PATH_SHAPES = {"generic": (2, 203, 40), "generic-split": (1, 2100, 40), "waiting": (20, 267, 512), "independent": (1, 2100, 64)}
LAST_TOL = {torch.float32: 1e-4, torch.bfloat16: 1e-3, torch.float16: 1e-3}   # fp32 state from the rounded inputs


@pytest.mark.parametrize("grad", [True, False], ids=["grad", "nograd"])
@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_last_state(path, dt, grad):
    """return_last_state=True: the state after the last token, (B, ED, N) fp32, written by selscan.cu (generic) and
    selscan_v4_fwd.cu (both schedules), with and without the checkpoint stream; outputs and gradients unchanged."""
    dtype = DTYPES[dt]
    B, L, ED = PATH_SHAPES[path]
    d = make_scan_inputs(B, L, ED, seed=L + ED + grad)
    t = _prep(d, dtype)
    got, n = launches(lambda: _run(t, grad=grad, last=True))
    assert_scan_path(path, B, L, ED, n, grad=grad)
    want = _oracle(t, grad=grad, last=True)
    assert got["last"].shape == (B, ED, N) and got["last"].dtype == torch.float32
    assert relerr(got["last"], want["last"]) < LAST_TOL[dtype]
    compare(got, want, TOL[dtype], keys=("out", "du", "ddelta", "dz", "dB", "dC", "dA_log", "dD", "ddt_bias") if grad else ("out",))


def _decode_from(t, hl, L, T):
    """ssm_step over tokens L..L+T-1 of t's inputs, starting from state hl."""
    from gfe_mamba_b200 import ops
    outs, h = [], hl
    with torch.no_grad():
        for s in range(L, L + T):
            y, h = ops.ssm_step(t["u"][:, s], t["draw"][:, s], t["A_log"], t["Bm"][:, s], t["Cm"][:, s], t["D"], h,
                                z=None if t["z"] is None else t["z"][:, s], dt_bias=t["bias"], delta_softplus=t["softplus"])
            outs.append(y)
    return torch.stack(outs, 1), h


def _slice_inputs(d, L):
    return {k: (v[:, :L] if k in ("u", "draw", "z", "Bm", "Cm", "dout") else v) for k, v in d.items()}


@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_prefill_then_decode(path):
    """Scan L tokens with return_last_state, continue T tokens with ssm_step from that state: the same outputs and final
    state as one scan over L + T tokens (the state layout of the scans is the one the decode kernel consumes)."""
    B, L, ED = PATH_SHAPES[path]
    T = 6
    d = make_scan_inputs(B, L + T, ED, seed=3 * L + ED)
    t = _prep(d, torch.float32)
    pre, n = launches(lambda: _run(_prep(_slice_inputs(d, L), torch.float32), grad=False, last=True))
    assert_scan_path(path, B, L, ED, n, grad=False)
    hl = pre["last"]
    full = _oracle(t, grad=False, last=True)
    ys, h = _decode_from(t, hl, L, T)
    assert relerr(ys, full["out"][:, L:]) < 1e-4
    assert relerr(h, full["last"]) < 1e-4
    whole = _run(t, grad=False, last=True)
    assert relerr(ys, whole["out"][:, L:]) < 1e-4 and relerr(h, whole["last"]) < 1e-4


# ------------------------------------------------------------------------------------------------- decode kernels
def _silu64(v):
    return v / (1.0 + np.exp(-v))


def _ssm_step_ref(u, delta, A_log, Bm, Cm, D, h, z, bias, softplus):
    """orc.ssm_step (the recurrence, fp64) behind softplus(delta + dt_bias) and in front of the gate, in fp64."""
    dl = delta.astype(np.float64) + (0.0 if bias is None else bias.astype(np.float64))
    if softplus:
        dl = np.where(dl > 20.0, dl, np.log1p(np.exp(np.minimum(dl, 20.0))))
    y, h_new = orc.ssm_step(u, dl.astype(np.float32), A_log, Bm, Cm, D, h)
    y = y.astype(np.float64)
    return (y if z is None else y * _silu64(z.astype(np.float64))), h_new


DECODE_FLAGS = [(True, True, True), (False, True, True), (True, False, True), (True, True, False), (False, False, False)]


@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("gate,use_bias,softplus", DECODE_FLAGS,
                         ids=[f"{'z' if g else 'noz'}-{'bias' if b else 'nobias'}-{'sp' if s else 'nosp'}" for g, b, s in DECODE_FLAGS])
@pytest.mark.parametrize("dt", list(DTYPES))
def test_decode_kernels(dt, gate, use_bias, softplus, K):
    """conv1d_step_kernel<T, K> and ssm_step_kernel<T> over a few tokens: xin / z as the strided halves of in_proj's output,
    B / C as slices of x_proj's output, ED = 200 (a partial 128-channel block), against numpy fp64 / orc.ssm_step; the
    rolled conv cache is exact, and neither op modifies its inputs."""
    from gfe_mamba_b200 import ops
    dtype = DTYPES[dt]
    Bsz, ED, T, R = 3, 200, 5, R_UNALIGNED
    r = np.random.default_rng(100 * K + 10 * gate + 2 * use_bias + softplus)
    dev = lambda a, dtp=dtype: torch.from_numpy(np.ascontiguousarray(a, np.float32)).to("cuda", dtp)
    xz = dev(r.standard_normal((T, Bsz, 2 * ED)))
    draw = r.standard_normal((T, Bsz, ED)) * 0.5
    p = make_scan_inputs(1, 1, ED, seed=K)
    if not softplus:
        draw, p = np.abs(draw) * 0.2 + 1e-3, _positive_delta(p)
    delta = dev(draw)
    dbc = dev(r.standard_normal((T, Bsz, R + 2 * N)))
    conv_w = dev(r.standard_normal((ED, 1, K)) * 0.5, torch.float32)
    conv_b = dev(r.standard_normal(ED) * 0.1, torch.float32) if use_bias else None
    A_log, D = dev(p["A_log"], torch.float32), dev(p["D"], torch.float32)
    bias = dev(p["bias"], torch.float32) if use_bias else None
    cache = dev(r.standard_normal((Bsz, ED, K - 1)))
    h = dev(r.standard_normal((Bsz, ED, N)) * 0.5, torch.float32)
    h_ref = h.cpu().numpy()
    w64 = conv_w.cpu().numpy().astype(np.float64)[:, 0, :]
    b64 = 0.0 if conv_b is None else conv_b.cpu().numpy().astype(np.float64)
    for s in range(T):
        xin, z = xz[s, :, :ED], xz[s, :, ED:]
        Bm, Cm = dbc[s, :, R:R + N], dbc[s, :, R + N:]
        before = [v.clone() for v in (xz, cache, h, delta, dbc)]
        with torch.no_grad():
            (u, cache_new), n = launches(lambda: ops.conv1d_step(xin, cache, conv_w, conv_b))
            y, h_new = ops.ssm_step(u, delta[s], A_log, Bm, Cm, D, h, z=z if gate else None, dt_bias=bias, delta_softplus=softplus)
        assert n == {"conv1d_step": 1}
        for v, v0 in zip((xz, cache, h, delta, dbc), before):
            assert torch.equal(v, v0), "a decode op modified its input"
        win = np.concatenate([_np(cache), _np(xin)[:, :, None]], -1).astype(np.float64)   # (B, ED, K)
        assert relerr(u, _silu64((win * w64).sum(-1) + b64)) < TOL[dtype], s
        assert np.array_equal(_np(cache_new), win[:, :, 1:]), "conv cache not rolled by one token"
        y_ref, h_ref = _ssm_step_ref(_np(u), _np(delta[s]), p["A_log"], _np(Bm), _np(Cm), p["D"], h_ref,
                                     _np(z) if gate else None, p["bias"] if use_bias else None, softplus)
        assert y.dtype == dtype and relerr(y, y_ref) < TOL[dtype], s
        assert relerr(h_new, h_ref) < 1e-4, s
        cache, h = cache_new, h_new


@pytest.mark.parametrize("dt", list(DTYPES))
def test_ssm_step_without_state_is_zero_state(dt):
    from gfe_mamba_b200 import ops
    dtype = DTYPES[dt]
    Bsz, ED = 2, 72
    d = make_scan_inputs(Bsz, 1, ED, seed=9)
    a = {k: torch.from_numpy(d[k][:, 0]).to("cuda", dtype) for k in ("u", "draw", "z", "Bm", "Cm")}
    A_log, D, bias = cuda(d["A_log"]), cuda(d["D"]), cuda(d["bias"])
    with torch.no_grad():
        y0, h0 = ops.ssm_step(a["u"], a["draw"], A_log, a["Bm"], a["Cm"], D, None, z=a["z"], dt_bias=bias)
        y1, h1 = ops.ssm_step(a["u"], a["draw"], A_log, a["Bm"], a["Cm"], D, torch.zeros(Bsz, ED, N, device="cuda"), z=a["z"],
                              dt_bias=bias)
    assert torch.equal(y0, y1) and torch.equal(h0, h1)
    y_ref, h_ref = _ssm_step_ref(_np(a["u"]), _np(a["draw"]), d["A_log"], _np(a["Bm"]), _np(a["Cm"]), d["D"], None, _np(a["z"]),
                                 d["bias"], True)
    assert relerr(y0, y_ref) < TOL[dtype] and relerr(h0, h_ref) < 1e-4


# ------------------------------------------------------------------------------------------------- conv gaps
def conv_vec(dtype, ED, *views):
    """conv_vec (conv1d.cu): 8-byte accesses (packed kernels) when ED and every base / batch / row stride allow them."""
    s = torch.empty((), dtype=dtype).element_size()
    V = 8 // s
    if ED % V:
        return 1
    return V if all(t.data_ptr() % 8 == 0 and (t.stride(0) * s) % 8 == 0 and (t.stride(1) * s) % 8 == 0 for t in views) else 1


def _conv_case(dtype, B, L, ED, K, off, seed):
    """xin = xz[..., off:off + ED] of a (B, L, 2 ED + off) tensor; forward + backward against the oracle."""
    from gfe_mamba_b200 import causal_conv1d_silu
    r = np.random.default_rng(seed)
    xz = torch.from_numpy(r.standard_normal((B, L, 2 * ED + off)).astype(np.float32)).to("cuda", dtype).requires_grad_()
    w = cuda((r.standard_normal((ED, 1, K)) * 0.5).astype(np.float32), grad=True)
    b = cuda((r.standard_normal(ED) * 0.1).astype(np.float32), grad=True)
    du = torch.from_numpy(r.standard_normal((B, L, ED)).astype(np.float32)).to("cuda", dtype)
    xin = xz[..., off:off + ED]

    def run():
        u = causal_conv1d_silu(xin, w, b)
        u.backward(du)
        return u
    u, n = launches(run)
    assert n == {"conv1d_silu_fwd": 1, "conv1d_silu_bwd": 1, "conv1d_bwd_finalize": 1}
    x64 = _np(xin)
    assert relerr(u, orc.conv1d_silu_fwd(x64, _np(w), _np(b))) < TOL[dtype]
    dxin, dw, db = orc.conv1d_silu_bwd(x64, _np(w), _np(b), _np(du))
    assert relerr(xz.grad[..., off:off + ED], dxin) < TOL[dtype]
    rest = torch.cat([xz.grad[..., :off], xz.grad[..., off + ED:]], -1)
    assert float(rest.abs().max()) == 0.0
    tol_w = 1e-4 if dtype == torch.float32 else 1e-3   # fp32 accumulation of exactly representable inputs
    assert relerr(w.grad, dw) < tol_w and relerr(b.grad, db) < tol_w
    return xin


@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("layout", ["ed42", "misaligned"])
@pytest.mark.parametrize("dt", ["bf16", "f16"])
def test_conv_unpacked_16bit(dt, layout, K):
    """conv1d_silu_{fwd,bwd}_kernel<bf16 | f16, K, 1>: ED % 4 != 0, or a view whose base is 2 bytes past an 8-byte boundary."""
    dtype = DTYPES[dt]
    ED, off = (42, 0) if layout == "ed42" else (64, 1)
    xin = _conv_case(dtype, 2, 300, ED, K, off, seed=K + ED)
    assert conv_vec(dtype, ED, xin) == 1   # the layout really rules out the packed kernels


@pytest.mark.parametrize("dt", ["f32", "bf16"])
def test_conv_long_many_tiles(dt):
    """L = 2000 over 3 rows: 16 tiles of 128 steps per row, so conv1d_bwd_finalize adds 48 partial rows per channel."""
    dtype = DTYPES[dt]
    B, L, ED, K = 3, 2000, 128, 4
    xin = _conv_case(dtype, B, L, ED, K, 0, seed=2000)
    assert conv_vec(dtype, ED, xin) == 8 // xin.element_size()   # the packed kernels


# ------------------------------------------------------------------------------------------------- small step sizes
def per_channel_err(got, want, axis):
    """For each channel: max |got - want| over the channel's values / max |want| of the channel."""
    g = np.moveaxis(np.asarray(_np(got) if torch.is_tensor(got) else got, np.float64), axis, 0)
    w = np.moveaxis(np.asarray(want, np.float64), axis, 0)
    assert g.shape == w.shape and np.isfinite(g).all()
    g, w = g.reshape(g.shape[0], -1), w.reshape(w.shape[0], -1)
    return np.abs(g - w).max(1) / np.maximum(np.abs(w).max(1), 1e-30)


@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_small_step_sizes_per_channel(path):
    """dt_bias spread over [-16, -4] across channels (trained long-memory channels): delta = softplus(x) down to ~1e-7.
    Per-channel errors of last_state, dA_log and the decode continuation, fp32."""
    B, L, ED = PATH_SHAPES[path]
    T = 6
    d = make_scan_inputs(B, L + T, ED, seed=17 + ED)
    d["bias"] = np.linspace(-16.0, -4.0, ED).astype(np.float32)
    t_pre = _prep(_slice_inputs(d, L), torch.float32)
    got, n = launches(lambda: _run(t_pre, grad=True, last=True))
    assert_scan_path(path, B, L, ED, n)
    want = _oracle(t_pre, grad=True, last=True)
    t = _prep(d, torch.float32)
    ys, h = _decode_from(t, got["last"], L, T)
    full = _oracle(t, grad=False, last=True)
    errs = dict(last_state=per_channel_err(got["last"], want["last"], 1), dA_log=per_channel_err(got["dA_log"], want["dA_log"], 0),
                decode_out=per_channel_err(ys, full["out"][:, L:], 2), decode_h=per_channel_err(h, full["last"], 1))
    worst = {k: (float(e.max()), float(d["bias"][int(e.argmax())])) for k, e in errs.items()}
    print(path, "per-channel max error (value, dt_bias of that channel):", worst)
    assert all(v < 1e-3 for v, _ in worst.values()), worst
