"""Training from a carried state: the backward of the from-state scan and conv kernels (ops.selective_scan_state,
ops.causal_conv1d_silu_state) and MambaBlock / Mamba.prefill under grad.

A sequence cut into chunks, each continued from the non-detached state the previous one left, must give the gradients of one
pass over the whole sequence.  Every scan case first proves which kernels each chunk reached (launch registry), so each
backward path -- generic kernels with and without the L split, chained kernels with waiting and with independent segments
(the reverse combine seeded with d h_last) -- is known to take dlast and return dh0.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_kernel_matrix import DTYPES, PATH_SHAPES, _prep, assert_scan_path, launches, per_channel_err, split_along_l
from test_gpu_parity import TOL, make_scan_inputs, relerr

pytestmark = pytest.mark.gpu

KEYS = ("u", "draw", "z", "A_log", "D", "bias")


def _sl(t, k, s0, s1):
    return None if t[k] is None else t[k][:, s0:s1]


def _state_call(t, s0, s1, h0):
    from gfe_mamba_b200 import ops
    return ops.selective_scan_state(_sl(t, "u", s0, s1), _sl(t, "draw", s0, s1), t["A_log"], _sl(t, "Bm", s0, s1),
                                    _sl(t, "Cm", s0, s1), t["D"], h0, z=_sl(t, "z", s0, s1), dt_bias=t["bias"],
                                    delta_softplus=t["softplus"])


def _grads(t, extra=()):
    """Gradients of the leaves; a leaf the loss does not reach (z and D of the fp64 recurrence under a loss on h_last
    alone) counts as zeros, which is what the kernels return for it."""
    grad = lambda x: torch.zeros_like(x) if x.grad is None else x.grad.clone()
    g = {k: (None if t[k] is None else grad(t[k])) for k in KEYS + ("Bm", "Cm")}
    for name, x in extra:
        g[name] = grad(x)
    return g


def _zero(t, extra=()):
    for k in KEYS + ("Bm", "Cm"):
        if t[k] is not None:
            t[k].grad = None
    for x in extra:
        x.grad = None


def _bwd_launches(path, B, L, ED, n, chunks):
    split = split_along_l(B, L, ED)
    want = dict(selscan_bwd=chunks, selscan_bwd_finalize_bc=chunks, selscan_bwd_finalize_par=chunks)
    if split:
        want["selscan_bwd_summary"] = chunks
    assert n == want, f"{path}: backward launched {n}, expected {want}"


def _ref64(t, h0, s0, s1):
    """fp64 torch recurrence with autograd over tokens [s0, s1) from h0, on the rounded leaves."""
    f = lambda k: None if t[k] is None else t[k][:, s0:s1].double()
    u, draw, z, Bm, Cm = f("u"), f("draw"), f("z"), f("Bm"), f("Cm")
    A = -torch.exp(t["A_log"].double())
    x = draw + (0 if t["bias"] is None else t["bias"].double())
    delta = F.softplus(x) if t["softplus"] else x
    h = torch.zeros(u.shape[0], u.shape[2], A.shape[1], dtype=torch.float64, device=u.device) if h0 is None else h0.double()
    ys = []
    for s in range(u.shape[1]):
        h = torch.exp(delta[:, s, :, None] * A) * h + (delta[:, s] * u[:, s])[:, :, None] * Bm[:, s, None, :]
        ys.append((h * Cm[:, s, None, :]).sum(-1) + t["D"].double() * u[:, s])
    y = torch.stack(ys, 1)
    return (y if z is None else y * F.silu(z)), h


SCAN_CASES = [pytest.param(path, dt, gate, 16, id=f"{path}-{dt}-{'z' if gate else 'noz'}-N16")
              for path in PATH_SHAPES for dt in DTYPES for gate in (True, False)]
SCAN_CASES += [pytest.param(path, dt, True, n, id=f"{path}-{dt}-z-N{n}")
               for path in ("generic", "generic-split") for dt in DTYPES for n in (32, 64)]


@pytest.mark.parametrize("path,dt,gate,N", SCAN_CASES)
def test_chunked_equals_whole(path, dt, gate, N):
    """Two chunks of the path's length, the second from the first's non-detached h_last.  A loss on both outputs gives the
    gradients of one selective_scan_fn pass; an added term on the final h_last gives those of one selective_scan_state pass
    and of the fp64 recurrence."""
    from gfe_mamba_b200 import selective_scan_fn
    dtype = DTYPES[dt]
    B, L, ED = PATH_SHAPES[path]
    d = make_scan_inputs(B, 2 * L, ED, N=N, seed=3 * L + ED + N + gate)
    t = _prep(d, dtype, use_z=gate)
    W = torch.randn(B, ED, N, device="cuda", generator=torch.Generator("cuda").manual_seed(ED + N))
    dout = t["dout"]

    def chunked(with_last):
        (y1, h1), n1 = launches(lambda: _state_call(t, 0, L, None))
        assert_scan_path(path, B, L, ED, n1, grad=False)
        (y2, h2), n2 = launches(lambda: _state_call(t, L, 2 * L, h1))
        assert_scan_path(path, B, L, ED, n2, grad=False)
        loss = (y1.float() * dout[:, :L].float()).sum() + (y2.float() * dout[:, L:].float()).sum()
        if with_last:
            loss = loss + (h2 * W).sum()
        _, nb = launches(loss.backward)
        _bwd_launches(path, B, L, ED, nb, 2)
        return _grads(t)

    tol = TOL[dtype]
    got = chunked(False)
    _zero(t)
    y = selective_scan_fn(t["u"], t["draw"], t["A_log"], t["Bm"], t["Cm"], t["D"], z=t["z"], dt_bias=t["bias"],
                          delta_softplus=t["softplus"])
    y.backward(dout)
    want = _grads(t)
    for k in want:
        if want[k] is not None:
            assert relerr(got[k], want[k]) < tol, (k, relerr(got[k], want[k]))

    _zero(t)
    got = chunked(True)
    _zero(t)
    y, h = _state_call(t, 0, 2 * L, None)
    ((y.float() * dout.float()).sum() + (h * W).sum()).backward()
    want = _grads(t)
    _zero(t)
    y64, h64 = _ref64(t, None, 0, 2 * L)
    ((y64 * dout.double()).sum() + (h64 * W.double()).sum()).backward()
    ref = _grads(t)
    for k in want:
        if want[k] is not None:
            assert relerr(got[k], want[k]) < tol, (k, "vs one pass", relerr(got[k], want[k]))
            assert relerr(got[k], ref[k]) < tol, (k, "vs fp64", relerr(got[k], ref[k]))


@pytest.mark.parametrize("only_last", [False, True], ids=["out-and-last", "last-only"])
@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_state_gradients_against_fp64(path, only_last):
    """dh0 for a caller-given h0 and dlast for a loss on h_last (alone: the output is unused and dout is zeros), fp32."""
    B, L, ED = PATH_SHAPES[path]
    t = _prep(make_scan_inputs(B, L, ED, seed=11 + ED + only_last), torch.float32)
    g = torch.Generator("cuda").manual_seed(L)
    h0 = torch.randn(B, ED, 16, device="cuda", generator=g).requires_grad_()
    W = torch.randn(B, ED, 16, device="cuda", generator=g)

    def loss(y, h):
        l = (h * W).sum()
        return l if only_last else l + (y * t["dout"]).sum()
    (y, h), n = launches(lambda: _state_call(t, 0, L, h0))
    assert_scan_path(path, B, L, ED, n, grad=False)
    loss(y, h).backward()
    got = _grads(t, [("h0", h0)])
    _zero(t, [h0])
    loss(*_ref64(t, h0, 0, L)).backward()
    want = _grads(t, [("h0", h0)])
    for k in want:
        if want[k] is not None:
            assert relerr(got[k], want[k]) < 1e-4, (k, relerr(got[k], want[k]))


@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_state_gradients_small_step_sizes_per_channel(path):
    """dt_bias over [-16, -4] across channels: per-channel errors of dh0 and dA_log stay small on the long-memory channels."""
    B, L, ED = PATH_SHAPES[path]
    d = make_scan_inputs(B, L, ED, seed=23 + ED)
    d["bias"] = np.linspace(-16.0, -4.0, ED).astype(np.float32)
    t = _prep(d, torch.float32)
    g = torch.Generator("cuda").manual_seed(ED)
    h0 = torch.randn(B, ED, 16, device="cuda", generator=g).requires_grad_()
    W = torch.randn(B, ED, 16, device="cuda", generator=g)
    y, h = _state_call(t, 0, L, h0)
    ((y * t["dout"]).sum() + (h * W).sum()).backward()
    got = _grads(t, [("h0", h0)])
    _zero(t, [h0])
    y64, h64 = _ref64(t, h0, 0, L)
    ((y64 * t["dout"].double()).sum() + (h64 * W.double()).sum()).backward()
    want = _grads(t, [("h0", h0)])
    errs = dict(dh0=per_channel_err(got["h0"], want["h0"].cpu().numpy(), 1),
                dA_log=per_channel_err(got["A_log"], want["A_log"].cpu().numpy(), 0))
    worst = {k: float(e.max()) for k, e in errs.items()}
    print(path, "per-channel max error:", worst)
    assert all(v < 1e-3 for v in worst.values()), worst


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_null_state_is_the_old_path(path, dt):
    """h0 = None and an unused h_last: the kernels run with dlast = dh0 = NULL, bitwise selective_scan_fn's gradients."""
    from gfe_mamba_b200 import selective_scan_fn
    dtype = DTYPES[dt]
    B, L, ED = PATH_SHAPES[path]
    t = _prep(make_scan_inputs(B, L, ED, seed=29 + L), dtype)
    y, _ = _state_call(t, 0, L, None)
    y.backward(t["dout"])
    got = _grads(t)
    _zero(t)
    y0 = selective_scan_fn(t["u"], t["draw"], t["A_log"], t["Bm"], t["Cm"], t["D"], z=t["z"], dt_bias=t["bias"])
    y0.backward(t["dout"])
    want = _grads(t)
    assert torch.equal(y, y0)
    for k in want:
        assert torch.equal(got[k], want[k]), k


# ------------------------------------------------------------------------------------------------------- conv
def _conv_inputs(dtype, B, L, ED, K, off, seed):
    r = np.random.default_rng(seed)
    mk = lambda a: torch.from_numpy(a.astype(np.float32))
    xz = mk(r.standard_normal((B, L, 2 * ED + off))).to("cuda", dtype).requires_grad_()
    inp = mk(r.standard_normal((B, ED, K - 1))).to("cuda", dtype).requires_grad_()
    w = mk(r.standard_normal((ED, 1, K)) * 0.5).cuda().requires_grad_()
    b = mk(r.standard_normal(ED) * 0.1).cuda().requires_grad_()
    du = mk(r.standard_normal((B, L, ED))).to("cuda", dtype)
    dn = mk(r.standard_normal((B, ED, K - 1))).to("cuda", dtype)
    return xz, inp, w, b, du, dn


@pytest.mark.parametrize("L", [300, 2, 1])
@pytest.mark.parametrize("layout", ["packed", "unpacked"])
@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("dt", list(DTYPES))
def test_conv_from_window_against_fp64(dt, K, layout, L):
    """u, dxin, dw, dbias and dinputs against fp64 torch over cat(inputs, xin); a loss on new_inputs too, whose gradient
    reaches both the window and xin.  packed: 8-byte aligned views; unpacked: a view 1 element into each row."""
    from gfe_mamba_b200 import ops
    from test_gpu_kernel_matrix import conv_vec
    dtype = DTYPES[dt]
    B, ED = 2, 64
    off = 0 if layout == "packed" else 1
    xz, inp, w, b, du, dn = _conv_inputs(dtype, B, L, ED, K, off, seed=K * 100 + L + off)
    xin = xz[..., off:off + ED]
    assert (conv_vec(dtype, ED, xin) > 1) == (layout == "packed")
    (u, new), n = launches(lambda: ops.causal_conv1d_silu_state(xin, inp, w, b))
    assert n == {"conv1d_silu_fwd": 1}
    ((u.float() * du.float()).sum() + (new.float() * dn.float()).sum()).backward()
    got = dict(x=xz.grad[..., off:off + ED].clone(), inp=inp.grad.clone(), w=w.grad.clone(), b=b.grad.clone())
    assert float(torch.cat([xz.grad[..., :off], xz.grad[..., off + ED:]], -1).abs().max()) == 0.0
    for x in (xz, inp, w, b):
        x.grad = None
    full = torch.cat([inp.double(), xin.double().transpose(1, 2)], 2)                      # (B, ED, K-1+L)
    u64 = F.silu(F.conv1d(full, w.double(), b.double(), groups=ED)).transpose(1, 2)
    new64 = full[:, :, -(K - 1):]
    assert relerr(u, u64) < TOL[dtype] and torch.equal(new, new64.to(dtype))
    ((u64 * du.double()).sum() + (new64 * dn.double()).sum()).backward()
    want = dict(x=xz.grad[..., off:off + ED], inp=inp.grad, w=w.grad, b=b.grad)
    tol_w = 1e-4 if dtype == torch.float32 else 1e-3
    for k in want:
        assert relerr(got[k], want[k]) < (tol_w if k in ("w", "b") else TOL[dtype]), (k, relerr(got[k], want[k]))


@pytest.mark.parametrize("dt", list(DTYPES))
def test_conv_null_window_is_the_old_path(dt):
    """inputs = None: bitwise causal_conv1d_silu, forward and every gradient."""
    from gfe_mamba_b200 import causal_conv1d_silu, ops
    dtype = DTYPES[dt]
    xz, _, w, b, du, _ = _conv_inputs(dtype, 2, 300, 64, 4, 0, seed=7)
    xin = xz[..., :64]
    u, _ = ops.causal_conv1d_silu_state(xin, None, w, b)
    u.backward(du)
    got = [xz.grad.clone(), w.grad.clone(), b.grad.clone()]
    for x in (xz, w, b):
        x.grad = None
    u0 = causal_conv1d_silu(xin, w, b)
    u0.backward(du)
    assert torch.equal(u, u0)
    for g, x in zip(got, (xz, w, b)):
        assert torch.equal(g, x.grad)


# ------------------------------------------------------------------------------------------------------- model
def _model(d_model=64, n_layers=2, seed=0, **kw):
    from gfe_mamba_b200 import Mamba, MambaConfig
    torch.manual_seed(seed)
    return Mamba(MambaConfig(d_model=d_model, n_layers=n_layers, **kw)).cuda()


def test_prefill_under_grad_reaches_the_fused_kernels():
    """No decode-step launches; one conv and one scan backward per layer."""
    m = _model()
    x = torch.randn(2, 40, 64, device="cuda", requires_grad=True)
    (y, caches), n = launches(lambda: m.prefill(x))
    assert "ssm_step" not in n and "conv1d_step" not in n and n["selscan_fwd"] == 2 and n["conv1d_silu_fwd"] == 2
    _, nb = launches(lambda: (y.square().mean() + sum(h.square().sum() for h, _ in caches)).backward())
    assert nb["selscan_bwd"] == 2 and nb["conv1d_silu_bwd"] == 2 and "ssm_step" not in nb


@pytest.mark.parametrize("autocast", [False, True], ids=["f32", "bf16-autocast"])
def test_chunked_prefill_equals_forward(autocast):
    """Three chunks with non-detached caches: the parameter gradients and x.grad of forward over the concatenation."""
    m = _model(seed=1)
    x = torch.randn(2, 300, 64, device="cuda", requires_grad=True)
    tol = 3e-2 if autocast else 1e-4
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        caches, ys = None, []
        for s0, s1 in ((0, 100), (100, 217), (217, 300)):
            y, caches = m.prefill(x[:, s0:s1], caches)
            ys.append(y)
        loss = torch.cat(ys, 1).float().square().mean()
    loss.backward()
    got = [p.grad.clone() for p in m.parameters()] + [x.grad.clone()]
    m.zero_grad()
    x.grad = None
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
        want_y = m(x)
        want = want_y.float().square().mean()
    want.backward()
    assert relerr(torch.cat(ys, 1), want_y) < tol
    for g, p in zip(got, list(m.parameters()) + [x]):
        assert relerr(g, p.grad) < tol


def test_gradients_reach_caller_caches():
    """A MambaBlock prefill under grad from caller-given (h, inputs): outputs, caches and every gradient (caches included)
    equal those of the step loop, the reference's differentiable composition."""
    m = _model(seed=2)
    blk = m.layers[0].mixer
    cfg = blk.config
    g = torch.Generator("cuda").manual_seed(0)
    x = torch.randn(2, 24, 64, device="cuda", generator=g, requires_grad=True)
    h = torch.randn(2, cfg.d_inner, cfg.d_state, device="cuda", generator=g).mul(0.5).requires_grad_()
    inp = torch.randn(2, cfg.d_inner, cfg.d_conv - 1, device="cuda", generator=g).requires_grad_()
    leaves = [x, h, inp] + list(blk.parameters())

    def grads_of(y, c):
        (y.square().mean() + c[0].square().mean() + c[1].square().mean()).backward()
        out = [None if t.grad is None else t.grad.clone() for t in leaves]
        for t in leaves:
            t.grad = None
        return out
    (y, c), n = launches(lambda: blk.prefill(x, (h, inp)))
    assert "ssm_step" not in n and n["selscan_fwd"] == 1
    got = grads_of(y, c)
    cache, ys = (h, inp), []
    for s in range(x.shape[1]):
        yt, cache = blk.step(x[:, s], cache)
        ys.append(yt)
    y0 = torch.stack(ys, 1)
    assert relerr(y, y0) < 1e-4 and relerr(c[0], cache[0]) < 1e-4 and relerr(c[1], cache[1]) < 1e-5
    want = grads_of(y0, cache)
    assert got[1] is not None and got[2] is not None
    for a, b in zip(got, want):
        assert relerr(a, b) < 1e-4


def test_truncated_bptt_peak_memory():
    """cfg 4's d_model, detached caches between 4096-token chunks: the peak of one chunk's forward + backward is that of
    forward + backward on one chunk, plus the caches and 2 % (measured on a B200: 363 against 357 MiB).  With inner
    layernorms, so that forward runs the same op-by-op structure (its one-node inner path writes some gradients in place,
    which the from-state path does not)."""
    m = _model(d_model=512, n_layers=2, seed=3, inner_layernorms=True)
    x = torch.randn(1, 2 * 4096, 512, device="cuda")

    def peak(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    _, caches = m.prefill(x[:, :4096])
    caches = [(h.detach(), i.detach()) for h, i in caches]

    def chunk():
        y, c = m.prefill(x[:, 4096:], caches)
        y.square().mean().backward()
    ref = peak(lambda: m(x[:, 4096:]).square().mean().backward())
    got = peak(chunk)
    cache_bytes = sum(h.numel() * 4 + i.numel() * i.element_size() for h, i in caches)
    print("peak MiB: prefill chunk", got / 2**20, "forward chunk", ref / 2**20)
    assert got <= 1.02 * ref + 2 * cache_bytes, (got, ref)
