"""Prefill from a decode cache: the scan and conv forward kernels started from a carried state (ops.ssm_prefill,
ops.conv1d_prefill) and Mamba.prefill.

The truth for a chunk that starts from a state is the fp64 oracle over the whole concatenated sequence: a sequence cut into
chunks, each continued from the state the previous one left, must give the outputs and the final state of one pass.  Every
scan case first proves which forward kernels it reached (launch registry), so each path -- generic kernels with and without
the L split, chained kernels with waiting and with independent segments -- is known to start from the state.
"""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from test_gpu_kernel_matrix import (DTYPES, LAST_TOL, PATH_SHAPES, R_UNALIGNED, _np, _oracle, _prep, assert_scan_path,
                                    conv_vec, launches, per_channel_err)
from test_gpu_parity import TOL, make_scan_inputs, relerr

pytestmark = pytest.mark.gpu


def _sl(t, k, s0, s1):
    return None if t[k] is None else t[k][:, s0:s1]


def _prefill(t, s0, s1, h):
    from gfe_mamba_b200 import ops
    with torch.no_grad():
        return ops.ssm_prefill(_sl(t, "u", s0, s1), _sl(t, "draw", s0, s1), t["A_log"], _sl(t, "Bm", s0, s1),
                               _sl(t, "Cm", s0, s1), t["D"], h, z=_sl(t, "z", s0, s1), dt_bias=t["bias"],
                               delta_softplus=t["softplus"])


def _two_chunks(path, t, B, L1, L2, ED):
    """tokens [0, L1) from h = None, then [L1, L1 + L2) from the state the first call left; asserts the kernels of both
    calls and that the state passed in is not modified."""
    (y1, h1), n1 = launches(lambda: _prefill(t, 0, L1, None))
    assert_scan_path(path, B, L1, ED, n1, grad=False)
    h1_before = h1.clone()
    (y2, h2), n2 = launches(lambda: _prefill(t, L1, L1 + L2, h1))
    assert_scan_path(path, B, L2, ED, n2, grad=False)
    assert torch.equal(h1, h1_before), "ssm_prefill modified the state it started from"
    return y1, h1, y2, h2


SCAN_CASES = [pytest.param(path, dt, gate, 16, id=f"{path}-{dt}-{'z' if gate else 'noz'}-N16")
              for path in PATH_SHAPES for dt in DTYPES for gate in (True, False)]
SCAN_CASES += [pytest.param(path, dt, True, n, id=f"{path}-{dt}-z-N{n}")
               for path in ("generic", "generic-split") for dt in DTYPES for n in (32, 64)]


@pytest.mark.parametrize("path,dt,gate,N", SCAN_CASES)
def test_ssm_prefill_every_path(path, dt, gate, N):
    """Two chunks of the path's length each: both hit the path (chained with two waiting segments, independent segments
    seeded through the combine pass, the generic L split folding h0 through the summaries)."""
    dtype = DTYPES[dt]
    B, L, ED = PATH_SHAPES[path]
    d = make_scan_inputs(B, 2 * L, ED, N=N, seed=L + ED + N + gate)
    t = _prep(d, dtype, use_z=gate)
    y1, _, y2, h2 = _two_chunks(path, t, B, L, L, ED)
    want = _oracle(t, grad=False, last=True)
    assert y1.dtype == dtype and h2.dtype == torch.float32 and h2.shape == (B, ED, N)
    assert relerr(y1, want["out"][:, :L]) < TOL[dtype]
    assert relerr(y2, want["out"][:, L:]) < TOL[dtype]
    assert relerr(h2, want["last"]) < LAST_TOL[dtype]


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_zero_start_is_the_forward(path, dt):
    """h = None runs exactly the kernels of selective_scan_fn: bitwise equal outputs and final state."""
    from gfe_mamba_b200 import selective_scan_fn
    dtype = DTYPES[dt]
    B, L, ED = PATH_SHAPES[path]
    t = _prep(make_scan_inputs(B, L, ED, seed=5 + L), dtype)
    y, h = _prefill(t, 0, L, None)
    with torch.no_grad():
        y0, h0 = selective_scan_fn(t["u"], t["draw"], t["A_log"], t["Bm"], t["Cm"], t["D"], z=t["z"], dt_bias=t["bias"],
                                   return_last_state=True)
    assert torch.equal(y, y0) and torch.equal(h, h0)


@pytest.mark.parametrize("T", [1, 15, 17])
@pytest.mark.parametrize("path", ["generic", "waiting"])
def test_short_second_chunks(path, T):
    """Chunks of 1, 15 and 17 tokens after a prefix (one partial kChunk, one just past it); one token equals ssm_step."""
    from gfe_mamba_b200 import ops
    B, L, ED = PATH_SHAPES[path]
    t = _prep(make_scan_inputs(B, L + T, ED, seed=T + ED), torch.float32)
    _, h1 = _prefill(t, 0, L, None)
    y2, h2 = _prefill(t, L, L + T, h1)
    want = _oracle(t, grad=False, last=True)
    assert relerr(y2, want["out"][:, L:]) < 1e-4 and relerr(h2, want["last"]) < 1e-4
    if T == 1:
        with torch.no_grad():
            ys, hs = ops.ssm_step(t["u"][:, L], t["draw"][:, L], t["A_log"], t["Bm"][:, L], t["Cm"][:, L], t["D"], h1,
                                  z=t["z"][:, L], dt_bias=t["bias"])
        assert relerr(y2[:, 0], ys) < 1e-5 and relerr(h2, hs) < 1e-5


@pytest.mark.parametrize("use_bias,softplus", [(False, True), (True, False), (False, False)],
                         ids=["nobias-sp", "bias-nosp", "nobias-nosp"])
@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_bias_and_softplus_flags(path, use_bias, softplus):
    B, L, ED = PATH_SHAPES[path]
    d = make_scan_inputs(B, 2 * L, ED, seed=41 + ED)
    if not softplus:
        d["draw"] = np.abs(d["draw"]) * 0.2 + 1e-3
        d["bias"] = np.abs(d["bias"]) * 0.01
    t = _prep(d, torch.float32, use_bias=use_bias, softplus=softplus)
    y1, _, y2, h2 = _two_chunks(path, t, B, L, L, ED)
    want = _oracle(t, grad=False, last=True)
    assert relerr(torch.cat([y1, y2], 1), want["out"]) < 1e-4 and relerr(h2, want["last"]) < 1e-4


@pytest.mark.parametrize("dt", ["f32", "bf16"])
@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_strided_halves_and_unaligned_slices(path, dt):
    """u / z as the two halves of one (B, L, 2 ED) tensor, B / C as slices at offset R_UNALIGNED of one (B, L, R + 2N) tensor
    (on the chained paths: the plain-load staging); nothing is copied or modified."""
    dtype = DTYPES[dt]
    B, L, ED = PATH_SHAPES[path]
    d = make_scan_inputs(B, 2 * L, ED, seed=77 + ED)
    t = _prep(d, dtype, R=R_UNALIGNED)
    uz = torch.cat([t["u"].detach(), t["z"].detach()], -1)
    t["u"], t["z"] = uz[..., :ED], uz[..., ED:]
    before = [uz.clone(), t["bc"].detach().clone()]
    y1, _, y2, h2 = _two_chunks(path, t, B, L, L, ED)
    assert torch.equal(uz, before[0]) and torch.equal(t["bc"].detach(), before[1])
    want = _oracle(t, grad=False, last=True)
    assert relerr(torch.cat([y1, y2], 1), want["out"]) < TOL[dtype] and relerr(h2, want["last"]) < LAST_TOL[dtype]


@pytest.mark.parametrize("path", list(PATH_SHAPES))
def test_small_step_sizes_from_state(path):
    """dt_bias spread over [-16, -4] (delta down to ~1e-7): per-channel errors of the second chunk and of the final state."""
    B, L, ED = PATH_SHAPES[path]
    d = make_scan_inputs(B, 2 * L, ED, seed=19 + ED)
    d["bias"] = np.linspace(-16.0, -4.0, ED).astype(np.float32)
    t = _prep(d, torch.float32)
    _, _, y2, h2 = _two_chunks(path, t, B, L, L, ED)
    want = _oracle(t, grad=False, last=True)
    errs = dict(out=per_channel_err(y2, want["out"][:, L:], 2), last=per_channel_err(h2, want["last"], 1))
    worst = {k: float(e.max()) for k, e in errs.items()}
    assert all(v < 1e-3 for v in worst.values()), worst


# ------------------------------------------------------------------------------------------------- conv
CONV_LAYOUTS = {"packed": (64, 0), "unpacked": (42, 0), "misaligned": (64, 1)}


@pytest.mark.parametrize("layout", list(CONV_LAYOUTS))
@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("dt", list(DTYPES))
def test_conv1d_prefill(dt, K, layout):
    """conv1d_prefill from a random cache, chunks of 1, K-2 (< K-1: the new window mixes old cache entries and new rows), 5 and
    300 (three row tiles) tokens: u bitwise equal to causal_conv1d_silu over cat(cache, xin) in the same layout, the new window
    equal to the cache conv1d_step leaves after the same tokens, the cache unmodified."""
    from gfe_mamba_b200 import causal_conv1d_silu, ops
    dtype = DTYPES[dt]
    ED, off = CONV_LAYOUTS[layout]
    B = 3
    want_vec = 8 // torch.empty((), dtype=dtype).element_size()
    r = np.random.default_rng(K * 10 + ED + off)
    w = torch.from_numpy((r.standard_normal((ED, 1, K)) * 0.5).astype(np.float32)).cuda()
    b = torch.from_numpy((r.standard_normal(ED) * 0.1).astype(np.float32)).cuda()
    for Lc in sorted({1, K - 2, 5, 300} - {0}):
        # rows [0, K-1) of big hold the cache (transposed), rows [K-1, K-1+Lc) the chunk: one layout for both calls
        big = torch.from_numpy(r.standard_normal((B, K - 1 + Lc, 2 * ED + off)).astype(np.float32)).to("cuda", dtype)
        full = big[..., off:off + ED]
        xin = full[:, K - 1:]
        cache = full[:, :K - 1].transpose(1, 2).contiguous()                       # (B, ED, K-1)
        vec = conv_vec(dtype, ED, xin)
        assert vec == conv_vec(dtype, ED, full)
        assert (vec == want_vec) == (layout == "packed" or (layout == "unpacked" and dtype == torch.float32)), vec
        cache0 = cache.clone()
        with torch.no_grad():
            (u, new), n = launches(lambda: ops.conv1d_prefill(xin, cache, w, b))
            ref = causal_conv1d_silu(full, w, b)[:, K - 1:]
        assert n == {"conv1d_silu_fwd": 1}
        assert torch.equal(cache, cache0), "conv1d_prefill modified the cache"
        assert u.dtype == dtype and torch.equal(u, ref), (Lc, float((u.float() - ref.float()).abs().max()))
        c = cache
        with torch.no_grad():
            for s in range(Lc):
                _, c = ops.conv1d_step(xin[:, s], c, w, b)
        assert new.shape == (B, ED, K - 1) and torch.equal(new, c), Lc
        # from an empty cache: the rows of the forward over the chunk itself
        with torch.no_grad():
            u0, _ = ops.conv1d_prefill(xin, None, w, b)
            assert torch.equal(u0, causal_conv1d_silu(xin, w, b))


def test_conv1d_prefill_matches_oracle_across_chunks():
    from gfe_mamba_b200 import ops
    B, L, ED, K = 2, 300, 64, 4
    r = np.random.default_rng(3)
    x = r.standard_normal((B, L, ED)).astype(np.float32)
    w = (r.standard_normal((ED, 1, K)) * 0.5).astype(np.float32)
    b = (r.standard_normal(ED) * 0.1).astype(np.float32)
    xt, wt, bt = (torch.from_numpy(a).cuda() for a in (x, w, b))
    outs, cache = [], None
    with torch.no_grad():
        for s0, s1 in ((0, 2), (2, 9), (9, 250), (250, 300)):
            u, cache = ops.conv1d_prefill(xt[:, s0:s1], cache, wt, bt)
            outs.append(u)
    assert relerr(torch.cat(outs, 1), orc.conv1d_silu_fwd(x, w, b)) < 1e-5
    assert torch.equal(cache, xt[:, -(K - 1):].transpose(1, 2))


# ------------------------------------------------------------------------------------------------- model
MODEL_CFGS = {"chained": dict(d_model=64), "generic": dict(d_model=40), "N32": dict(d_model=64, d_state=32),
              "layernorms": dict(d_model=64, inner_layernorms=True), "dstate8": dict(d_model=32, d_state=8),
              "dconv5": dict(d_model=32, d_conv=5)}


def _model(name, seed=0):
    from gfe_mamba_b200 import Mamba, MambaConfig
    torch.manual_seed(seed)
    m = Mamba(MambaConfig(n_layers=2, **MODEL_CFGS[name])).cuda()
    with torch.no_grad():
        for layer in m.layers:
            layer.mixer.A_log.add_(0.1 * torch.randn_like(layer.mixer.A_log))
            layer.mixer.D.add_(0.1 * torch.randn_like(layer.mixer.D))
    return m


def _zero_caches(m, B, dtype):
    cfg = m.config
    return [(None, torch.zeros(B, cfg.d_inner, cfg.d_conv - 1, dtype=dtype, device="cuda")) for _ in m.layers]


def _steps(m, x, caches):
    ys = []
    for s in range(x.shape[1]):
        y, caches = m.step(x[:, s], list(caches))
        ys.append(y)
    return torch.stack(ys, 1), caches


def _cache_err(a, b):
    err = 0.0
    for (ha, wa), (hb, wb) in zip(a, b):
        err = max(err, relerr(ha, hb), relerr(wa, wb))
    return err


@pytest.mark.parametrize("amp", [False, True], ids=["f32", "bf16-autocast"])
@pytest.mark.parametrize("name", list(MODEL_CFGS))
def test_mamba_prefill_against_forward_and_step(name, amp):
    m = _model(name)
    B, P, T = 2, 40, 5
    x = torch.randn(B, P + T, m.config.d_model, device="cuda")
    tol = 3e-2 if amp else 1e-4
    dt = torch.bfloat16 if amp else torch.float32
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        y_fwd = m(x)
        y_pre, caches = m.prefill(x[:, :P])
        assert caches[0][1].dtype == dt
        y_dec, caches = _steps(m, x[:, P:], caches)
        y_ref, c_ref = _steps(m, x, _zero_caches(m, B, dt))
    assert relerr(y_pre, y_fwd[:, :P]) < tol
    assert relerr(y_dec, y_fwd[:, P:]) < tol
    assert relerr(torch.cat([y_pre, y_dec], 1), y_ref) < tol
    assert _cache_err(caches, c_ref) < tol


@pytest.mark.parametrize("amp", [False, True], ids=["f32", "bf16-autocast"])
@pytest.mark.parametrize("name", ["chained", "generic", "N32", "dstate8"])
def test_mamba_prefill_in_chunks(name, amp):
    """Prefill in uneven chunks (1, 7, 300, rest) equals one prefill; the chunks' inputs are not modified."""
    m = _model(name, seed=1)
    B, L = 2, 330
    x = torch.randn(B, L, m.config.d_model, device="cuda")
    tol = 3e-2 if amp else 1e-4
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        y_one, c_one = m.prefill(x)
        ys, caches = [], None
        for s0, s1 in ((0, 1), (1, 8), (8, 308), (308, L)):
            before = None if caches is None else [(None if h is None else h.clone(), w.clone()) for h, w in caches]
            y, new = m.prefill(x[:, s0:s1], caches)
            if before is not None:
                assert _cache_err(caches, before) == 0.0, "Mamba.prefill modified the caches it started from"
            ys.append(y)
            caches = new
    assert relerr(torch.cat(ys, 1), y_one) < tol
    assert _cache_err(caches, c_one) < tol


@pytest.mark.parametrize("name", ["chained", "generic", "N32"])
def test_graphed_decoder_from_prefill(name):
    from gfe_mamba_b200.decode import GraphedDecoder
    m = _model(name, seed=2)
    B, P, T = 2, 50, 6
    x = torch.randn(B, P + T, m.config.d_model, device="cuda")
    dec = GraphedDecoder(m, B)
    with torch.no_grad():
        _, caches = m.prefill(x[:, :P])
        dec.load_caches(caches)
        ys = torch.stack([dec.step(x[:, P + s]).clone() for s in range(T)], 1)
        y_ref, _ = _steps(m, x[:, P:], caches)
    assert relerr(ys, y_ref) < 1e-4


def test_prefill_under_grad_takes_the_step_loop():
    """Trainable parameters under grad: a differentiable output (the step loop) whose backward runs; the prefill ops refuse
    inputs that require grad."""
    from gfe_mamba_b200 import ops
    m = _model("chained", seed=3)
    x = torch.randn(2, 12, 64, device="cuda", requires_grad=True)
    y, caches = m.prefill(x)
    assert y.requires_grad
    y.square().mean().backward()
    assert torch.isfinite(x.grad).all() and m.layers[0].mixer.A_log.grad is not None
    with torch.no_grad():
        y0, _ = m.prefill(x)
    assert relerr(y.detach(), y0) < 1e-4
    mixer = m.layers[0].mixer
    xin = torch.randn(2, 12, mixer.config.d_inner, device="cuda", requires_grad=True)
    with pytest.raises(RuntimeError, match="inference-only"):
        ops.conv1d_prefill(xin, None, mixer.conv1d.weight, mixer.conv1d.bias)
    N = mixer.config.d_state
    bc = torch.randn(2, 12, N, device="cuda")
    with pytest.raises(RuntimeError, match="inference-only"):
        ops.ssm_prefill(xin, xin.detach(), mixer.A_log.detach(), bc, bc, mixer.D.detach(), None)


def test_prefill_peak_memory_at_the_production_shape():
    """B=2, L=1858, d_model=512, 6 layers under no_grad: no checkpoints are allocated -- the peak of prefill stays within that
    of forward plus the caches (2 MiB of allocator granularity allowed; one layer's checkpoints would be ~45 MB)."""
    from gfe_mamba_b200 import Mamba, MambaConfig
    torch.manual_seed(0)
    m = Mamba(MambaConfig(d_model=512, n_layers=6)).cuda()
    x = torch.randn(2, 1858, 512, device="cuda")

    def peak(fn):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        with torch.no_grad():
            res = fn()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base, res

    peak(lambda: m.prefill(x))   # warm-up (cuBLAS workspaces)
    p_fwd, _ = peak(lambda: m(x))
    p_pre, (_, caches) = peak(lambda: m.prefill(x))
    cache_bytes = sum(h.numel() * h.element_size() + w.numel() * w.element_size() for h, w in caches)
    assert p_pre <= p_fwd + cache_bytes + (2 << 20), (p_pre, p_fwd, cache_bytes)
