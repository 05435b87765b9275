"""GPU kernel matrix of the bandwidth kernels: every reachable variant of pscan, add + RMSNorm, pooling and clip + Adam
against plain fp64 references.

Like test_gpu_kernel_matrix.py this file is organised by the template instantiations the host code picks at run time, and
every case first proves which one it reached, from Python mirrors of the launch plans (pscan_plan + pscan_use_chain + the
16-byte alignment rule in pscan.cu, nv_for and norm_grid in addnorm.cu, the coef grid in optim.cu), from the library's
launch registry (whether the pscan summary passes ran) and from the arguments the C ABI received.  A changed plan therefore
fails the case instead of quietly moving it onto another kernel.
  * pscan: sequential forward <4,16> and <1,32>, sequential backward <4,8>, <2,16> and <1,32>, the L-split (summary pass,
    then <1,32>, both directions), the chained kernels with V = 4 and V = 1; each once with fresh tensors and once through
    contiguous views that start 1 element into a flat buffer (V = 1); L in {1, 7, 8, 9, 31, 32, 33} and ragged split
    lengths; A from [-1, 1] and [0.3, 1].  Reference: the sequential recurrence and its exact adjoint in fp64.
  * add + RMSNorm: (stream, branch) in {f32/f32, bf16/bf16, f16/f16, f32/bf16, f32/f16} x NV in {1, 2, 3, 4, 6, 8} (the
    row one vector short of 32 NV, so the last lane idles) and the two-pass wide kernels (257 vectors, and d_model 8192) x
    with / without `a` x with / without the dres stream, plus rows = 3 x (4 CTAs x 8 warps x SMs) + 5 for one NV and the wide
    kernels per pair (grid-stride row loop, dw over several rows per lane and the dw_wide row slices); dw is bitwise
    reproducible.
  * pooling: f32 / bf16 / f16, with / without r, L from 1 to 1858, D from 1 to 129; fp32 next to a 16-bit operand in either
    order (fp32 output, gradients in each operand's dtype); Mamba.forward_mean under bf16 / fp16 autocast.
  * clip + Adam: parameters and gradients at offsets that are not multiples of 4 elements (the scalar paths of the sum of
    squares and the update); state_dict round trips through torch.save, into the same optimiser, and to and from
    torch.optim.Adam; a graph captured over the step replays correctly after a state load.
Tolerances: test_gpu_parity.TOL (max-normalised per tensor) unless a case says otherwise.
"""
import contextlib
import copy
import io

import numpy as np
import pytest
import torch

from test_gpu_kernel_matrix import _sms, launches
from test_gpu_parity import TOL, relerr

pytestmark = pytest.mark.gpu

DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


@contextlib.contextmanager
def abi_calls(name):
    """Record the arguments of every call of the C entry point ``name`` made through _native.lib() in the block."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    fn = getattr(lib, name)
    calls = []

    def spy(*args):
        calls.append(args)
        return fn(*args)
    setattr(lib, name, spy)
    try:
        yield calls
    finally:
        setattr(lib, name, fn)


def _addr(p):
    """A c_void_p argument as an integer address (0 for NULL)."""
    return p.value or 0


# ================================================================================================================= pscan
K_MAX_SEG = 256   # common.cuh kMaxSeg


def pscan_plan(B, L, DN, nloads):
    """pscan_plan (pscan.cu): (V, U, nseg)."""
    target = 12e6 * _sms() / 148.0
    per_u = float(B) * float(DN) * 4.0 * nloads
    if nloads == 2:
        V, U = 4, 16
        if DN % 4 != 0 or per_u * 16 < target:
            V, U = 1, 32
    else:
        V, U = 4, 8
        if DN % 4 != 0 or per_u * 8 < target:
            V, U = 2, 16
        if DN % 2 != 0 or per_u * 16 < target:
            V, U = 1, 32
    S = 1
    if per_u * U * 2 < target:
        S = max(1, min(int(target / (per_u * U)), L // 64, K_MAX_SEG))
    seg_len = -(-(-(-L // S)) // 32) * 32
    return V, U, -(-L // seg_len)


def pscan_variant(B, L, D, N, nloads, aligned):
    """The kernel gfe_pscan_fwd (nloads = 2) / gfe_pscan_bwd (3) launches: 'seq<V,U>', 'split<1,32>' (summary pass first)
    or 'chain<V>'."""
    DN = D * N
    V, U, nseg = pscan_plan(B, L, DN, nloads)
    if nseg > 1:
        assert V == 1, "the plan splits L only after falling to (1, 32)"
        return "split<1,32>"
    if L >= 32:   # pscan_use_chain
        return f"chain<{4 if aligned and DN % 4 == 0 else 1}>"
    return f"seq<{V},{U}>" if aligned else "seq<1,32>"


def _batch_for(D, N, L, fwd, bwd):
    """The smallest batch whose launch plans give the wanted fresh-tensor variants."""
    for B in range(1, 513):
        if pscan_variant(B, L, D, N, 2, True) == fwd and pscan_variant(B, L, D, N, 3, True) == bwd:
            return B
    raise AssertionError(f"no batch up to 512 gives {fwd} / {bwd} at (L={L}, D={D}, N={N}) on {_sms()} SMs")


def pscan_ref(A, X, dH):
    """H[t] = A[t] H[t-1] + X[t] over dim 1 and its exact adjoint, in fp64."""
    A, X, dH = (np.asarray(t, np.float64) for t in (A, X, dH))
    L = A.shape[1]
    H, dX = np.empty_like(X), np.empty_like(X)
    h = np.zeros_like(X[:, 0])
    for t in range(L):
        h = A[:, t] * h + X[:, t]
        H[:, t] = h
    g = np.zeros_like(X[:, 0])
    for t in reversed(range(L)):
        g = dH[:, t] + (A[:, t + 1] * g if t + 1 < L else 0.0)
        dX[:, t] = g
    dA = np.zeros_like(X)
    dA[:, 1:] = H[:, :-1] * dX[:, 1:]
    return H, dA, dX


def _operand(a, misaligned):
    """A fresh CUDA tensor, or a contiguous view starting 1 element into a flat buffer (4 bytes past 16-byte alignment)."""
    t = torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()
    if not misaligned:
        return t
    flat = torch.full((t.numel() + 1,), float("nan"), device="cuda")
    v = flat[1:].view(t.shape)
    v.copy_(t)
    return v


# (fwd variant, bwd variant) -> (D, N, L values); the batch comes from the plan mirror
PSCAN_GROUPS = {
    ("seq<4,16>", "seq<4,8>"): (1024, 16, [1, 7, 8, 9, 20, 31]),
    ("seq<1,32>", "seq<2,16>"): (1025, 2, [7, 24]),
    ("seq<1,32>", "seq<1,32>"): (5, 3, [1, 7, 8, 9, 31]),
    ("chain<4>", "chain<4>"): (1024, 16, [32, 33]),
    ("chain<1>", "chain<1>"): (5, 3, [32, 33, 100]),
    ("split<1,32>", "split<1,32>"): (4, 4, [2100, 1000]),
}
PSCAN_CASES = [pytest.param(fwd, bwd, L, mis, arange, id=f"{fwd}-{bwd}-L{L}-{'misaligned' if mis else 'fresh'}-A{arange}")
               for (fwd, bwd), (_, _, Ls) in PSCAN_GROUPS.items() for L in Ls for mis in (False, True)
               for arange in ("pm1", "pos")]


@pytest.mark.parametrize("fwd,bwd,L,misaligned,arange", PSCAN_CASES)
def test_pscan_matrix(fwd, bwd, L, misaligned, arange):
    """pscan_fwd_kernel / pscan_bwd_kernel <V, U, SUMMARY> and pscan_{fwd,bwd}_chain_kernel<V>: H, dA and dX against the fp64
    recurrence; dA[:, 0] == 0 exactly; A, X and dH unmodified."""
    from gfe_mamba_b200 import pscan
    D, N, _ = PSCAN_GROUPS[(fwd, bwd)]
    Bsz = _batch_for(D, N, L, fwd, bwd)
    shape = (Bsz, L, D, N)
    r = np.random.default_rng(L * 31 + D + misaligned)
    A = r.uniform(-1.0, 1.0, shape) if arange == "pm1" else r.uniform(0.3, 1.0, shape)
    A = A.astype(np.float32)
    X, dH = r.standard_normal(shape).astype(np.float32), r.standard_normal(shape).astype(np.float32)
    At, Xt, dHt = _operand(A, misaligned), _operand(X, misaligned), _operand(dH, misaligned)
    aligned = all(t.data_ptr() % 16 == 0 for t in (At, Xt, dHt))
    assert aligned != misaligned
    want_f = pscan_variant(*shape, 2, aligned)
    want_b = pscan_variant(*shape, 3, aligned)
    if misaligned:   # V = 1 whatever the plan; the split and the chain keep their schedule
        want_f_named = {"split<1,32>": "split<1,32>", "chain<4>": "chain<1>", "chain<1>": "chain<1>"}.get(fwd, "seq<1,32>")
        want_b_named = {"split<1,32>": "split<1,32>", "chain<4>": "chain<1>", "chain<1>": "chain<1>"}.get(bwd, "seq<1,32>")
    else:
        want_f_named, want_b_named = fwd, bwd
    assert (want_f, want_b) == (want_f_named, want_b_named), f"the plans of {shape} give {want_f} / {want_b}"
    before = [t.clone() for t in (At, Xt, dHt)]
    At.requires_grad_()
    Xt.requires_grad_()

    def run():
        H = pscan(At, Xt)
        H.backward(dHt)
        return H.detach()
    with abi_calls("gfe_pscan_fwd") as fw, abi_calls("gfe_pscan_bwd") as bw:
        H, n = launches(run)
    # the kernels read the tensors themselves (the alignment above is theirs), not copies
    assert [_addr(v) for v in fw[0][:2]] == [At.data_ptr(), Xt.data_ptr()]
    assert [_addr(v) for v in (bw[0][0], bw[0][2])] == [At.data_ptr(), dHt.data_ptr()]
    want_n = {"pscan_fwd": 1, "pscan_bwd": 1}
    if want_f.startswith("split"):
        want_n["pscan_fwd_summary"] = 1
    if want_b.startswith("split"):
        want_n["pscan_bwd_summary"] = 1
    assert n == want_n, f"launched {n}, expected {want_n}"
    for t, t0 in zip((At, Xt, dHt), before):
        assert torch.equal(t.detach(), t0), "pscan modified an input"
    H_ref, dA_ref, dX_ref = pscan_ref(A, X, dH)
    assert float(At.grad[:, 0].abs().max()) == 0.0, "dA[:, 0] must be exactly 0 (no state before step 0)"
    assert relerr(H, H_ref) < 1e-5
    assert relerr(Xt.grad, dX_ref) < 1e-5
    assert relerr(At.grad, dA_ref) < 1e-5


# ========================================================================================================= add + RMSNorm
NORM_PAIRS = {"f32/f32": (torch.float32, torch.float32), "bf16/bf16": (torch.bfloat16, torch.bfloat16),
              "f16/f16": (torch.float16, torch.float16), "f32/bf16": (torch.float32, torch.bfloat16),
              "f32/f16": (torch.float32, torch.float16)}
NORM_WARPS = 8


def _vec(tr):
    return 16 // torch.empty((), dtype=tr).element_size()


def nv_for(D, tr):
    """nv_for (addnorm.cu): 16-byte vectors per lane held in registers; 0 = the two-pass wide kernels."""
    nvec = D // _vec(tr)
    for nv in (1, 2, 3, 4, 6, 8):
        if nvec <= 32 * nv:
            return nv
    return 0


def norm_grid(rows):
    """norm_grid (addnorm.cu): one warp per row, at most 4 CTAs of 8 warps per SM (persistent, grid-stride over rows)."""
    return min(max(-(-rows // NORM_WARPS), 1), 4 * _sms())


def norm_cap_rows():
    return 4 * NORM_WARPS * _sms()


def _norm_d(width, tr):
    """d_model of a width: NV -> one vector short of 32 NV vectors; 'wide257' -> 257 vectors; 'wide8192' -> 8192."""
    if width == "wide257":
        return 257 * _vec(tr)
    if width == "wide8192":
        return 8192
    return (32 * width - 1) * _vec(tr)


NORM_WIDTHS = [1, 2, 3, 4, 6, 8, "wide257", "wide8192"]
NORM_CASES = [pytest.param(pair, w, has_a, has_dres, "small", id=f"{pair}-{'NV' + str(w) if isinstance(w, int) else w}-"
                           f"{'a' if has_a else 'noa'}-{'dres' if has_dres else 'nodres'}")
              for pair in NORM_PAIRS for w in NORM_WIDTHS for has_a in (True, False) for has_dres in (True, False)]
NORM_CASES += [pytest.param(pair, w, True, True, "many", id=f"{pair}-{'NV' + str(w) if isinstance(w, int) else w}-many-rows")
               for pair in NORM_PAIRS for w in (2, "wide257")]


def _norm_run(x0, a0, w0, dres, dy):
    from gfe_mamba_b200 import add_rmsnorm
    x = x0.clone().requires_grad_()
    a = None if a0 is None else a0.clone().requires_grad_()
    w = w0.clone().requires_grad_()
    resid, y = add_rmsnorm(x, a, w, 1e-5, out_dtype=dy.dtype)
    loss = (y.float() * dy.float()).sum()
    if dres is not None:
        loss = loss + (resid.float() * dres.float()).sum()
    loss.backward()
    return dict(resid=resid.detach(), y=y.detach(), dx=x.grad, da=None if a is None else a.grad, dw=w.grad)


@pytest.mark.parametrize("pair,width,has_a,has_dres,rows_kind", NORM_CASES)
def test_add_rmsnorm_matrix(pair, width, has_a, has_dres, rows_kind):
    """add_rmsnorm_{fwd,bwd}_kernel<TR, TB, NV, HAS_A / HAS_DRES> and the *_wide kernels (+ dw_wide, dw_finalize): resid, y,
    dx, da, dw against torch fp64 on the values the kernels read; dw bitwise reproducible."""
    tr, tb = NORM_PAIRS[pair]
    D = _norm_d(width, tr)
    rows = 3 * norm_cap_rows() + 5 if rows_kind == "many" else 37
    want_nv = 0 if isinstance(width, str) else width
    assert nv_for(D, tr) == want_nv, f"d_model {D} selects NV = {nv_for(D, tr)}"
    if want_nv:
        assert D // _vec(tr) == 32 * want_nv - 1   # the last lane of the last vector column idles
    if rows_kind == "many":
        assert norm_grid(rows) * NORM_WARPS < rows / 3, "the grid-stride loop must run every warp over several rows"
    g = torch.Generator(device="cpu").manual_seed(rows + D + 7 * has_a + 3 * has_dres)
    x0 = torch.randn(rows, D, generator=g).to(tr).cuda()
    a0 = torch.randn(rows, D, generator=g).to(tb).cuda() if has_a else None
    w0 = (1 + 0.1 * torch.randn(D, generator=g)).cuda()
    dres = torch.randn(rows, D, generator=g).to(tr).cuda() if has_dres else None
    dy = torch.randn(rows, D, generator=g).to(tb).cuda()
    with abi_calls("gfe_add_rmsnorm_fwd_mixed") as fw, abi_calls("gfe_add_rmsnorm_bwd_mixed") as bw:
        got, n = launches(lambda: _norm_run(x0, a0, w0, dres, dy))
    assert n == {"add_rmsnorm_fwd": 1, "add_rmsnorm_bwd": 1, "add_rmsnorm_dw_finalize": 1}, n
    assert len(fw) == 1 and len(bw) == 1
    assert (_addr(fw[0][1]) != 0) == has_a, "HAS_A"
    assert (_addr(bw[0][4]) != 0) == has_dres, "HAS_DRES: an unused resid must reach the kernels as no dres stream"
    assert (_addr(bw[0][6]) != 0) == (has_a and tb != tr), "da written by the kernel only for a branch of another dtype"
    # fp64 reference on the rounded inputs: resid rounded to the stream dtype, the gradient of the exact sum
    xd = x0.double().requires_grad_()
    ad = a0.double().requires_grad_() if has_a else None
    wd = w0.double().requires_grad_()
    rd = (xd + ad).detach().to(tr).double() + ((xd + ad) - (xd + ad).detach()) if has_a else xd
    yd = rd * torch.rsqrt(rd.pow(2).mean(-1, keepdim=True) + 1e-5) * wd
    loss = (yd * dy.double()).sum()
    if has_dres:
        loss = loss + (rd * dres.double()).sum()
    loss.backward()
    assert got["resid"].dtype == tr and got["y"].dtype == tb and got["dx"].dtype == tr
    if tr == tb:
        tol = TOL[tr]
        assert relerr(got["resid"], rd.detach()) < tol and relerr(got["y"], yd.detach()) < tol
        assert relerr(got["dx"], xd.grad) < tol and relerr(got["dw"], wd.grad) < tol
        if has_a:
            assert relerr(got["da"], ad.grad) < tol
    else:
        assert relerr(got["resid"], rd.detach()) < 1e-6 and relerr(got["y"], yd.detach()) < TOL[tb]
        assert relerr(got["dx"], xd.grad) < 1e-5 and relerr(got["dw"], wd.grad) < 1e-4
        if has_a:
            assert got["da"].dtype == tb and relerr(got["da"], ad.grad) < TOL[tb]
            assert torch.equal(got["da"], got["dx"].to(tb))   # the same values, rounded once
    again = _norm_run(x0, a0, w0, dres, dy)
    assert torch.equal(again["dw"], got["dw"]), "dw is not bitwise reproducible"


# ================================================================================================================ pooling
POOL_LS = [1, 2, 63, 64, 65, 1858]
POOL_DS = [1, 127, 128, 129]
POOL_CASES = [pytest.param(dt, dt if has_r else None, L, D, id=f"{dt}-{'r' if has_r else 'nor'}-L{L}-D{D}")
              for i, dt in enumerate(DTYPES) for has_r in (True, False) for j, L in enumerate(POOL_LS)
              for k, D in enumerate(POOL_DS) if (i + j + k + has_r) % 2 == 0]
POOL_CASES += [pytest.param(a, r, L, D, id=f"{a}+{r}-L{L}-D{D}") for a, r in (("bf16", "f32"), ("f32", "bf16"), ("f16", "f32"),
                                                                              ("f32", "f16"))
               for L, D in ((1, 129), (65, 128), (1858, 127))]


@pytest.mark.parametrize("adt,rdt,L,D", POOL_CASES)
def test_add_mean_pool_matrix(adt, rdt, L, D):
    """add_mean_pool_partial_kernel<TA, TR> + add_mean_pool_final_kernel<TO>, mean_pool_bwd_kernel<TA, TR>: the mean of the
    rounded operands in fp64, the output in torch's promoted dtype, and each gradient (dout / L rounded once to its
    operand's dtype) exact; no dtype cast of the (B, L, D) operands or their gradients outside the kernels."""
    from gfe_mamba_b200 import add_mean_pool
    ta = DTYPES[adt]
    tr = None if rdt is None else DTYPES[rdt]
    to = ta if tr is None else torch.promote_types(ta, tr)
    B = 3
    g = torch.Generator(device="cpu").manual_seed(L * 131 + D)
    a = (torch.randn(B, L, D, generator=g) + 3.0).to(ta).cuda().requires_grad_()   # nonzero means: the max-normalised
    r = None if tr is None else (torch.randn(B, L, D, generator=g) - 1.0).to(tr).cuda().requires_grad_()   # error is meaningful
    dout = torch.randn(B, 1, D, generator=g).to(to).cuda()

    def run():
        out = add_mean_pool(a, r)
        out.backward(dout)
        return out.detach()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU]) as prof:
        out, n = launches(run)
    assert n == {"add_mean_pool_fwd": 1, "mean_pool_bwd": 1}, n
    casts = [e.key for e in prof.key_averages() if e.key == "aten::_to_copy"]
    assert not casts, "a dtype cast pass over the (B, L, D) operands or their gradients"
    ref = a.detach().double() + (0.0 if r is None else r.detach().double())
    ref = ref.mean(1, keepdim=True)
    assert out.shape == (B, 1, D) and out.dtype == to
    assert relerr(out, ref) < (1e-6 if to == torch.float32 else TOL[to])
    gd = torch.from_numpy(dout.float().cpu().numpy() / np.float32(L)).cuda()   # correctly rounded, as the kernel divides
    assert a.grad.dtype == ta and torch.equal(a.grad, gd.to(ta).expand(B, L, D))
    if r is not None:
        assert r.grad.dtype == tr and torch.equal(r.grad, gd.to(tr).expand(B, L, D))


def test_add_mean_pool_rejects_two_16bit_dtypes():
    """bf16 with fp16 has no native kernel (torch would promote to fp32): refused, not cast behind the caller's back."""
    from gfe_mamba_b200 import add_mean_pool
    a = torch.randn(2, 5, 8, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(TypeError):
        add_mean_pool(a, a.half())


@pytest.mark.parametrize("dt", ["bf16", "f16"])
def test_mamba_forward_mean_under_autocast(dt):
    """Mamba.forward_mean == torch.mean(model(x), 1, keepdim=True) under the same autocast: fp32 output (the last 16-bit
    branch plus the fp32 residual stream), the same values, and the same gradients for the same upstream gradient (a loss
    of the output would hand the two backward passes gradients that differ in the last fp32 bit, enough to flip the 16-bit
    rounding of the branch gradient here and there)."""
    from gfe_mamba_b200 import Mamba, MambaConfig
    torch.manual_seed(4)
    model = Mamba(MambaConfig(d_model=64, n_layers=2)).cuda()
    x = torch.randn(2, 77, 64, device="cuda")
    dy = torch.randn(2, 1, 64, device="cuda")
    x1, x2 = x.clone().requires_grad_(), x.clone().requires_grad_()
    with torch.autocast("cuda", dtype=DTYPES[dt]):
        y1 = torch.mean(model(x1), dim=1, keepdim=True)
    y1.backward(dy)
    g1 = [p.grad.clone() for p in model.parameters()]
    model.zero_grad()
    with torch.autocast("cuda", dtype=DTYPES[dt]):
        y2 = model.forward_mean(x2)
    assert y1.dtype == torch.float32 and y2.dtype == y1.dtype
    y2.backward(dy)
    assert relerr(y2, y1) <= 1e-5
    assert relerr(x2.grad, x1.grad) <= 1e-4
    for (name, p), ga in zip(model.named_parameters(), g1):
        assert relerr(p.grad, ga) <= 1e-4, name


# =========================================================================================================== clip + Adam
OPT_TENSORS_PER_CTA = 8   # opt_coef_kernel: one warp per tensor, 256 threads


def _set_grads(ps, gs):
    for p, g in zip(ps, gs):
        p.grad.copy_(g)


def _grads(seed, shapes, steps, scale=1.0):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return [[torch.randn(s, device="cuda", generator=gen) * scale for s in shapes] for _ in range(steps)]


def _torch_step(ref, opt_ref, grads, max_norm):
    for q, g in zip(ref, grads):
        q.grad = g.clone()
    if max_norm is not None:
        for q in ref:
            torch.nn.utils.clip_grad_norm_(q, max_norm=max_norm)
    opt_ref.step()


def test_clip_adam_unaligned_views():
    """Parameters and gradients as views into flat fp32 buffers at element offsets that are not multiples of 4: the scalar
    paths of opt_sumsq_kernel and opt_adam_kernel, against torch's clip loop + Adam over 4 steps."""
    from gfe_mamba_b200.optim import ClipAdam
    shapes = [(1000,), (37, 5), (4097,), (3,), (64, 65), (9000,)]
    numels = [int(np.prod(s)) for s in shapes]
    offs, o = [], 1
    for n in numels:
        offs.append(o)
        o += n + 2 + (1 if (o + n + 2) % 4 == 0 else 0)
    assert all(off % 4 != 0 for off in offs)
    gen = torch.Generator(device="cuda").manual_seed(11)
    flat_p, flat_g = torch.randn(o + 3, device="cuda", generator=gen), torch.zeros(o + 3, device="cuda")
    pad0 = float(flat_p[0])
    ours = [flat_p[off:off + n].view(s) for off, n, s in zip(offs, numels, shapes)]
    for p, off, n, s in zip(ours, offs, numels, shapes):
        p.grad = flat_g[off:off + n].view(s)
    chunk = 4096
    for p in ours:   # every chunk starts off 16-byte alignment: the vector paths are ruled out
        assert all((p.data_ptr() + 4 * st) % 16 != 0 and (p.grad.data_ptr() + 4 * st) % 16 != 0 for st in range(0, p.numel(), chunk))
    ref = [torch.nn.Parameter(p.detach().clone()) for p in ours]
    grads = _grads(12, shapes, 4, scale=3.0)
    opt_ref = torch.optim.Adam(ref, lr=1e-2)
    opt = ClipAdam(ours, lr=1e-2, max_norm=1.0, per_parameter_clip=True, zero_grad=False)
    for step in range(4):
        _set_grads(ours, grads[step])
        _torch_step(ref, opt_ref, grads[step], 1.0)
        _, n = launches(opt.step)
        assert n == {"clip_adam_sumsq": 1, "clip_adam_coef": 1, "clip_adam_update": 1}, n
        for p, q in zip(ours, ref):
            assert torch.allclose(p, q, rtol=2e-6, atol=2e-7), (step, p.shape, (p - q).abs().max().item())
            assert torch.allclose(p.grad, q.grad, rtol=1e-5, atol=1e-8), "clipped gradients differ"
    assert float(flat_g[0]) == 0.0 and float(flat_p[0]) == pad0   # the element in front of the first view is untouched


STATE_SHAPES = [(300, 16), (300,), (64, 300), (7,), (4097,)]


def _opt_run(opt_cls, params, grads, **kw):
    opt = opt_cls(params, **kw)
    for g in grads:
        for p, gi in zip(params, g):
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            p.grad.copy_(gi)
        opt.step()
    return opt


def _fresh_params(seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return [torch.nn.Parameter(torch.randn(s, device="cuda", generator=gen)) for s in STATE_SHAPES]


def _copies(ps):
    return [torch.nn.Parameter(p.detach().clone()) for p in ps]


def test_clip_adam_state_round_trip_through_torch_save():
    """3 steps, state_dict through torch.save / torch.load, a fresh ClipAdam over copies of the parameters, 3 more steps:
    bitwise the uninterrupted 6 steps (moments and the bias-correction step both come back)."""
    from gfe_mamba_b200.optim import ClipAdam
    kw = dict(lr=1e-2, max_norm=1.0)
    grads = _grads(21, STATE_SHAPES, 6, scale=2.0)
    whole = _fresh_params(20)
    part = _copies(whole)
    _opt_run(ClipAdam, whole, grads, **kw)
    first = _opt_run(ClipAdam, part, grads[:3], **kw)
    sd = first.state_dict()
    assert all(float(st["step"]) == 3.0 and st["step"].dtype == torch.float32 and st["step"].device.type == "cpu"
               for st in sd["state"].values())
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    resumed = _copies(part)
    opt = ClipAdam(resumed, **kw)
    opt.load_state_dict(torch.load(buf))
    for g in grads[3:]:
        for p, gi in zip(resumed, g):
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            p.grad.copy_(gi)
        opt.step()
    for p, q in zip(resumed, whole):
        assert torch.equal(p, q), (p - q).abs().max().item()
    assert all(float(st["step"]) == 6.0 for st in opt.state_dict()["state"].values())


def test_clip_adam_reload_earlier_state_into_same_optimizer():
    """Load an earlier, deep-copied state into the SAME optimiser after it moved on: the moments are copied into the buffers
    its device tables point at, the step counter is rewound, and 3 more steps match the uninterrupted run bitwise."""
    from gfe_mamba_b200.optim import ClipAdam
    kw = dict(lr=1e-2, max_norm=1.0)
    grads = _grads(31, STATE_SHAPES, 6, scale=2.0)
    detour = _grads(32, STATE_SHAPES, 2, scale=5.0)
    whole = _fresh_params(30)
    ps = _copies(whole)
    _opt_run(ClipAdam, whole, grads, **kw)
    opt = _opt_run(ClipAdam, ps, grads[:3], **kw)
    sd = copy.deepcopy(opt.state_dict())
    snap = [p.detach().clone() for p in ps]
    for g in detour:
        _set_grads(ps, g)
        opt.step()
    held = [(st["exp_avg"], st["exp_avg_sq"]) for st in opt.state.values()]   # alive whatever load_state_dict does
    addrs = [(m.data_ptr(), v.data_ptr()) for m, v in held]
    with torch.no_grad():
        for p, s in zip(ps, snap):
            p.copy_(s)
    opt.load_state_dict(sd)
    assert [(st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()) for st in opt.state.values()] == addrs
    assert all("step" not in st for st in opt.state.values())
    for g in grads[3:]:
        _set_grads(ps, g)
        opt.step()
    for p, q in zip(ps, whole):
        assert torch.equal(p, q), (p - q).abs().max().item()
    del held


def test_clip_adam_rejects_mixed_steps_in_one_group():
    from gfe_mamba_b200.optim import ClipAdam
    ps = _fresh_params(40)
    opt = _opt_run(ClipAdam, ps, _grads(41, STATE_SHAPES, 2))
    sd = copy.deepcopy(opt.state_dict())
    sd["state"][1]["step"] = torch.tensor(5.0)
    with pytest.raises(ValueError, match="step"):
        opt.load_state_dict(sd)


@pytest.mark.parametrize("direction", ["adam_to_clipadam", "clipadam_to_adam"])
def test_clip_adam_state_interop_with_torch_adam(direction):
    """A torch.optim.Adam state dict continues in ClipAdam(max_norm=None) as Adam does, and the reverse."""
    from gfe_mamba_b200.optim import ClipAdam
    grads = _grads(51, STATE_SHAPES, 6, scale=2.0)
    whole = _fresh_params(50)
    part = _copies(whole)
    _opt_run(torch.optim.Adam, whole, grads, lr=1e-2)
    if direction == "adam_to_clipadam":
        first, second = _opt_run(torch.optim.Adam, part, grads[:3], lr=1e-2), ClipAdam
    else:
        first, second = _opt_run(ClipAdam, part, grads[:3], lr=1e-2, max_norm=None), torch.optim.Adam
    sd = copy.deepcopy(first.state_dict())
    resumed = _copies(part)
    opt = second(resumed, lr=1e-2, **({"max_norm": None} if second is ClipAdam else {}))
    opt.load_state_dict(sd)
    for g in grads[3:]:
        for p, gi in zip(resumed, g):
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            p.grad.copy_(gi)
        opt.step()
    for p, q in zip(resumed, whole):
        assert torch.allclose(p, q, rtol=2e-6, atol=2e-7), (p - q).abs().max().item()


def test_graphed_train_step_replays_after_state_load():
    """GraphedTrainStep after ClipAdam.load_state_dict: the captured graph keeps its addresses (moments refilled in place,
    device step counter rewound), so replaying the same inputs after the load repeats the first replays."""
    from gfe_mamba_b200 import ClipAdam, Mamba, MambaConfig
    from gfe_mamba_b200.train import GraphedTrainStep, TrainStep
    xs = [torch.randn(2, 130, 64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(i)) for i in range(4)]
    torch.manual_seed(7)
    m = Mamba(MambaConfig(d_model=64, n_layers=2)).cuda()
    opt = ClipAdam(m.parameters(), lr=1e-3, max_norm=1.0, zero_grad=True)
    g = GraphedTrainStep(TrainStep(m, opt), xs[0], warmup=3)
    for x in xs[:2]:
        g(x)
    sd = copy.deepcopy(opt.state_dict())
    snap = [p.detach().clone() for p in m.parameters()]
    held = [(st["exp_avg"], st["exp_avg_sq"]) for st in opt.state.values()]
    addrs = [(a.data_ptr(), b.data_ptr()) for a, b in held]
    first = [float(g(x)) for x in xs[2:]]
    after = [p.detach().clone() for p in m.parameters()]
    with torch.no_grad():
        for p, s in zip(m.parameters(), snap):
            p.copy_(s)
    opt.load_state_dict(sd)
    assert [(st["exp_avg"].data_ptr(), st["exp_avg_sq"].data_ptr()) for st in opt.state.values()] == addrs
    second = [float(g(x)) for x in xs[2:]]
    assert np.allclose(first, second, rtol=1e-6, atol=0), (first, second)
    for p, q in zip(m.parameters(), after):
        assert torch.allclose(p, q, rtol=1e-6, atol=1e-9), (p - q).abs().max().item()
    del held
