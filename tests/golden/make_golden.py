"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED reference.

Needs a checkout of the original GFE-Mamba:
            GFE_REFERENCE=<checkout> python tests/golden/make_golden.py

The fixtures pin the oracle (tests/test_oracle_golden.py, CPU) and are compared
with the CUDA path directly (tests/test_gpu_parity.py, GPU).  What is recorded:

  pscan_small.npz     reference pscan(A, X) + its custom backward, L in {1,2,3,4,5,8,37,64}
                      (every branch of cross_atten/pscan.py:65-75,168-174,206-211)
  selscan_small.npz   MambaBlock.selective_scan and selective_scan_seq (mamba.py:265-318) with
                      autograd gradients, L = 37 (pads to 64) and L = 64
  block_small.npz     one MambaBlock: state dict, forward, gradients of every parameter and of
                      the input, and step() replayed over the same sequence (mamba.py:197-225,342-405)
  mamba_cfg1.npz      BASELINE config 1: Mamba(d_model=128, n_layers=2), B=8, L=64, fp32; the seeded tensors
                      (state dict, x, dy) as shape + every SAMPLE_STRIDE-th value, redrawn from the seed by
                      the mamba_cfg1 fixture (tests/conftest.py): whole, the file would be over 1 MB
  block_ln.npz        the same as block_small for jamba's configuration, inner_layernorms=True (mamba.py:169-176,188-195)
  block_odd.npz       the same for d_state=8, d_conv=5: shapes outside the fused kernels (pscan composition, cuDNN conv)
"""
import os
import sys

import numpy as np
import torch

REF = os.environ.get("GFE_REFERENCE", "")
HERE = os.path.dirname(os.path.abspath(__file__))
CFG1_SEED, SAMPLE_STRIDE = 404, 17   # a prime stride: samples do not line up with the rows of any parameter


def _load_reference():
    if not REF or not os.path.isdir(os.path.join(REF, "cross_atten")):
        raise SystemExit("set GFE_REFERENCE to a checkout of the original GFE-Mamba")
    # make sure it is the reference's cross_atten that gets imported, not this repo's drop-in
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") != os.path.abspath(os.path.join(HERE, "..", ".."))]
    sys.path.insert(0, REF)
    for m in [k for k in sys.modules if k.startswith("cross_atten")]:
        del sys.modules[m]
    from cross_atten import mamba as ref_mamba, pscan as ref_pscan
    assert os.path.abspath(ref_mamba.__file__).startswith(os.path.abspath(REF)), ref_mamba.__file__
    return ref_mamba, ref_pscan


def np32(t):
    return t.detach().cpu().contiguous().numpy().astype(np.float32)


def gen_pscan(ref_pscan, out):
    g = torch.Generator().manual_seed(101)
    for L in (1, 2, 3, 4, 5, 8, 37, 64):
        B, D, N = 2, 3, 4
        A = (0.5 + 0.5 * torch.rand(B, L, D, N, generator=g)).requires_grad_()
        X = torch.randn(B, L, D, N, generator=g).requires_grad_()
        dH = torch.randn(B, L, D, N, generator=g)
        H = ref_pscan.pscan(A, X)
        H.backward(dH)
        for k, v in (("A", A), ("X", X), ("dH", dH), ("H", H), ("dA", A.grad), ("dX", X.grad)):
            out[f"L{L}_{k}"] = np32(v)


def gen_selscan(ref_mamba, out):
    g = torch.Generator().manual_seed(202)
    for tag, (B, L, D) in (("L37", (2, 37, 4)), ("L64", (2, 64, 8))):
        cfg = ref_mamba.MambaConfig(d_model=D, n_layers=1)
        blk = ref_mamba.MambaBlock(cfg)
        ED, N = cfg.d_inner, cfg.d_state
        x = torch.randn(B, L, ED, generator=g).requires_grad_()
        delta = torch.nn.functional.softplus(torch.randn(B, L, ED, generator=g) - 2.0).requires_grad_()
        A = (-torch.exp(torch.log(torch.arange(1, N + 1).float()).repeat(ED, 1)
                        + 0.1 * torch.randn(ED, N, generator=g))).requires_grad_()
        Bm = torch.randn(B, L, N, generator=g).requires_grad_()
        Cm = torch.randn(B, L, N, generator=g).requires_grad_()
        Dp = (1.0 + 0.1 * torch.randn(ED, generator=g)).requires_grad_()
        dy = torch.randn(B, L, ED, generator=g)
        y = blk.selective_scan(x, delta, A, Bm, Cm, Dp)                  # mamba.py:265 (pscan)
        y.backward(dy)
        with torch.no_grad():
            y_seq = blk.selective_scan_seq(x, delta, A, Bm, Cm, Dp)      # mamba.py:288
        for k, v in (("x", x), ("delta", delta), ("A", A), ("B", Bm), ("C", Cm), ("D", Dp), ("dy", dy),
                     ("y", y), ("y_seq", y_seq), ("dx", x.grad), ("ddelta", delta.grad), ("dA", A.grad),
                     ("dB", Bm.grad), ("dC", Cm.grad), ("dD", Dp.grad)):
            out[f"{tag}_{k}"] = np32(v)


def gen_block(ref_mamba, out, seed=303, d_model=16, B=2, L=19, **cfg_kw):
    torch.manual_seed(seed)
    cfg = ref_mamba.MambaConfig(d_model=d_model, n_layers=1, **cfg_kw)
    blk = ref_mamba.MambaBlock(cfg)
    with torch.no_grad():   # move A_log / D off their special init so their gradients are exercised
        blk.A_log.add_(0.1 * torch.randn_like(blk.A_log))
        blk.D.add_(0.1 * torch.randn_like(blk.D))
        for ln in (blk.dt_layernorm, blk.B_layernorm, blk.C_layernorm):
            if ln is not None:   # RMSNorm weights start at one: move them too
                ln.weight.add_(0.2 * torch.randn_like(ln.weight))
    x = torch.randn(B, L, cfg.d_model).requires_grad_()
    dy = torch.randn(B, L, cfg.d_model)
    y = blk(x)                                                           # mamba.py:197
    y.backward(dy)
    out["meta"] = np.array([cfg.d_model, cfg.d_state, cfg.expand_factor, cfg.d_conv, cfg.dt_rank, B, L], np.int64)
    out["x"], out["dy"], out["y"], out["dx"] = np32(x), np32(dy), np32(y), np32(x.grad)
    for k, v in blk.state_dict().items():
        out[f"sd.{k}"] = np32(v)
    for k, v in blk.named_parameters():
        out[f"grad.{k}"] = np32(v.grad)
    # step(): replay the same sequence token by token (mamba.py:342-373); cache init per mamba.py:335
    with torch.no_grad():
        cache = (None, torch.zeros(B, cfg.d_inner, cfg.d_conv - 1))
        ys = []
        for t in range(L):
            yt, cache = blk.step(x[:, t].detach(), cache)
            ys.append(yt)
        out["y_step"] = np32(torch.stack(ys, 1))
        out["h_last"] = np32(cache[0])
        out["inputs_last"] = np32(cache[1])


def gen_cfg1(ref_mamba, out):
    torch.manual_seed(CFG1_SEED)
    cfg = ref_mamba.MambaConfig(d_model=128, n_layers=2)                 # BASELINE.json configs[0]
    model = ref_mamba.Mamba(cfg)
    B, L = 8, 64
    x = torch.randn(B, L, cfg.d_model).requires_grad_()
    dy = torch.randn(B, L, cfg.d_model)
    y = model(x)
    y.backward(dy)
    out["meta"] = np.array([cfg.d_model, cfg.n_layers, cfg.d_state, cfg.expand_factor, cfg.d_conv, cfg.dt_rank, B, L],
                           np.int64)
    out["x"], out["dy"], out["y"], out["dx"] = np32(x), np32(dy), np32(y), np32(x.grad)
    for k, v in model.state_dict().items():
        out[f"sd.{k}"] = np32(v)
    for k, v in model.named_parameters():
        if k.startswith("layers.0.") and any(s in k for s in ("A_log", ".D", "dt_proj", "conv1d", "norm")):
            out[f"grad.{k}"] = np32(v.grad)
    sample_seeded(out)


def sample_seeded(out):
    """Replaces the tensors drawn from CFG1_SEED (state dict, x, dy) by their shapes and every SAMPLE_STRIDE-th value."""
    for k in [k for k in out if k.startswith("sd.") or k in ("x", "dy")]:
        v = out.pop(k)
        out[f"shape.{k}"] = np.array(v.shape, np.int64)
        out[f"sample.{k}"] = np.ascontiguousarray(v.reshape(-1)[::SAMPLE_STRIDE])
    out["seed"] = np.array(CFG1_SEED, np.int64)
    out["sample_stride"] = np.array(SAMPLE_STRIDE, np.int64)


def gen_block_ln(ref_mamba, out):
    gen_block(ref_mamba, out, seed=505, d_model=32, B=2, L=45, inner_layernorms=True)


def gen_block_odd(ref_mamba, out):
    gen_block(ref_mamba, out, seed=606, d_model=16, B=2, L=21, d_state=8, d_conv=5)


def main():
    ref_mamba, ref_pscan = _load_reference()
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    only = set(sys.argv[1:])
    for name, fn, mod in (("pscan_small", gen_pscan, ref_pscan), ("selscan_small", gen_selscan, ref_mamba),
                          ("block_small", gen_block, ref_mamba), ("mamba_cfg1", gen_cfg1, ref_mamba),
                          ("block_ln", gen_block_ln, ref_mamba), ("block_odd", gen_block_odd, ref_mamba)):
        if only and name not in only:
            continue
        out = {}
        fn(mod, out)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        print(f"{name}: {len(out)} arrays, {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
