"""CPU-only checks: the C-ABI library loads and exports every symbol include/gfe_mamba_b200.h declares (no compute
without a GPU), size queries answer, the Python surface mirrors the reference (names, defaults, state-dict keys,
seeded initialisation), and the product path refuses CPU tensors instead of falling back."""
import ctypes
import dataclasses
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "gfe_mamba_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"GFE_API\s+[\w\s\*]+?\b(gfe_\w+)\s*\(", src)))


def test_header_declares_expected_entry_points():
    syms = _declared_symbols()
    for must in ("gfe_pscan_fwd", "gfe_pscan_bwd", "gfe_selscan_fwd", "gfe_selscan_bwd", "gfe_conv1d_silu_fwd",
                 "gfe_conv1d_silu_bwd", "gfe_conv1d_step", "gfe_ssm_step", "gfe_version", "gfe_last_error_string"):
        assert must in syms
    assert len(syms) >= 19


def test_library_exports_every_declared_symbol():
    from gfe_mamba_b200 import _native
    raw = ctypes.CDLL(_native.LIB_PATH)
    for name in _declared_symbols():
        assert hasattr(raw, name), f"{name} declared in the header but not exported"
    lib = _native.lib()                      # also checks every signature in the ctypes table resolves
    assert set(_native.SIGNATURES) == set(_declared_symbols())
    assert lib.gfe_version() == 100
    assert lib.gfe_timing_kernel_count() == 23 and lib.gfe_timing_kernel_name(3) == b"selscan_bwd"


def test_size_queries_without_gpu():
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    B, L, ED, N = 16, 4096, 1536, 16
    states = B * (L // 8) * ED * N * 4                              # chained kernels checkpoint every 8 steps
    assert lib.gfe_selscan_ckpt_bytes(B, L, ED, N) == states + B * L * ED * 4
    assert lib.gfe_selscan_ckpt_bytes(1, 65536, 1024, N) == (65536 // 8) * 1024 * N * 4 + 65536 * 1024 * 4   # independent segments: same layout
    assert lib.gfe_selscan_ckpt_bytes(1, 65536, 1000, N) == (65536 // 16) * 1000 * N * 4 + 65536 * 1000 * 4  # generic kernels (ED % 32 != 0): every 16
    assert lib.gfe_selscan_ckpt_bytes(B, L, ED, 8) == 0            # unsupported d_state -> 0
    # bf16 activations: bf16 state checkpoints and y before the gate in bf16 -- half of everything saved for backward
    assert lib.gfe_selscan_ckpt_bytes_dt(B, L, ED, N, _native.GFE_BF16) == states // 2 + B * L * ED * 2 <= 0.61e9
    assert lib.gfe_selscan_ckpt_bytes_dt(B, L, ED, N, _native.GFE_F16) == states + B * L * ED * 2     # fp16 keeps fp32 states (range)
    assert lib.gfe_selscan_ckpt_bytes_dt(B, L, ED, N, _native.GFE_F32) == lib.gfe_selscan_ckpt_bytes(B, L, ED, N)
    # one dB|dC row (32 fp32) per (channel block of <= 64 channels, token)
    assert (ED // 64) * B * L * 32 * 4 <= lib.gfe_selscan_bwd_workspace_bytes(B, L, ED, N) < (ED // 32) * B * L * 32 * 4
    # chained segments: counter + flags + one (B, ED, N) fp32 carry; far below one activation tensor
    assert B * ED * N * 4 < lib.gfe_selscan_fwd_workspace_bytes(B, L, ED, N) < B * L * ED
    assert lib.gfe_selscan_fwd_workspace_bytes(1, 65536, 1024, N) > 0   # cfg4 splits L
    assert lib.gfe_pscan_workspace_bytes(32, 256, 512, 16) == 0
    assert lib.gfe_pscan_workspace_bytes(1, 65536, 4, 16) > 0
    assert lib.gfe_conv1d_bwd_workspace_bytes(2, 130, 64, 4) == 2 * 2 * 5 * 64 * 4   # B x ceil(L / 128) tiles x (K + 1) x ED fp32


def test_independent_segment_workspaces_without_gpu():
    """Small B * ED: the chained kernels run independent L-segments; the workspace carries one (B, ED, N) aggregate and one
    (B, ED) sum of delta per segment boundary (size queries assume a 148-SM device when none is present)."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    B, L, ED, N = 2, 1858, 1024, 16                 # the production shape: 13 segments of 144 steps in both directions
    nseg, nblk = 13, ED // 64
    seg = 256 + (nseg - 1) * B * ED * N * 4 + (nseg - 1) * B * ED * 4
    assert lib.gfe_selscan_fwd_workspace_bytes(B, L, ED, N) == seg
    assert lib.gfe_selscan_bwd_workspace_bytes(B, L, ED, N) == seg + nblk * B * L * 32 * 4 + B * nseg * 18 * ED * 4
    # a 128-channel shard of one 65 536-token sequence: the segment count saturates at 256 (255 boundaries)
    assert lib.gfe_selscan_fwd_workspace_bytes(1, 65536, 128, N) == 256 + 255 * 128 * N * 4 + 255 * 128 * 4
    # checkpoints keep the chained layout (every 8 steps) whatever the segment plan
    assert lib.gfe_selscan_ckpt_bytes(B, L, ED, N) == B * ((L + 7) // 8) * ED * N * 4 + B * L * ED * 4


def test_add_rmsnorm_mixed_argument_validation_without_gpu():
    """The two-dtype entry points reject unsupported pairs and widths before any launch."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    fake = ctypes.c_void_p(4096)                     # non-null, 16-byte aligned, never dereferenced on these paths
    eps = ctypes.c_float(1e-5)
    assert lib.gfe_add_rmsnorm_fwd_mixed(fake, None, fake, None, fake, None, 5, 64, eps, _native.GFE_BF16, _native.GFE_F32, None) == -2
    assert b"dtype pair" in lib.gfe_last_error_string()
    assert lib.gfe_add_rmsnorm_fwd_mixed(fake, None, fake, None, fake, None, 5, 66, eps, _native.GFE_F32, _native.GFE_BF16, None) == -1
    assert b"multiple of 4" in lib.gfe_last_error_string()
    assert lib.gfe_add_rmsnorm_fwd_mixed(fake, None, fake, None, fake, None, 0, 64, eps, _native.GFE_F32, _native.GFE_BF16, None) == 0   # no rows: nothing to do
    assert lib.gfe_add_rmsnorm_bwd_mixed(fake, fake, fake, fake, None, fake, None, fake, 5, 64, _native.GFE_F16, _native.GFE_BF16,
                                         fake, 1 << 20, None) == -2


def test_add_mean_pool_mixed_argument_validation_without_gpu():
    """Pooling takes fp32 next to a 16-bit operand in either order; two different 16-bit dtypes are refused before any launch."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    fake = ctypes.c_void_p(4096)
    ws = lib.gfe_add_mean_pool_workspace_bytes(2, 5, 8)
    assert lib.gfe_add_mean_pool_fwd_mixed(fake, fake, fake, 2, 5, 8, _native.GFE_BF16, _native.GFE_F16, fake, ws, None) == -2
    assert b"dtype pair" in lib.gfe_last_error_string()
    assert lib.gfe_mean_pool_bwd_mixed(fake, fake, fake, 2, 5, 8, _native.GFE_F16, _native.GFE_BF16, None) == -2
    assert lib.gfe_mean_pool_bwd_mixed(fake, fake, fake, 2, 5, 8, 7, _native.GFE_F32, None) == -2
    assert lib.gfe_add_mean_pool_fwd_mixed(fake, None, fake, 2, 5, 8, _native.GFE_F32, _native.GFE_BF16, fake, ws - 4, None) == -4


def test_argument_validation_without_gpu():
    """Bad arguments are rejected before any launch, with a message."""
    from gfe_mamba_b200 import _native
    lib = _native.lib()
    a = _native.SelscanArgs()
    assert lib.gfe_selscan_fwd(ctypes.byref(a), None) == -1
    assert b"shape" in lib.gfe_last_error_string()
    a.batch, a.seqlen, a.d_inner, a.d_state = 1, 8, 32, 8
    assert lib.gfe_selscan_fwd(ctypes.byref(a), None) == -3
    assert b"d_state" in lib.gfe_last_error_string()
    assert lib.gfe_pscan_fwd(None, None, None, 1, 1, 1, 1, None, 0, None) == -1
    assert lib.gfe_conv1d_silu_fwd(None, 0, 0, None, None, None, 0, 0, 1, 1, 1, 4, 0, None) == -1


def test_selscan_args_struct_matches_header_field_order():
    from gfe_mamba_b200 import _native
    src = open(os.path.join(ROOT, "include", "gfe_mamba_b200.h")).read()
    start = src.index("typedef struct gfe_selscan_args {") + len("typedef struct gfe_selscan_args {")
    body = src[start:src.index("} gfe_selscan_args;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl or decl.startswith("typedef"):
            continue
        decl = re.sub(r"^(const\s+)?(void|float|int32_t|uint32_t|int64_t|size_t)\s*", "", decl)
        names += [n.strip().lstrip("*") for n in decl.split(",")]
    assert names == [f[0] for f in _native.SelscanArgs._fields_]


def test_config_mirrors_reference():
    from cross_atten.mamba import MambaConfig
    cfg = MambaConfig(d_model=768, n_layers=2)
    assert (cfg.d_inner, cfg.dt_rank, cfg.d_state, cfg.d_conv, cfg.expand_factor) == (1536, 48, 16, 4, 2)
    assert cfg.pscan is True and cfg.use_cuda is False and cfg.bias is False and cfg.conv_bias is True
    fields = [f.name for f in dataclasses.fields(cfg)]
    assert fields == ["d_model", "n_layers", "dt_rank", "d_state", "expand_factor", "d_conv", "dt_min", "dt_max", "dt_init",
                      "dt_scale", "rms_norm_eps", "bias", "conv_bias", "inner_layernorms", "pscan", "use_cuda"]
    assert MambaConfig.dt_init_floor == 1e-4 and "dt_init_floor" not in fields     # class attribute, as in the reference
    assert MambaConfig(d_model=512, n_layers=6, use_cuda=True).use_cuda is True    # mamba_transformer.py:65


def test_state_dict_keys_and_seeded_init_match_reference(golden_dir):
    """Same parameter names/shapes AND the same values under the same seed as the reference (mamba.py:126-168)."""
    from cross_atten.mamba import MambaBlock, MambaConfig
    g = dict(np.load(os.path.join(golden_dir, "block_small.npz")))
    torch.manual_seed(303)                                   # tests/golden/make_golden.py: gen_block
    blk = MambaBlock(MambaConfig(d_model=16, n_layers=1))
    with torch.no_grad():
        blk.A_log.add_(0.1 * torch.randn_like(blk.A_log))
        blk.D.add_(0.1 * torch.randn_like(blk.D))
    sd = blk.state_dict()
    assert sorted(sd) == sorted(k[3:] for k in g if k.startswith("sd."))
    for k, v in sd.items():
        assert np.array_equal(v.numpy(), g["sd." + k]), k
    assert blk.A_log._no_weight_decay and blk.D._no_weight_decay


def test_mamba_state_dict_layout(mamba_cfg1):
    from cross_atten.mamba import Mamba, MambaConfig
    g = mamba_cfg1
    m = Mamba(MambaConfig(d_model=128, n_layers=2, inner_layernorms=False))
    want = {k[3:]: v.shape for k, v in g.items() if k.startswith("sd.")}
    assert {k: tuple(v.shape) for k, v in m.state_dict().items()} == want
    m.load_state_dict({k: torch.from_numpy(g["sd." + k]) for k in want}, strict=True)
    j = Mamba(MambaConfig(d_model=32, n_layers=1, inner_layernorms=True))
    assert {"layers.0.mixer.dt_layernorm.weight", "layers.0.mixer.B_layernorm.weight",
            "layers.0.mixer.C_layernorm.weight"} <= set(j.state_dict())


def test_drop_in_module_names():
    import cross_atten.mamba as m
    import cross_atten.pscan as ps
    for name in ("MambaConfig", "Mamba", "ResidualBlock", "MambaBlock", "RMSNorm", "pscan"):
        assert hasattr(m, name)
    for name in ("pscan", "PScan", "npo2", "pad_npo2"):
        assert hasattr(ps, name)
    assert ps.npo2(1858) == 2048 and ps.npo2(4096) == 4096 and ps.npo2(1) == 1
    assert tuple(ps.pad_npo2(torch.zeros(2, 5, 3, 4)).shape) == (2, 8, 3, 4)
    assert os.path.abspath(m.__file__).startswith(ROOT)


def test_no_cpu_fallback():
    from cross_atten.mamba import Mamba, MambaConfig
    from cross_atten.pscan import pscan
    from gfe_mamba_b200 import causal_conv1d_silu, selective_scan_fn
    m = Mamba(MambaConfig(d_model=16, n_layers=1))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(1, 4, 16))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pscan(torch.rand(1, 4, 2, 2), torch.rand(1, 4, 2, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        causal_conv1d_silu(torch.randn(1, 4, 8), torch.randn(8, 1, 4), None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        selective_scan_fn(torch.randn(1, 4, 32), torch.randn(1, 4, 32), torch.zeros(32, 16), torch.randn(1, 4, 16),
                          torch.randn(1, 4, 16), torch.ones(32))


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under gfe_mamba_b200/ or cross_atten/ may reference it."""
    for pkg in ("gfe_mamba_b200", "cross_atten"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, pkg)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    txt = open(os.path.join(dirpath, f)).read()
                    assert "oracle" not in txt.lower(), os.path.join(dirpath, f)


def test_host_pipeline_chunk_schedule():
    """Row chunks of the host-buffer pipeline: cover the batch exactly, never exceed the device buffers, and keep the
    first copy-in / last copy-out (the only transfers nothing overlaps with) one row long when the batch allows it."""
    from gfe_mamba_b200.host_pipeline import chunk_schedule
    for B in (1, 2, 3, 5, 7, 16, 32, 100, 256):
        for big in (1, 2, 3, 4, 8, 64):
            if big > B:
                continue
            sched = chunk_schedule(B, big)
            assert sum(sched) == B and all(1 <= n <= big for n in sched), (B, big, sched)
            if B >= 8 and big >= 2:
                assert sched[0] == 1 and sched[-1] == 1, (B, big, sched)
    assert chunk_schedule(16, 4) == [1, 1, 2, 4, 4, 2, 1, 1]


def test_host_pipeline_requires_cuda():
    import torch
    from gfe_mamba_b200.host_pipeline import HostScanPipeline
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        HostScanPipeline(2, 8, 32, 16, torch.float32, torch.device("cpu"))


def test_bench_helpers():
    """bench.py's byte accounting (SURVEY 8d) and the traffic lookup keyed by workload and per-GPU batch."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    fwd, bwd = bench.algorithmic_bytes(16, 4096, 1536, 2)
    assert fwd == 16 * 4096 * (4 * 1536 + 2 * 16) * 2 == 809500672
    assert bwd == 16 * 4096 * (7 * 1536 + 4 * 16) * 2 == 1417674752
    t, note = bench.measured_traffic("cfg3", "selscan_bwd", 16)
    assert (t is None and "stale" in note) or t > bwd   # checkpoints, saved y and the dB|dC rows ride on top of the algorithmic bytes
    assert bench.measured_traffic("cfg3", "selscan_bwd", 3)[0] is None and bench.measured_traffic("nope", "selscan_bwd", 16)[0] is None
    # a capture is only quoted for the kernel sources it was taken from
    import json, tempfile
    real_root = bench.ROOT
    with tempfile.TemporaryDirectory() as td:
        os.makedirs(os.path.join(td, "profiles"))
        rec = {"cfgX": {"batch_per_gpu": 4, "kernels": {"selscan_bwd": 123}, "source": "t", "source_hash": "deadbeef"}}
        json.dump(rec, open(os.path.join(td, "profiles", "traffic.json"), "w"))
        bench.ROOT = td
        try:
            assert bench.measured_traffic("cfgX", "selscan_bwd", 4)[0] is None          # hash of an empty tree differs
            rec["cfgX"]["source_hash"] = bench.kernel_source_hash()
            json.dump(rec, open(os.path.join(td, "profiles", "traffic.json"), "w"))
            assert bench.measured_traffic("cfgX", "selscan_bwd", 4) == (123, "t")
        finally:
            bench.ROOT = real_root


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs: float32 files named after the step's outputs, whole when small, the same seeded sample of a large
    output in every run, and the all-reduced sums in place of a rank's own gradients under N GPUs."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    big = torch.arange(bench.DUMP_SAMPLE + 999, dtype=torch.float32)
    grads = [torch.ones(2, 3, dtype=torch.bfloat16) * i for i in range(8)]
    flat = torch.arange(2 * 3 * 3, dtype=torch.float32)
    arrays = bench.step_outputs(big, grads, flat, by_channels=False)
    assert list(arrays) == list(bench.OUTPUT_NAMES)
    assert torch.equal(arrays["dA_log"], flat[:6].view(2, 3)) and torch.equal(arrays["ddt_bias"], flat[12:].view(2, 3))
    assert torch.equal(arrays["dB"], grads[3])
    chan = bench.step_outputs(big, grads, flat[:12], by_channels=True)
    assert torch.equal(chan["dC"], flat[6:12].view(2, 3)) and torch.equal(chan["dD"], grads[6])
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    total = 0
    for name in bench.OUTPUT_NAMES:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b), name
        total += a.nbytes
    out = np.load(tmp_path / "a" / "out.npy")
    assert out.shape == (bench.DUMP_SAMPLE,) and np.all(np.diff(out) > 0)   # sorted distinct indices of a ramp
    assert np.array_equal(np.load(tmp_path / "a" / "dz.npy"), grads[2].float().numpy())
    assert 9 * bench.DUMP_SAMPLE * 4 <= 64e6 and total <= 64e6


def test_numa_binding_is_a_no_op_without_topology():
    import torch
    from gfe_mamba_b200.host_pipeline import bind_host_to_gpu_node
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    before = os.sched_getaffinity(0)
    assert bind_host_to_gpu_node(torch.device("cpu")) is None
    assert os.sched_getaffinity(0) == before
