"""ctypes binding of the C ABI in include/gfe_mamba_b200.h.

There is deliberately no fallback: if the shared library is missing or a call fails this module raises.
"""
from __future__ import annotations

import ctypes
import os
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
# GFE_LIB_VARIANT=<tag> loads lib/libgfe_mamba_b200.<tag>.so (A/B builds of the same sources, `build.py --tag=`); it
# must exist -- there is no fallback either way.
_VARIANT = os.environ.get("GFE_LIB_VARIANT", "")
LIB_PATH = os.path.join(_PKG, "lib", f"libgfe_mamba_b200.{_VARIANT}.so" if _VARIANT else "libgfe_mamba_b200.so")

GFE_F32, GFE_BF16, GFE_F16 = 0, 1, 2
GFE_FLAG_DELTA_SOFTPLUS = 1

c_i32, c_i64, c_u32, c_sz, c_vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_size_t, ctypes.c_void_p


class SelscanArgs(ctypes.Structure):
    """Mirror of ``struct gfe_selscan_args`` (field order is ABI)."""

    _fields_ = [
        ("batch", c_i32), ("seqlen", c_i32), ("d_inner", c_i32), ("d_state", c_i32),
        ("dtype", c_i32), ("flags", c_u32),
        ("u", c_vp), ("u_bs", c_i64), ("u_rs", c_i64),
        ("delta", c_vp), ("delta_bs", c_i64), ("delta_rs", c_i64),
        ("z", c_vp), ("z_bs", c_i64), ("z_rs", c_i64),
        ("Bm", c_vp), ("B_bs", c_i64), ("B_rs", c_i64),
        ("Cm", c_vp), ("C_bs", c_i64), ("C_rs", c_i64),
        ("A_log", c_vp), ("D", c_vp), ("dt_bias", c_vp),
        ("out", c_vp), ("out_bs", c_i64), ("out_rs", c_i64),
        ("last_state", c_vp),
        ("ckpt", c_vp), ("ckpt_bytes", c_sz),
        ("ws", c_vp), ("ws_bytes", c_sz),
        ("dout", c_vp), ("dout_bs", c_i64), ("dout_rs", c_i64),
        ("du", c_vp), ("du_bs", c_i64), ("du_rs", c_i64),
        ("ddelta", c_vp), ("ddelta_bs", c_i64), ("ddelta_rs", c_i64),
        ("dz", c_vp), ("dz_bs", c_i64), ("dz_rs", c_i64),
        ("dBm", c_vp), ("dB_bs", c_i64), ("dB_rs", c_i64),
        ("dCm", c_vp), ("dC_bs", c_i64), ("dC_rs", c_i64),
        ("dA_log", c_vp), ("dD", c_vp), ("ddt_bias", c_vp),
    ]


# name -> (restype, argtypes); every symbol include/gfe_mamba_b200.h declares
SIGNATURES = {
    "gfe_version": (ctypes.c_int, []),
    "gfe_last_error_string": (ctypes.c_char_p, []),
    "gfe_pscan_workspace_bytes": (c_sz, [ctypes.c_int] * 4),
    "gfe_pscan_fwd": (ctypes.c_int, [c_vp, c_vp, c_vp] + [ctypes.c_int] * 4 + [c_vp, c_sz, c_vp]),
    "gfe_pscan_bwd": (ctypes.c_int, [c_vp] * 5 + [ctypes.c_int] * 4 + [c_vp, c_sz, c_vp]),
    "gfe_selscan_ckpt_bytes": (c_sz, [ctypes.c_int] * 4),
    "gfe_selscan_ckpt_bytes_dt": (c_sz, [ctypes.c_int] * 5),
    "gfe_selscan_fwd_workspace_bytes": (c_sz, [ctypes.c_int] * 4),
    "gfe_selscan_bwd_workspace_bytes": (c_sz, [ctypes.c_int] * 4),
    "gfe_selscan_fwd": (ctypes.c_int, [ctypes.POINTER(SelscanArgs), c_vp]),
    "gfe_selscan_bwd": (ctypes.c_int, [ctypes.POINTER(SelscanArgs), c_vp]),
    "gfe_selscan_fwd_state": (ctypes.c_int, [ctypes.POINTER(SelscanArgs), c_vp, c_vp]),
    "gfe_conv1d_silu_fwd": (ctypes.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64] + [ctypes.c_int] * 5 + [c_vp]),
    "gfe_conv1d_silu_fwd_state": (ctypes.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64]
                                  + [ctypes.c_int] * 5 + [c_vp]),
    "gfe_conv1d_bwd_workspace_bytes": (c_sz, [ctypes.c_int] * 4),
    "gfe_conv1d_silu_bwd": (ctypes.c_int, [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_i64, c_vp, c_vp]
                            + [ctypes.c_int] * 5 + [c_vp, c_sz, c_vp]),
    "gfe_conv1d_step": (ctypes.c_int, [c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64] + [ctypes.c_int] * 4 + [c_vp]),
    "gfe_ssm_step": (ctypes.c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp,
                                    c_vp, c_i64, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_u32, ctypes.c_int, c_vp]),
    "gfe_add_rmsnorm_fwd": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, ctypes.c_int, ctypes.c_float, ctypes.c_int, c_vp]),
    "gfe_add_rmsnorm_bwd_workspace_bytes": (c_sz, [c_i64, ctypes.c_int]),
    "gfe_add_rmsnorm_bwd": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, ctypes.c_int, ctypes.c_int, c_vp, c_sz, c_vp]),
    "gfe_add_rmsnorm_fwd_mixed": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, ctypes.c_int, ctypes.c_float, ctypes.c_int, ctypes.c_int, c_vp]),
    "gfe_add_rmsnorm_bwd_mixed": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, ctypes.c_int, ctypes.c_int, ctypes.c_int, c_vp, c_sz, c_vp]),
    "gfe_add_mean_pool_workspace_bytes": (c_sz, [ctypes.c_int] * 3),
    "gfe_add_mean_pool_fwd": (ctypes.c_int, [c_vp, c_vp, c_vp] + [ctypes.c_int] * 4 + [c_vp, c_sz, c_vp]),
    "gfe_mean_pool_bwd": (ctypes.c_int, [c_vp, c_vp] + [ctypes.c_int] * 4 + [c_vp]),
    "gfe_add_mean_pool_fwd_mixed": (ctypes.c_int, [c_vp, c_vp, c_vp] + [ctypes.c_int] * 5 + [c_vp, c_sz, c_vp]),
    "gfe_mean_pool_bwd_mixed": (ctypes.c_int, [c_vp, c_vp, c_vp] + [ctypes.c_int] * 5 + [c_vp]),
    "gfe_clip_adam_chunk_elems": (ctypes.c_int, []),
    "gfe_clip_adam_step": (ctypes.c_int, [c_vp] * 11 + [ctypes.c_int] * 2 + [ctypes.c_float] * 5 + [ctypes.c_int] * 2 + [c_vp]),
    "gfe_timing_enable": (ctypes.c_int, [ctypes.c_int]),
    "gfe_timing_kernel_count": (ctypes.c_int, []),
    "gfe_timing_kernel_name": (ctypes.c_char_p, [ctypes.c_int]),
    "gfe_timing_collect": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64), ctypes.c_int]),
}

_lib = None
_lock = threading.Lock()


def lib() -> ctypes.CDLL:
    """Load libgfe_mamba_b200.so (once).  Raises if it has not been built -- there is no other path."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"gfe_mamba_b200: CUDA library {LIB_PATH} not found. Build it with "
                        "`python -m gfe_mamba_b200.build` (needs nvcc). There is no CPU or PyTorch fallback.")
                l = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(l, name)   # AttributeError if the library does not export the symbol
                    fn.restype, fn.argtypes = res, args
                _lib = l
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().gfe_last_error_string()
        raise RuntimeError(f"gfe_mamba_b200.{what} failed (status {rc}): {msg.decode() if msg else ''}")


def timing_enable(on: bool) -> None:
    lib().gfe_timing_enable(1 if on else 0)


def timing_collect() -> dict:
    """{kernel name: (total_ms, launches)} since the last collect; synchronises the recorded events."""
    l = lib()
    n = l.gfe_timing_kernel_count()
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_int64 * n)()
    check(l.gfe_timing_collect(ms, cnt, n), "timing_collect")
    return {l.gfe_timing_kernel_name(i).decode(): (ms[i], cnt[i]) for i in range(n) if cnt[i] > 0}
