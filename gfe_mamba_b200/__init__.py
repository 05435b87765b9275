"""gfe_mamba_b200 -- B200 (sm_100a) selective-scan hot path behind GFE-Mamba's Python API.

    from gfe_mamba_b200 import Mamba, MambaConfig, MambaBlock, pscan

or, as a drop-in for the reference's module names, put this repository ahead of the reference on
``sys.path`` and keep ``from cross_atten.mamba import Mamba, MambaConfig`` unchanged.
"""
from .mamba import Mamba, MambaBlock, MambaConfig, ResidualBlock, RMSNorm  # noqa: F401
from .ops import (add_mean_pool, add_rmsnorm, causal_conv1d_silu, causal_conv1d_silu_state, conv1d_prefill,  # noqa: F401
                  conv1d_step, mamba_inner_fn, selective_scan_fn, selective_scan_state, ssm_prefill, ssm_step)
from .optim import ClipAdam  # noqa: F401
from .pscan import PScan, npo2, pad_npo2, pscan  # noqa: F401

__version__ = "0.1.0"
