import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:  # pragma: no cover
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def mamba_cfg1(golden_dir):
    """tests/golden/mamba_cfg1.npz with the reference's seeded tensors restored.

    The file keeps the reference's outputs whole and, of the tensors it drew from one seed (state dict, x, dy), the shape
    and every ``sample_stride``-th value.  They are drawn again here with the drop-in under the same seed and must match
    those samples: the drop-in creates its parameters in the reference's order with the reference's initialisation."""
    import numpy as np
    import torch
    from cross_atten.mamba import Mamba, MambaConfig
    g = dict(np.load(os.path.join(golden_dir, "mamba_cfg1.npz")))
    d_model, n_layers, B, L = (int(g["meta"][i]) for i in (0, 1, 6, 7))
    torch.manual_seed(int(g.pop("seed")))
    model = Mamba(MambaConfig(d_model=d_model, n_layers=n_layers))
    drawn = {f"sd.{k}": v.numpy().copy() for k, v in model.state_dict().items()}
    drawn["x"] = torch.randn(B, L, d_model).numpy()
    drawn["dy"] = torch.randn(B, L, d_model).numpy()
    assert sorted(drawn) == sorted(k[len("shape."):] for k in g if k.startswith("shape."))
    stride = int(g.pop("sample_stride"))
    for k, v in drawn.items():
        assert v.shape == tuple(g.pop(f"shape.{k}")), k
        want = g.pop(f"sample.{k}")
        assert np.abs(v.reshape(-1)[::stride] - want).max() <= 1e-6 * max(np.abs(want).max(), 1e-30), k
        g[k] = v
    return g
