"""The reference's own callers of the path, built on the drop-in (CPU; needs GFE_REFERENCE, a checkout of the original
GFE-Mamba, whose caller modules are not part of this repository): cross_atten/mamba_transformer.py:65-66
(Cross_mamba_both -> Mamba(MambaConfig(use_cuda=True))) and
cross_atten/jamba.py:9,406 (MambaLayer -> MambaBlock(inner_layernorms=True), RMSNorm).  With this repository ahead of the
reference on sys.path, `cross_atten.mamba` / `cross_atten.pscan` resolve here and every other module of the namespace
package to the reference; the models must come out with the same parameter names and shapes as on the reference alone
(their checkpoints load strictly either way)."""
import json
import os
import subprocess
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("GFE_REFERENCE", "")

PROBE = r"""
import json, sys
import torch
import cross_atten.mamba as m, cross_atten.mamba_transformer as mt, cross_atten.jamba as jb
torch.manual_seed(0)
model = mt.Cross_mamba_both(categories=(3, 4, 5), num_continuous=6, dim=32, depth=2, heads=2)
cfg = jb.JambaLMConfig(d_model=32, n_layers=2, mlp_size=64, num_attention_heads=2, num_key_value_heads=1, num_experts=1)
layer = jb.MambaLayer(cfg, num_experts=1)
out = dict(mamba_file=m.__file__, transformer_file=mt.__file__, jamba_file=jb.__file__,
           mamba_module=type(model.transformer).__module__, block_module=type(layer.mamba).__module__,
           rmsnorm_module=type(layer.input_layernorm).__module__, use_cuda=bool(model.transformer.config.use_cuda),
           inner_layernorms=bool(layer.mamba.config.inner_layernorms),
           cross=[(k, list(v.shape)) for k, v in model.state_dict().items()],
           jamba=[(k, list(v.shape)) for k, v in layer.state_dict().items()],
           a_log_sum=float(model.transformer.layers[0].mixer.A_log.sum()),
           dt_bias_sum=float(model.transformer.layers[1].mixer.dt_proj.bias.sum()))
print("PROBE" + json.dumps(out))
"""


def _probe(pythonpath):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join(pythonpath))
    r = subprocess.run([sys.executable, "-c", PROBE], capture_output=True, text=True, cwd=tempfile.gettempdir(), env=env,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = next(l for l in r.stdout.splitlines() if l.startswith("PROBE"))
    return json.loads(line[5:])


@pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "cross_atten")),
                    reason="GFE_REFERENCE does not name a checkout of the original GFE-Mamba")
def test_reference_callers_build_on_the_drop_in():
    ours = _probe([ROOT, REF])
    ref = _probe([REF])
    # the seam: only mamba.py / pscan.py come from this repository
    assert ours["mamba_file"].startswith(ROOT) and ours["transformer_file"].startswith(REF) and ours["jamba_file"].startswith(REF)
    assert ours["mamba_module"] == ours["block_module"] == ours["rmsnorm_module"] == "gfe_mamba_b200.mamba"
    assert ref["mamba_file"].startswith(REF) and ref["mamba_module"] == "cross_atten.mamba"
    # mamba_transformer.py:65 passes use_cuda=True: accepted here as it is; the reference flips it off (no mamba_ssm, mamba.py:186)
    assert ours["use_cuda"] is True and ours["inner_layernorms"] is True
    # same parameter names, order and shapes: strict load_state_dict works in both directions
    assert ours["cross"] == ref["cross"]
    assert ours["jamba"] == ref["jamba"]
    # same draws from the same seed (initialisation order is the reference's)
    assert abs(ours["a_log_sum"] - ref["a_log_sum"]) < 1e-4 and abs(ours["dt_bias_sum"] - ref["dt_bias_sum"]) < 1e-4
