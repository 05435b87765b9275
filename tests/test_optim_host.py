"""Host logic of the multi-tensor optimiser (no GPU): the chunk table that describes a parameter list to the kernels."""
import pytest
import torch


def test_chunk_plan_covers_every_element_once():
    from gfe_mamba_b200.optim import ClipAdam
    numels = [1, 4096, 4097, 10000, 3]
    ct, cs, tc0 = ClipAdam.plan_chunks(numels, 4096)
    assert tc0 == [0, 1, 2, 4, 7, 8] and len(ct) == len(cs) == 8
    for t, n in enumerate(numels):
        starts = [s for tt, s in zip(ct, cs) if tt == t]
        assert starts == list(range(0, n, 4096))
        assert ct[tc0[t]:tc0[t + 1]] == [t] * (tc0[t + 1] - tc0[t])


def test_clip_adam_rejects_cpu_parameters():
    from gfe_mamba_b200.optim import ClipAdam
    p = torch.nn.Parameter(torch.ones(4))
    p.grad = torch.ones(4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ClipAdam([p], lr=1e-3).step()
    with pytest.raises(ValueError):
        ClipAdam([p], lr=-1.0)


def _adam_state(steps, weight_decay=0.0):
    ps = [torch.nn.Parameter(torch.randn(5, 3)), torch.nn.Parameter(torch.randn(7))]
    opt = torch.optim.Adam(ps, lr=1e-2, weight_decay=weight_decay)
    for _ in range(steps):
        for p in ps:
            p.grad = torch.randn_like(p)
        opt.step()
    return ps, opt.state_dict()


def test_clip_adam_state_dict_in_adam_format_without_gpu():
    """A torch.optim.Adam state dict loads (moments and step), and state_dict() gives it back in Adam's format: a float32
    CPU ``step`` per parameter, ``weight_decay`` 0 per group; ClipAdam's own settings come from its constructor."""
    from gfe_mamba_b200.optim import ClipAdam
    ps, sd = _adam_state(3)
    opt = ClipAdam([torch.nn.Parameter(p.detach().clone()) for p in ps], lr=1e-2, max_norm=None)
    opt.load_state_dict(sd)
    assert all("step" not in st for st in opt.state.values())   # the step counter is the group's, not per tensor
    g = opt.param_groups[0]
    assert g["max_norm"] is None and g["per_parameter_clip"] is True and g["zero_grad"] is False
    out = opt.state_dict()
    assert out["param_groups"][0]["weight_decay"] == 0.0
    for i in (0, 1):
        st = out["state"][i]
        assert st["step"].dtype == torch.float32 and st["step"].device.type == "cpu" and float(st["step"]) == 3.0
        assert torch.equal(st["exp_avg"], sd["state"][i]["exp_avg"]) and torch.equal(st["exp_avg_sq"], sd["state"][i]["exp_avg_sq"])
    back = torch.optim.Adam([torch.nn.Parameter(p.detach().clone()) for p in ps], lr=1e-2)
    back.load_state_dict(out)                                    # and torch.optim.Adam takes it back
    assert float(back.state_dict()["state"][0]["step"]) == 3.0


def test_clip_adam_refuses_state_it_cannot_continue_without_gpu():
    from gfe_mamba_b200.optim import ClipAdam
    ps, sd = _adam_state(2)
    opt = ClipAdam([torch.nn.Parameter(p.detach().clone()) for p in ps], lr=1e-2)
    sd["state"][1]["step"] = torch.tensor(5.0)
    with pytest.raises(ValueError, match="step"):                 # one device step counter per group
        opt.load_state_dict(sd)
    _, sd_wd = _adam_state(1, weight_decay=0.1)
    with pytest.raises(ValueError, match="weight decay"):
        opt.load_state_dict(sd_wd)
