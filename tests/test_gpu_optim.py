"""GPU parity of the multi-tensor clip + Adam step (csrc/optim.cu) against the reference training loop's own calls:
per-parameter torch.nn.utils.clip_grad_norm_ followed by torch.optim.Adam.step (classify_mamba.py:104-109)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _params(seed, shapes, scale):
    g = torch.Generator(device="cuda").manual_seed(seed)
    ps = [torch.nn.Parameter(torch.randn(s, device="cuda", generator=g)) for s in shapes]
    gs = [[torch.randn(s, device="cuda", generator=g) * sc for s, sc in zip(shapes, scale)] for _ in range(4)]
    return ps, gs


@pytest.mark.parametrize("per_param", [True, False])
@pytest.mark.parametrize("max_norm", [1.0, None])
def test_clip_adam_matches_torch(per_param, max_norm):
    from gfe_mamba_b200.optim import ClipAdam
    shapes = [(1024, 16), (1024,), (2048, 512), (1024, 1, 4), (7,), (48 + 32, 1024), (4097,), (3, 5, 7),
              (0,), (1,), (33,), (5, 3), (8193,), (64, 64), (2,), (130, 3), (4096,)]
    scale = [10.0, 1e-3, 1.0, 0.1, 5.0, 1e-2, 1.0, 100.0,   # some tensors clipped hard, some not at all
             1.0, 50.0, 1e-4, 2.0, 0.5, 30.0, 1.0, 1e-2, 3.0]
    # the per-tensor coef kernel runs one warp per tensor, 8 per CTA: 17 tensors need 3 CTAs (an empty one and a
    # one-element one among them)
    assert len(shapes) == len(scale) and -(-len(shapes) // 8) == 3
    ours, grads = _params(3, shapes, scale)
    ref = [torch.nn.Parameter(p.detach().clone()) for p in ours]
    opt_ref = torch.optim.Adam(ref, lr=1e-2)
    opt = ClipAdam(ours, lr=1e-2, max_norm=max_norm, per_parameter_clip=per_param, zero_grad=False)
    for step in range(4):
        for p, q, g in zip(ours, ref, grads[step]):
            p.grad = g.clone()
            q.grad = g.clone()
        if max_norm is not None:
            if per_param:
                for q in ref:   # the reference's loop, classify_mamba.py:106-107
                    torch.nn.utils.clip_grad_norm_(q, max_norm=max_norm)
            else:
                torch.nn.utils.clip_grad_norm_(ref, max_norm=max_norm)
        opt_ref.step()
        opt.step()
        torch.cuda.synchronize()
        for p, q in zip(ours, ref):
            assert torch.allclose(p, q, rtol=2e-6, atol=2e-7), (step, p.shape, (p - q).abs().max().item())
            assert torch.allclose(p.grad, q.grad, rtol=1e-5, atol=1e-8), "clipped gradients differ"
    st = opt.state[ours[2]]
    assert torch.allclose(st["exp_avg"], opt_ref.state[ref[2]]["exp_avg"], rtol=1e-5, atol=1e-6)   # lerp vs fma rounding near zero
    assert torch.allclose(st["exp_avg_sq"], opt_ref.state[ref[2]]["exp_avg_sq"], rtol=1e-4, atol=1e-8)


def test_clip_adam_zero_grad_and_graph_capture():
    """zero_grad=True leaves the gradients zeroed in place (fixed addresses); a captured step replays with the right bias
    corrections because the step counter lives on the device."""
    from gfe_mamba_b200.optim import ClipAdam
    shapes = [(300, 16), (300,), (64, 300)]
    ours, grads = _params(5, shapes, [1.0, 1.0, 1.0])
    ref = [torch.nn.Parameter(p.detach().clone()) for p in ours]
    opt_ref = torch.optim.Adam(ref, lr=1e-3)
    opt = ClipAdam(ours, lr=1e-3, max_norm=1.0, zero_grad=True)
    static_g = [torch.zeros_like(p) for p in ours]
    for p, g in zip(ours, static_g):
        p.grad = g
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):   # warm-up outside the capture (builds the tables)
        for g, src in zip(static_g, grads[0]):
            g.copy_(src)
        opt.step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        opt.step()
    for q, src in zip(ref, grads[0]):
        q.grad = src.clone()
    for q in ref:
        torch.nn.utils.clip_grad_norm_(q, max_norm=1.0)
    opt_ref.step()
    for step in range(1, 4):
        for g, src in zip(static_g, grads[step]):
            assert float(g.abs().max()) == 0.0, "gradients were not zeroed by the previous step"
            g.copy_(src)
        graph.replay()
        for q, src in zip(ref, grads[step]):
            q.grad = src.clone()
        for q in ref:
            torch.nn.utils.clip_grad_norm_(q, max_norm=1.0)
        opt_ref.step()
    torch.cuda.synchronize()
    for p, q in zip(ours, ref):
        assert torch.allclose(p, q, rtol=2e-6, atol=2e-7), (p - q).abs().max().item()


# ------------------------------------------------------------------------------------------- head pooling (SURVEY 8f rank 4)
@pytest.mark.parametrize("B,L,D,dtype,with_r", [(2, 1858, 512, torch.float32, True), (3, 65, 96, torch.float32, False),
                                                (4, 1000, 768, torch.bfloat16, True)])
def test_add_mean_pool_vs_torch(B, L, D, dtype, with_r):
    """mean over L of (a + r): the stack's last residual add fused with mamba_transformer.py:123, forward and backward."""
    from gfe_mamba_b200 import add_mean_pool
    g = torch.Generator(device="cuda").manual_seed(B * L)
    a = torch.randn(B, L, D, device="cuda", generator=g).to(dtype).requires_grad_()
    r = torch.randn(B, L, D, device="cuda", generator=g).to(dtype).requires_grad_() if with_r else None
    dout = torch.randn(B, 1, D, device="cuda", generator=g).to(dtype)
    out = add_mean_pool(a, r)
    out.backward(dout)
    a64 = a.detach().double().requires_grad_()
    r64 = r.detach().double().requires_grad_() if with_r else None
    ref = torch.mean(a64 + r64 if with_r else a64, dim=1, keepdim=True)
    ref.backward(dout.double())
    tol = 1e-6 if dtype == torch.float32 else 1e-2
    assert out.shape == (B, 1, D) and out.dtype == dtype
    assert float((out.double() - ref).abs().max() / ref.abs().max()) < tol
    assert float((a.grad.double() - a64.grad).abs().max() / a64.grad.abs().max()) < tol
    if with_r:
        assert float((r.grad.double() - r64.grad).abs().max() / r64.grad.abs().max()) < tol


def test_mamba_forward_mean_matches_forward_then_mean():
    from gfe_mamba_b200 import Mamba, MambaConfig
    torch.manual_seed(4)
    model = Mamba(MambaConfig(d_model=64, n_layers=2)).cuda()
    x = torch.randn(2, 77, 64, device="cuda")
    x1, x2 = x.clone().requires_grad_(), x.clone().requires_grad_()
    y1 = torch.mean(model(x1), dim=1, keepdim=True)
    y1.square().sum().backward()
    g1 = [p.grad.clone() for p in model.parameters()]
    model.zero_grad()
    y2 = model.forward_mean(x2)
    y2.square().sum().backward()
    assert torch.allclose(y1, y2, rtol=1e-5, atol=1e-6)
    assert torch.allclose(x1.grad, x2.grad, rtol=1e-4, atol=1e-6)
    for a, p in zip(g1, model.parameters()):
        assert torch.allclose(a, p.grad, rtol=1e-4, atol=1e-6)


# -------------------------------------------------------------------------------------- whole training step, eager vs graph
def test_graphed_train_step_matches_eager():
    """GraphedTrainStep replays forward + backward + ClipAdam from one CUDA graph: same parameters as the eager steps."""
    from gfe_mamba_b200 import ClipAdam, Mamba, MambaConfig
    from gfe_mamba_b200.train import GraphedTrainStep, TrainStep
    xs = [torch.randn(2, 130, 64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(i)) for i in range(5)]

    def build():
        torch.manual_seed(7)
        m = Mamba(MambaConfig(d_model=64, n_layers=2)).cuda()
        return m, TrainStep(m, ClipAdam(m.parameters(), lr=1e-3, max_norm=1.0, zero_grad=True))

    m1, s1 = build()
    m2, s2 = build()
    for _ in range(3):                         # GraphedTrainStep warms up with 3 eager steps on its example input (they build
        s1(xs[0])                              # the optimiser tables and the launch caches OUTSIDE the capture): same here
    g = GraphedTrainStep(s2, xs[0], warmup=3)
    losses1 = [float(s1(x)) for x in xs]
    losses2 = [float(g(x)) for x in xs]
    torch.cuda.synchronize()
    assert all(abs(a - b) <= 1e-5 * max(1.0, abs(a)) for a, b in zip(losses1, losses2)), (losses1, losses2)
    for p, q in zip(m1.parameters(), m2.parameters()):
        assert torch.allclose(p, q, rtol=1e-4, atol=1e-6)
