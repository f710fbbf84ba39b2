"""GPU tests of the stage-1 RGB-sigma network (nerf/network.py:10-207) and its training step (nerf/utils.py:536-632):
fused inference must equal the instance-stage network's sigma / colour bit for bit (same kernels, head switched off),
the modular autograd path must agree with the fused one, and a few optimisation steps must reduce the photometric loss
with finite gradients in every trained tensor (sigma table, sigma-net, colour-net)."""
import pytest
import torch

from helpers import bits_equal, make_rays, scene_arrays
from test_field_gpu import build_model

pytestmark = pytest.mark.gpu


def _stage1_from(m2, cuda):
    from instance_nerf_b200.nerf.network import NeRFNetwork
    m1 = NeRFNetwork(bound=m2.bound, cuda_ray=True, density_scale=m2.density_scale, density_thresh=10)
    sd = {k: v for k, v in m2.state_dict().items() if not (k.startswith("encoder_mask") or k.startswith("mask_net"))}
    m1.load_state_dict(sd)                      # identical key set: stage-1 tensors are a subset of the instance-stage ones
    return m1.to(cuda).eval()


def test_state_dict_keys_match_reference_layout():
    from instance_nerf_b200.nerf.network import NeRFNetwork
    m = NeRFNetwork(bound=8, cuda_ray=True)
    assert list(m.state_dict().keys()) == ["aabb_train", "aabb_infer", "density_grid", "density_bitfield", "step_counter",
                                           "encoder.embeddings", "encoder.offsets", "sigma_net.0.weight", "sigma_net.1.weight",
                                           "color_net.0.weight", "color_net.1.weight", "color_net.2.weight"]
    assert [tuple(l.weight.shape) for l in (*m.sigma_net, *m.color_net)] == [(64, 32), (16, 64), (64, 31), (64, 64), (3, 64)]


def test_fused_inference_equals_instance_stage(cuda):
    m2, sc = build_model(cuda, 32)
    m1 = _stage1_from(m2, cuda)
    g = torch.Generator().manual_seed(1)
    B = 128 * 11 + 9
    x = ((torch.rand(B, 3, generator=g) * 2 - 1) * 7.9).to(cuda)
    d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g), dim=-1).to(cuda)
    with torch.no_grad():
        s1, c1 = m1(x, d)
        s2, c2, _ = m2(x, d)
        assert bits_equal(s1, s2) and bits_equal(c1, c2)
        m1.use_fused = False
        with torch.autocast("cuda", dtype=torch.float16):
            s0, c0 = m1(x, d)
        m1.use_fused = True
    torch.testing.assert_close(s1, s0.float(), rtol=2e-2, atol=1e-3)
    torch.testing.assert_close(c1, c0.float(), rtol=0, atol=2e-3)
    o, dd = make_rays(sc, 48, 64)
    o, dd = o.to(cuda), dd.to(cuda)
    kw = dict(dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4, perturb=False, bg_color=1)
    with torch.no_grad():
        r1 = m1.render(o[None], dd[None], staged=True, **kw)
        r2 = m2.render(o[None], dd[None], staged=True, render_mask=False, **kw)
    assert r1["instance_mask_logits"] is None
    # one-launch renderer: the order in which slots pick up rays is dynamic, per-ray arithmetic is not
    assert bits_equal(r1["image"], r2["image"]) and bits_equal(r1["depth"], r2["depth"])


def test_rgb_train_step_learns(cuda):
    from instance_nerf_b200.nerf.trainer import RGBTrainStep
    m2, sc = build_model(cuda, 4)
    teacher = _stage1_from(m2, cuda)
    o, d = make_rays(sc, 64, 64)
    o, d = o.to(cuda)[None], d.to(cuda)[None]
    with torch.no_grad():
        target = teacher.render(o, d, staged=True, dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4, perturb=False, bg_color=1)["image"]
    student = _stage1_from(m2, cuda)
    with torch.no_grad():   # perturb what is trained: tables and colour head
        student.encoder.embeddings.mul_(0.5)
        student.color_net[2].weight.mul_(0.3)
    ts = RGBTrainStep(student, lr=5e-3, fp16=True)
    data = dict(rays_o=o, rays_d=d, images=target)
    losses = [float(ts.step(data)) for _ in range(30)]
    ts._forward_backward(data)                  # gradients of one more batch, before the optimizer pass clears them (FusedAdam)
    for p in (student.encoder.embeddings, *[l.weight for l in (*student.sigma_net, *student.color_net)]):
        assert p.grad is not None and torch.isfinite(p.grad).all() and float(p.grad.abs().sum()) > 0
    ts._optimizer_step()
    assert losses[-1] < 0.5 * losses[0], losses
    # RGBA target with an explicit per-pixel background (utils.py:563-571)
    rgba = torch.cat([target, torch.full_like(target[..., :1], 0.75)], -1)
    out = ts.train_step(dict(rays_o=o, rays_d=d, images=rgba, bg_color=torch.rand_like(target)))
    assert out[0].shape == target.shape and torch.isfinite(out[2])


def _rel(a, b):
    return float((a - b).norm() / b.norm().clamp(min=1e-12))


@pytest.mark.parametrize("B,bound", [(128 * 9 + 17, 8.0), (128 * 2, 8.0), (77, 8.0), (128 * 9 + 17, 2.0)], ids=["1169", "256", "77", "1169-bound2"])
def test_fused_rgb_backward_matches_autograd(cuda, B, bound):
    """inerf_field_forward_train_rgb + inerf_field_backward_rgb (tcgen05) against the reference operator sequence through
    autograd (network.py:96-127: grid-encode kernels + nn.Linear + sigmoid / trunc_exp), under fp16 autocast and in fp32:
    the fused gradients of the sigma table and the five weight matrices must be at least as close to the fp32 run as the
    autocast run is (fp32 accumulators where autocast rounds GEMM outputs and table atomics to fp16)."""
    m2, _ = build_model(cuda, 4, bound=bound)
    m = _stage1_from(m2, cuda)
    m.train()
    g = torch.Generator().manual_seed(3)
    x = ((torch.rand(B, 3, generator=g) * 2 - 1) * 7.5 * bound / 8).to(cuda)
    x[:3] = torch.tensor([[8.5, 0.0, 0.0], [0.0, -9.0, 1.0], [1.0, 2.0, 8.01]], device=cuda) * (bound / 8)   # outside the grid: zero features, no table gradient
    d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g), dim=-1).to(cuda)
    Gs = (torch.randn(B, generator=g) * 0.3).to(cuda)
    Gc = torch.randn(B, 3, generator=g).to(cuda)
    params = [m.encoder.embeddings, *[l.weight for l in (*m.sigma_net, *m.color_net)]]

    def grads(use_fused, autocast):
        for p in params:
            p.grad = None
        m.use_fused = use_fused
        with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
            assert m.fused_train_available(x, d) == (use_fused and autocast)
            s, c = m(x, d)
            loss = (s.float() * Gs).sum() + (c.float() * Gc).sum()
        loss.backward()
        m.use_fused = True
        return [p.grad.detach().float().clone() for p in params], (s.detach().float(), c.detach().float())

    g_fused, out_fused = grads(True, True)
    g_amp, out_amp = grads(False, True)
    g_fp32, _ = grads(False, False)
    torch.testing.assert_close(out_fused[0], out_amp[0], rtol=2e-2, atol=1e-3)
    torch.testing.assert_close(out_fused[1], out_amp[1], rtol=0, atol=2e-3)
    names = ["table", "sigma0", "sigma1", "color0", "color1", "color2"]
    for n, a, b, c in zip(names, g_fused, g_amp, g_fp32):
        assert a.shape == c.shape and torch.isfinite(a).all()
        e_fused, e_amp = _rel(a, c), _rel(b, c)
        assert e_fused < max(2e-2, 1.5 * e_amp), f"{n}: fused vs fp32 {e_fused:.3e}, autocast vs fp32 {e_amp:.3e}"
    nz_f, nz_r = g_fused[0].abs().sum(1) > 0, g_fp32[0].abs().sum(1) > 0
    assert float((nz_f ^ nz_r).float().mean()) < 1e-3


def test_rgb_train_step_fused_equals_modular_first_steps(cuda):
    """RGBTrainStep on the fused path and on the op-level / cuBLAS path from the same initial state and the same injected ray
    jitter: same loss at step 0 (forward parity) and the same loss trajectory within fp16 noise after a few Adam steps."""
    from instance_nerf_b200.nerf.trainer import RGBTrainStep
    m2, sc = build_model(cuda, 4)
    teacher = _stage1_from(m2, cuda)
    o, d = make_rays(sc, 64, 64)
    o, d = o.to(cuda)[None], d.to(cuda)[None]
    with torch.no_grad():
        target = teacher.render(o, d, staged=True, dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4, perturb=False, bg_color=1)["image"]
    noises = torch.rand(o.shape[1], generator=torch.Generator().manual_seed(4)).to(cuda)
    traj = {}
    for fused in (True, False):
        student = _stage1_from(m2, cuda)
        with torch.no_grad():
            student.encoder.embeddings.mul_(0.5)
            student.color_net[2].weight.mul_(0.3)
        student.use_fused = fused
        ts = RGBTrainStep(student, lr=2e-3, fp16=True)
        traj[fused] = [float(ts.step(dict(rays_o=o, rays_d=d, images=target, noises=noises))) for _ in range(8)]
    a, b = traj[True], traj[False]
    assert abs(a[0] - b[0]) < 2e-3 * abs(b[0]), (a, b)                    # same forward
    for i in range(1, 5):                                                  # same first Adam steps (fp16 noise compounds after that)
        assert abs(a[i] - b[i]) < 5e-2 * abs(b[i]), (i, a, b)
    assert a[-1] < 0.6 * a[0] and b[-1] < 0.6 * b[0], (a, b)
