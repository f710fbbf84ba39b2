"""GPU parity of the fused instance-stage training path (inerf_field_forward_train + inerf_field_backward_mask, tcgen05)
against the reference operator sequence (network_mask.py:119-158 through autograd: grid-encode kernels + nn.Linear), and an
end-to-end training step (MaskTrainer.train_step semantics, nerf/utils.py:1287-1373)."""
import numpy as np
import pytest
import torch

from helpers import scene_arrays
from test_field_gpu import build_model

pytestmark = pytest.mark.gpu


def _freeze(m):
    for mod in (m.encoder, m.sigma_net, m.encoder_dir, m.color_net):
        mod.requires_grad_(False)


def _rel(a, b):
    return float((a - b).norm() / b.norm().clamp(min=1e-12))


@pytest.mark.parametrize("K,B,bound", [(32, 128 * 9 + 17, 8.0), (16, 128 * 3, 8.0), (5, 77, 8.0), (32, 128 * 9 + 17, 2.0)],
                         ids=["32-1169", "16-384", "5-77", "32-1169-bound2"])
def test_fused_backward_matches_autograd(cuda, K, B, bound):
    m, _ = build_model(cuda, K, bound=bound)
    m.train()
    _freeze(m)
    g = torch.Generator().manual_seed(3)
    x = ((torch.rand(B, 3, generator=g) * 2 - 1) * 7.5 * bound / 8).to(cuda)
    d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g), dim=-1).to(cuda)
    G = torch.randn(B, K, generator=g).to(cuda)
    params = [m.encoder_mask.embeddings, *[l.weight for l in m.mask_net]]

    def grads(use_fused, autocast):
        for p in params:
            p.grad = None
        m.use_fused = use_fused
        with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
            assert m.fused_train_available(x, d) == (use_fused and autocast)
            s, c, k = m(x, d)
            loss = (k.float() * G).sum()
        loss.backward()
        m.use_fused = True
        return [p.grad.detach().float().clone() for p in params], (s.detach().float(), c.detach().float(), k.detach().float())

    g_fused, out_fused = grads(True, True)
    g_amp, out_amp = grads(False, True)       # the reference's fp16 autocast sequence (fp16 GEMM outputs, fp16 table atomics)
    g_fp32, _ = grads(False, False)           # fp32 reference of the same op sequence
    torch.testing.assert_close(out_fused[2], out_amp[2], rtol=2e-2, atol=2e-2)
    names = ["table", "w0", "w1", "w2"]
    for n, a, b, c in zip(names, g_fused, g_amp, g_fp32):
        e_fused, e_amp = _rel(a, c), _rel(b, c)
        # the fused path keeps fp32 accumulators where autocast rounds to fp16: it must be at least as close to fp32 as autocast is
        assert e_fused < max(2e-2, 1.5 * e_amp), f"{n}: fused vs fp32 {e_fused:.3e}, autocast vs fp32 {e_amp:.3e}"
    # table gradient support is identical (same corners touched)
    nz_f, nz_r = g_fused[0].abs().sum(1) > 0, g_fp32[0].abs().sum(1) > 0
    assert float((nz_f ^ nz_r).float().mean()) < 1e-3


def test_train_step_runs_fused_and_learns(cuda):
    from instance_nerf_b200 import synthetic
    from oracle import host_oracle
    from instance_nerf_b200.nerf.trainer import MaskTrainStep
    K = 16
    m, sc = build_model(cuda, K, density_scale=10.0)
    H, W = 96, 128
    poses = torch.from_numpy(synthetic.camera_poses(sc, 1, 1))
    r = host_oracle.get_rays(poses, synthetic.intrinsics(H, W), H, W, N=1024, patch_size=8, generator=torch.Generator().manual_seed(0))
    o, d = r["rays_o"].reshape(-1, 3).contiguous(), r["rays_d"].reshape(-1, 3).contiguous()
    labels = torch.from_numpy(sc.first_hit_labels(o.numpy().astype(np.float64), d.numpy().astype(np.float64)))
    data = {"rays_o": o[None].to(cuda), "rays_d": d[None].to(cuda), "masks": labels[None].to(cuda),
            "noises": torch.rand(o.shape[0], generator=torch.Generator().manual_seed(1)).to(cuda)}
    tr = MaskTrainStep(m, lr=1e-2, fp16=True, label_regularization_weight=0.1)
    # first-step loss: fused vs modular forward on identical weights
    m.train()
    with torch.no_grad():
        pass
    with torch.autocast("cuda", dtype=torch.float16):
        _, _, l_fused = tr.train_step(data)
        m.use_fused = False
        _, _, l_mod = tr.train_step(data)
        m.use_fused = True
    assert abs(float(l_fused) - float(l_mod)) < 2e-2 * max(1.0, abs(float(l_mod)))
    table0 = m.encoder_mask.embeddings.detach().clone()
    losses = [float(tr.step(data)) for _ in range(40)]
    assert np.isfinite(losses).all()
    assert np.mean(losses[-5:]) < 0.6 * np.mean(losses[:3]), losses
    # FusedAdam (nerf/optim.py) clears every gradient inside its update pass; the table itself must have moved
    assert m.encoder_mask.embeddings.grad is not None and float(m.encoder_mask.embeddings.grad.abs().sum()) == 0.0
    assert float((m.encoder_mask.embeddings.detach() - table0).abs().max()) > 1e-3


@pytest.mark.parametrize("K,reg", [(32, 0.1), (7, 0.0), (16, 1.0)])
def test_fused_loss_tail_matches_torch(cuda, K, reg):
    """inerf_mask_loss(+_backward) against the reference formulation (nerf/utils.py:1262-1285, 1310-1314) as restated in
    oracle/host_oracle.py, which is pinned to the reference's own MaskTrainer.train_step (tests/golden/ref_host.npz)."""
    from instance_nerf_b200.nerf.trainer import _MaskLoss
    from oracle import host_oracle
    g = torch.Generator().manual_seed(0)
    N, p = 64 * 12, 8
    logits = (torch.randn(N, K, generator=g) * 3).to(cuda).requires_grad_(True)
    depth = torch.rand(N, generator=g).to(cuda)
    labels = torch.randint(-1, K, (N,), generator=g).to(cuda)
    ref = host_oracle.mask_train_loss(logits, depth, labels, p, K, reg)
    ref.backward()
    g_ref = logits.grad.clone(); logits.grad = None
    out = _MaskLoss.apply(logits, depth, labels, p, reg)
    (out * 3.0).backward()
    torch.testing.assert_close(out, ref.detach(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(logits.grad / 3.0, g_ref, rtol=1e-4, atol=1e-7)


def _train_setup(cuda, K=16, n_rays=1024, seed=0):
    from instance_nerf_b200 import synthetic
    from oracle import host_oracle
    m, sc = build_model(cuda, K, density_scale=10.0)
    H, W = 96, 128
    poses = torch.from_numpy(synthetic.camera_poses(sc, 1, 1))
    r = host_oracle.get_rays(poses, synthetic.intrinsics(H, W), H, W, N=n_rays, patch_size=8, generator=torch.Generator().manual_seed(seed))
    o, d = r["rays_o"].reshape(-1, 3).contiguous(), r["rays_d"].reshape(-1, 3).contiguous()
    labels = torch.from_numpy(sc.first_hit_labels(o.numpy().astype(np.float64), d.numpy().astype(np.float64)))
    data = {"rays_o": o[None].to(cuda), "rays_d": d[None].to(cuda), "masks": labels[None].to(cuda),
            "noises": torch.rand(o.shape[0], generator=torch.Generator().manual_seed(1)).to(cuda)}
    return m, data


def test_graphed_train_step_matches_eager(cuda):
    """MaskTrainStep(cuda_graph=True): the whole step replayed as one CUDA graph over a fixed-size sample stream gives the
    same losses / parameters as the eager step (hash-table gradients are float atomics: compared with a tolerance), and a
    batch that marches more samples than the captured budget is NOT applied from the truncated stream: the device-side
    guard skips it, the host redoes it eagerly and re-captures."""
    from instance_nerf_b200.nerf.trainer import MaskTrainStep
    m_e, data = _train_setup(cuda)
    m_g, _ = _train_setup(cuda)
    tr_e = MaskTrainStep(m_e, lr=1e-2, fp16=True, label_regularization_weight=0.1)
    tr_g = MaskTrainStep(m_g, lr=1e-2, fp16=True, label_regularization_weight=0.1, cuda_graph=True)
    assert tr_g.cuda_graph
    le = [float(tr_e.step(data)) for _ in range(12)]
    lg = [float(tr_g.step(data)) for _ in range(12)]
    assert tr_g.graph_captures == 1 and tr_g.graph_replays == 12 - MaskTrainStep.GRAPH_WARMUP_STEPS
    np.testing.assert_allclose(lg, le, rtol=2e-3, atol=2e-4)
    for pe, pg in zip(m_e.mask_net.parameters(), m_g.mask_net.parameters()):
        torch.testing.assert_close(pg, pe, rtol=2e-2, atol=2e-4)
    # table gradients are float atomics in a nondeterministic order and Adam (eps 1e-15) turns a sign flip of a ~0 gradient into
    # a full lr-sized step: all but a handful of the 13.3 M entries agree
    te, tg = m_e.encoder_mask.embeddings.detach(), m_g.encoder_mask.embeddings.detach()
    bad = ((tg - te).abs() > 2e-4 + 2e-2 * te.abs()).float().mean().item()
    assert bad < 1e-5, bad
    # inference after graph replays sees the replayed parameters (packed fp16 copies are refreshed)
    m_e.eval(); m_g.eval()
    with torch.no_grad():
        kw = dict(staged=True, render_mask=True, perturb=False, dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4, bg_color=1)
        re_, rg_ = m_e.render(data["rays_o"], data["rays_d"], **kw), m_g.render(data["rays_o"], data["rays_d"], **kw)
    torch.testing.assert_close(rg_["instance_mask_logits"], re_["instance_mask_logits"], rtol=5e-2, atol=5e-3)

    # ---- overflow: shrink the budget below the marched total and re-capture ----
    total = tr_g._samples_seen
    tr_g._graph = None
    tr_g._samples_seen = total // 4
    before = [p.detach().clone() for p in m_g.mask_net.parameters()]
    caps = tr_g.graph_captures
    l1 = float(tr_g.step(data))          # captures with a too-small budget, replays (guard trips), redoes the batch eagerly
    le1 = float(tr_e.step(data))
    assert tr_g.graph_captures == caps + 1 and tr_g._graph is None and tr_g._samples_seen == total
    assert abs(l1 - le1) < 2e-3 * max(1.0, abs(le1))
    assert any(float((a - b).abs().max()) > 0 for a, b in zip(before, m_g.mask_net.parameters()))
    for pe, pg in zip(m_e.mask_net.parameters(), m_g.mask_net.parameters()):
        torch.testing.assert_close(pg, pe, rtol=2e-2, atol=3e-4)
    l2, le2 = float(tr_g.step(data)), float(tr_e.step(data))   # re-captured with a sufficient budget
    assert tr_g.graph_captures == caps + 2 and tr_g._graph is not None
    assert abs(l2 - le2) < 2e-3 * max(1.0, abs(le2))


def test_fused_adam_matches_torch_adam(cuda):
    """nerf/optim.py FusedAdam (one pass: unscale + Adam + clear gradient) against torch.optim.Adam with the reference's
    hyper-parameters (main_nerf_mask.py:182), including GradScaler's grad_scale / found_inf protocol."""
    from instance_nerf_b200.nerf.optim import FusedAdam
    g = torch.Generator().manual_seed(0)
    shapes = [(100003, 2), (64, 47), (7,)]
    p0 = [torch.randn(s, generator=g).to(cuda) for s in shapes]
    pa = [torch.nn.Parameter(t.clone()) for t in p0]
    pb = [torch.nn.Parameter(t.clone()) for t in p0]
    oa = FusedAdam([{"params": pa[:1], "lr": 1e-2}, {"params": pa[1:], "lr": 1e-3}], betas=(0.9, 0.99), eps=1e-15)
    ob = torch.optim.Adam([{"params": pb[:1], "lr": 1e-2}, {"params": pb[1:], "lr": 1e-3}], betas=(0.9, 0.99), eps=1e-15)
    scale = torch.tensor(1024.0, device=cuda)
    for it in range(6):
        grads = [torch.randn(s, generator=g).to(cuda) * (10.0 ** (it - 3)) for s in shapes]
        grads[0][::7] = 0.0                                         # untouched hash entries: zero gradient, momentum still moves them
        inf_step = it == 3
        for a, b, gr in zip(pa, pb, grads):
            a.grad = (gr * scale).clone()
            b.grad = gr.clone()
        oa.grad_scale, oa.found_inf = scale, torch.tensor(1.0 if inf_step else 0.0, device=cuda)
        oa.step()
        if not inf_step:
            ob.step()
        for a, b in zip(pa, pb):
            assert float(a.grad.abs().sum()) == 0.0                 # cleared by the step (also on a skipped step)
            torch.testing.assert_close(a.detach(), b.detach(), rtol=2e-6, atol=1e-7)
    for a, b in zip(pa, pb):
        # the gradients of successive steps span five orders of magnitude: compare the moments to fp32 rounding of their LARGEST
        # entries (entries that cancel to ~0 carry the absolute rounding error of the big terms in both implementations)
        ma, mb = oa.state[a]["exp_avg"], ob.state[b]["exp_avg"]
        va, vb = oa.state[a]["exp_avg_sq"], ob.state[b]["exp_avg_sq"]
        torch.testing.assert_close(ma, mb, rtol=1e-5, atol=2e-7 * float(mb.abs().max()))
        torch.testing.assert_close(va, vb, rtol=1e-5, atol=2e-7 * float(vb.abs().max()))
        assert float(oa.state[a]["step"]) == 5.0


def _host_gold():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_host.npz"))


def _gold_model(cuda, g, cuda_ray=True, **kw):
    """The product network carrying the state of the golden's reference network (small tensors stored, tables from the seed)."""
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork
    K, bound, seed = g["model_cfg"]
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")}
    gen = torch.Generator().manual_seed(int(seed))
    n_rows = int(sd["encoder.offsets"][-1])
    for name in ("encoder.embeddings", "encoder_mask.embeddings"):
        sd[name] = (torch.rand(n_rows, 2, generator=gen) * 2 - 1) * 0.5
    m = NeRFNetwork(bound=float(bound), cuda_ray=cuda_ray, num_instances=int(K), **kw)
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all(k.startswith("density") or k == "step_counter" for k in missing.missing_keys), missing
    return m.to(cuda)


@pytest.mark.parametrize("tag", ["ce", "reg"])
def test_fused_loss_matches_reference_train_step_golden(cuda, tag):
    """inerf_mask_loss / _backward against the loss and dloss/dlogits of the REFERENCE's MaskTrainer.train_step run on the CPU
    (tests/golden/make_golden_host.py, render stubbed to return these maps)."""
    from instance_nerf_b200.nerf.trainer import _MaskLoss
    g = _host_gold()
    want, reg_w, _ = g[f"loss_{tag}"]
    logits = torch.from_numpy(g["loss_logits"])[0].to(cuda).requires_grad_(True)
    depth, labels = torch.from_numpy(g["loss_depth"])[0].to(cuda), torch.from_numpy(g["loss_labels"])[0].to(cuda)
    loss = _MaskLoss.apply(logits, depth, labels, int(g["loss_patch"]), float(reg_w))
    loss.backward()
    assert abs(float(loss) - float(want)) < 1e-5 * max(1.0, abs(float(want)))
    np.testing.assert_allclose(logits.grad.cpu().numpy(), g[f"loss_{tag}_grad"][0], rtol=1e-4, atol=1e-7)
    # every pixel unlabelled: the cross-entropy term is 0 (nerf/utils.py:1313-1314)
    l0 = _MaskLoss.apply(logits.detach(), depth, torch.full_like(labels, -1), int(g["loss_patch"]), 0.0)
    assert float(l0) == float(g["loss_unlabelled"]) == 0.0


def test_mask3d_loss_matches_reference(cuda):
    """MaskTrainStep.mask3d_loss (nerf/utils.py:1250-1260) and the full train_step loss with mask3d_loss_weight > 0 against
    the reference: the 3D-mask query runs the one-launch fused field (fp16 operands) where the golden is the reference net in
    fp32 on the CPU, hence the 2e-2 tolerance on logits; the modular path under fp32 must agree to 1e-4."""
    from instance_nerf_b200.nerf.trainer import MaskTrainStep
    g = _host_gold()
    m = _gold_model(cuda, g).train()
    tr = MaskTrainStep(m, fp16=True, patch_size=int(g["loss_patch"]), label_regularization_weight=0.1, mask3d_loss_weight=0.5)
    data = {"mask3d_coords": torch.from_numpy(g["m3_coords"]).to(cuda), "mask3d_labels": torch.from_numpy(g["m3_labels"]).to(cuda)}
    with torch.autocast("cuda", dtype=torch.float16):
        assert m.fused_train_available(data["mask3d_coords"], data["mask3d_coords"])
        l_fused = tr.mask3d_loss(data)
    assert l_fused.requires_grad and l_fused.shape == (200,)
    assert abs(float(l_fused.mean()) - float(g["m3_loss"])) < 2e-2 * max(1.0, float(g["m3_loss"]))
    l_fused.mean().backward()
    assert float(m.encoder_mask.embeddings.grad.abs().sum()) > 0 and all(float(l.weight.grad.abs().sum()) > 0 for l in m.mask_net)
    m.use_fused = False
    l_mod = tr.mask3d_loss(data)       # fp32 modular path: GridEncoder kernels + nn.Linear
    assert abs(float(l_mod.mean()) - float(g["m3_loss"])) < 1e-4 * max(1.0, float(g["m3_loss"]))
    # whole loss of train_step with the three terms, render stubbed to the golden's maps exactly as in the generator
    logits = torch.from_numpy(g["loss_logits"]).to(cuda).requires_grad_(True)
    depth, labels = torch.from_numpy(g["loss_depth"]).to(cuda), torch.from_numpy(g["loss_labels"]).to(cuda)
    m.render = lambda *a, **kw: {"instance_mask_logits": logits, "depth": depth}
    _, _, loss = tr.train_step({"rays_o": None, "rays_d": None, "masks": labels, **data})
    want = float(g["loss_all"][0])
    assert abs(float(loss) - want) < 1e-4 * max(1.0, abs(want))
    (grad,) = torch.autograd.grad(loss, logits)
    np.testing.assert_allclose(grad.cpu().numpy(), g["loss_all_grad"], rtol=1e-4, atol=1e-7)


def test_train_step_with_mask3d_and_density_scale_fused_vs_modular(cuda):
    """density_scale != 1 through the training path: the fused field returns the UNSCALED sigma (as network_mask.py:119-158
    does) and run_cuda applies density_scale once (mask_renderer.py:273) -- fused and modular steps must composite alike, and
    the fused render (which scales inside the kernel) must agree with the alive-ray loop on the same model."""
    from instance_nerf_b200.nerf.trainer import MaskTrainStep
    m, data = _train_setup(cuda)          # density_scale = 10
    B = 4096
    g = torch.Generator().manual_seed(5)
    x = ((torch.rand(B, 3, generator=g) * 2 - 1) * 7.5).to(cuda)
    d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g), dim=-1).to(cuda)
    with torch.no_grad():
        s_f = m.forward_fused(x, d)[0]
        m.use_fused = False
        with torch.autocast("cuda", dtype=torch.float16):
            s_m = m(x, d)[0].float()
        m.use_fused = True
    torch.testing.assert_close(s_f, s_m, rtol=2e-2, atol=1e-3)            # both unscaled
    tr = MaskTrainStep(m, lr=1e-2, fp16=True, label_regularization_weight=0.1)
    m.train()
    with torch.autocast("cuda", dtype=torch.float16):
        out_f = m.render(data["rays_o"], data["rays_d"], render_mask=True, bg_color=1, perturb=True, force_all_rays=True, noises=data["noises"],
                         dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4)
        m.use_fused = False
        out_m = m.render(data["rays_o"], data["rays_d"], render_mask=True, bg_color=1, perturb=True, force_all_rays=True, noises=data["noises"],
                         dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4)
        m.use_fused = True
    for k in ("weights_sum", "depth", "image"):
        torch.testing.assert_close(out_f[k].float(), out_m[k].float(), rtol=0, atol=2e-3)
    torch.testing.assert_close(out_f["instance_mask_logits"].float(), out_m["instance_mask_logits"].float(), rtol=2e-2, atol=2e-2)
    # a semi-transparent medium makes the squared scale visible: thin the density so that weights_sum is well inside (0, 1)
    m.eval()
    m.density_scale = 0.05
    kw = dict(render_mask=True, dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4)
    with torch.no_grad():
        o, dd = data["rays_o"].view(-1, 3), data["rays_d"].view(-1, 3)
        from instance_nerf_b200 import raymarching as rm
        nears, fars = rm.near_far_from_aabb(o, dd, m.aabb_infer, m.min_near)
        ws_f = m._render_fused(o, dd, nears, fars, True, 1 / 128, 1024, 1e-4)[0]
        ws_l = m.run_cuda_loop(o, dd, nears, fars, True, 1 / 128, False, 1024, 1e-4)[0]     # loop on the fused per-sample field
    assert 0.05 < float(ws_f.mean()) < 0.95
    torch.testing.assert_close(ws_f, ws_l, rtol=0, atol=2e-3)
