"""GPU parity of the fused instance field (tcgen05 MLP + hash gathers in one kernel) against the reference
operator sequence (network_mask.py:119-158 under fp16 autocast = the reference's `-O` preset), which here runs
on the op-level kernels already proven bit-exact against the reference (test_ops_vs_ref_gpu.py) + nn.Linear."""
import numpy as np
import pytest
import torch

from helpers import make_rays, scene_arrays

pytestmark = pytest.mark.gpu


def build_model(cuda, K=32, bound=8.0, seed=0, density_scale=1.0):
    from instance_nerf_b200 import synthetic
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork
    torch.manual_seed(seed)
    m = NeRFNetwork(bound=bound, cuda_ray=True, num_instances=K, density_scale=density_scale, density_thresh=10)
    synthetic.randomize_tables(m, seed)
    sc, cascade, grid, bits = scene_arrays(16, bound, 0)
    with torch.no_grad():
        m.density_grid.copy_(torch.from_numpy(grid))
        m.density_bitfield.copy_(torch.from_numpy(bits))
    return m.to(cuda).eval(), sc


# bound 2 (the reference's default): levels 4-7 form a mixed quarter, which the fused kernels encode on their generic path
@pytest.mark.parametrize("K,B,bound", [(32, 128 * 37 + 5, 8.0), (16, 1000, 8.0), (2, 64, 8.0), (48, 300, 8.0), (32, 128 * 37 + 5, 2.0)],
                         ids=["32-4741", "16-1000", "2-64", "48-300", "32-4741-bound2"])
def test_field_fused_vs_modular(cuda, K, B, bound):
    m, _ = build_model(cuda, K, bound=bound)
    g = torch.Generator().manual_seed(1)
    x = ((torch.rand(B, 3, generator=g) * 2 - 1) * 7.9 * bound / 8).to(cuda)
    x[:4] = torch.tensor([[1.0, -1.0, 0.0], [0.0, 0.0, 0.0], [1.0, 1.0, 1.0], [-1.0, -1.0, -1.0]], device=cuda) * bound
    d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g), dim=-1).to(cuda)
    with torch.no_grad():
        s1, c1, k1 = m.forward_fused(x, d)
        m.use_fused = False
        with torch.autocast("cuda", dtype=torch.float16):
            s0, c0, k0 = m(x, d)
        m.use_fused = True
    s0, c0, k0 = s0.float(), c0.float(), k0.float()
    # fp16 activations: one half-ulp rounding flip in a hidden unit moves an output by ~1e-3 relative
    exact = (s0 == s1).float().mean().item()
    assert exact > 0.5, f"only {exact:.3f} of sigmas bit-identical"
    torch.testing.assert_close(s1, s0, rtol=2e-2, atol=1e-3)
    torch.testing.assert_close(c1, c0, rtol=0, atol=2e-3)
    torch.testing.assert_close(k1, k0, rtol=2e-2, atol=2e-2)
    assert (k1 - k0).abs().mean().item() < 1e-3


def test_field_fused_oob_is_zero_features(cuda):
    """Coordinates outside [-bound, bound] get zero encoder features (gridencoder.cu:110-135)."""
    m, _ = build_model(cuda, 32)
    x = torch.tensor([[9.0, 0.0, 0.0], [0.0, -8.5, 1.0]], device=cuda)
    d = torch.tensor([[0.0, 0.0, 1.0], [1.0, 0.0, 0.0]], device=cuda)
    with torch.no_grad():
        s1, c1, k1 = m.forward_fused(x, d)
        m.use_fused = False
        with torch.autocast("cuda", dtype=torch.float16):
            s0, c0, k0 = m(x, d)
    assert torch.equal(s1, s0.float())            # sigma = exp(0) = 1 exactly
    torch.testing.assert_close(c1, c0.float(), rtol=0, atol=2e-3)
    torch.testing.assert_close(k1, k0.float(), rtol=2e-2, atol=2e-2)


def _render_both(m, o, d, **kw):
    with torch.no_grad():
        m.use_fused = True
        r1 = m.render(o[None], d[None], staged=True, render_mask=True, perturb=False, **kw)
        m.use_fused = False
        with torch.autocast("cuda", dtype=torch.float16):
            r0 = m.render(o[None], d[None], staged=True, render_mask=True, perturb=False, **kw)
        m.use_fused = True
    return r1, r0


@pytest.mark.parametrize("K,density_scale,bound", [(32, 1.0, 8.0), (16, 25.0, 8.0), (16, 25.0, 2.0), (16, 25.0, 3.0)],
                         ids=["32-1.0", "16-25.0", "16-25.0-bound2", "16-25.0-bound3"])
def test_render_fused_vs_reference_loop(cuda, K, density_scale, bound):
    """Whole-frame inference: the one-launch fused renderer against the reference's alive-ray loop
    (mask_renderer.py:330-381) run on the op-level kernels.  North-star tolerance: maps within 1e-3.  Bound 2 has 2 cascades,
    bound 3 has 3 with the coarsest one clipped to the box, and both encode levels 4-7 as a mixed quarter."""
    m, sc = build_model(cuda, K, bound=bound, density_scale=density_scale)
    o, d = make_rays(sc, 96, 128)
    o, d = o.to(cuda), d.to(cuda)
    r1, r0 = _render_both(m, o, d, dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4)
    for key in ("image", "depth"):
        err = (r1[key] - r0[key]).abs()
        assert err.max().item() < 1e-3, f"{key}: max err {err.max().item():.3e}"
    p1 = torch.softmax(r1["instance_mask_logits"], -1)
    p0 = torch.softmax(r0["instance_mask_logits"], -1)
    assert (p1 - p0).abs().max().item() < 1e-3
    assert r1["image"].shape == (1, 96 * 128, 3) and r1["instance_mask_logits"].shape == (1, 96 * 128, K)


def test_render_fused_perturb_vs_reference_loop(cuda):
    """perturb=True at inference (mask_renderer.py:334-337: one uniform draw per ray jitters the first step, raymarching.cu:1004):
    the one-launch renderer with the draws injected against the alive-ray loop with the same draws; and a perturbed frame
    differs from the unperturbed one (the jitter is really applied)."""
    m, sc = build_model(cuda, 16, density_scale=25.0)
    o, d = make_rays(sc, 64, 96)
    o, d = o.to(cuda), d.to(cuda)
    noises = torch.rand(o.shape[0], generator=torch.Generator().manual_seed(5)).to(cuda)
    kw = dict(dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4, staged=True, render_mask=True, bg_color=1)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        r1 = m.render(o[None], d[None], perturb=True, noises=noises, **kw)
        m.use_fused = False
        try:
            r0 = m.render(o[None], d[None], perturb=True, noises=noises, **kw)
        finally:
            m.use_fused = True
        plain = m.render(o[None], d[None], perturb=False, **kw)
        drawn = m.render(o[None], d[None], perturb=True, **kw)        # own draw: runs, finite, differs from the plain frame
    for key in ("image", "depth"):
        assert (r1[key] - r0[key]).abs().max().item() < 1e-3, key
    assert (torch.softmax(r1["instance_mask_logits"], -1) - torch.softmax(r0["instance_mask_logits"], -1)).abs().max().item() < 1e-3
    assert (r1["depth"] - plain["depth"]).abs().max().item() > 1e-5
    assert torch.isfinite(drawn["image"]).all() and (drawn["depth"] - plain["depth"]).abs().max().item() > 1e-5


def test_render_fused_no_mask_and_misses(cuda):
    m, sc = build_model(cuda, 32, density_scale=25.0)
    o, d = make_rays(sc, 32, 32)
    o = torch.cat([o, torch.tensor([[20.0, 20.0, 20.0]])]).to(cuda)      # a ray that misses the volume
    d = torch.cat([d, torch.tensor([[0.0, 1.0, 0.0]])]).to(cuda)
    with torch.no_grad():
        r = m.render(o[None], d[None], staged=True, render_mask=False, perturb=False, dt_gamma=1 / 128, max_steps=1024, bg_color=1)
        rm_ = m.render(o[None], d[None], staged=True, render_mask=True, perturb=False, dt_gamma=1 / 128, max_steps=1024, bg_color=1)
    assert r["instance_mask_logits"] is None
    torch.testing.assert_close(r["image"], rm_["image"], rtol=0, atol=1e-6)
    assert torch.allclose(r["image"][0, -1], torch.ones(3, device=cuda))    # miss -> pure background
    assert float(rm_["instance_mask_logits"][0, -1].abs().sum()) == 0.0


@pytest.mark.parametrize("H,W", [(480, 640), (1080, 1920)])
def test_render_fused_full_size_split_invariance(cuda, H, W):
    """BASELINE.json's full frame sizes (c2 640x480, c4 1920x1080) through size-independent properties: rays are
    independent, so (a) a frame rendered in one launch equals, BIT FOR BIT, the same rays rendered as two launches of
    uneven, non-multiple-of-32 halves (different tile / slot / patch assignment of every ray), (b) two runs agree bit for
    bit (no scheduling-dependent arithmetic), (c) weights_sum stays in [0, 1] and every ray that hits nothing is background."""
    m, sc = build_model(cuda, 32, density_scale=10.0)
    o, d = make_rays(sc, H, W)
    o, d = o.to(cuda), d.to(cuda)
    N = o.shape[0]
    kw = dict(staged=True, render_mask=True, perturb=False, dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4, bg_color=1)
    cut = N // 3 + 17
    with torch.no_grad():
        full = m.render(o[None], d[None], **kw)
        again = m.render(o[None], d[None], **kw)
        a = m.render(o[None, :cut], d[None, :cut], **kw)
        b = m.render(o[None, cut:], d[None, cut:], **kw)
    for key in ("image", "depth", "instance_mask_logits"):
        assert torch.equal(full[key], again[key]), key
        assert torch.equal(full[key], torch.cat([a[key], b[key]], dim=1)), key
    assert torch.isfinite(full["image"]).all() and torch.isfinite(full["instance_mask_logits"]).all()
    assert float(full["image"].min()) >= 0.0 and float(full["image"].max()) <= 1.0 + 1e-5


def test_update_extra_state_full_sweep_vs_oracle(cuda):
    """SURVEY.md section 8a row 12: the full-sweep branch of update_extra_state (mask_renderer.py:466-495 -> EMA -> mean ->
    threshold -> packbits) with injected jitter, against the CPU restatement: a sample of cells per cascade is recomputed
    on the host (query point from the Morton index and the cell's row of the jitter block, fp32 field) and the whole
    grid -> (mean, bitfield) tail is recomputed from the GPU grid with the numpy EMA / packbits restatement (bit-exact)."""
    _full_sweep_vs_oracle(cuda, 8.0)


def test_update_extra_state_full_sweep_vs_oracle_bound2(cuda):
    """The same at bound 2 (2 cascades), where the sweep kernel encodes levels 4-7 as a mixed quarter."""
    _full_sweep_vs_oracle(cuda, 2.0)


def _full_sweep_vs_oracle(cuda, bound):
    from oracle import field_oracle as fo
    m, _ = build_model(cuda, 8, bound=bound, density_scale=1.0)
    m.train()
    m.reset_extra_state()
    G, C = m.grid_size, m.cascade
    g = torch.Generator().manual_seed(5)
    noises = [torch.rand(G ** 3, 3, generator=g) for _ in range(C)]          # the reference's draw order: meshgrid rows
    # the device sweep walks the cells in Morton order: row m of cascade c takes the draw of the cell with Morton index m
    from oracle import raymarch_oracle as ro
    cc = ro.morton3D_invert(np.arange(G ** 3, dtype=np.int32)).astype(np.int64)
    lin = torch.from_numpy((cc[:, 0] * G + cc[:, 1]) * G + cc[:, 2])
    with torch.autocast("cuda", dtype=torch.float16):
        m.update_extra_state(decay=0.95, noises=torch.cat([n[lin] for n in noises]).to(cuda))
    torch.cuda.synchronize()
    grid = m.density_grid.detach().cpu().numpy()
    assert m.iter_density == 1 and np.isfinite(grid).all() and (grid >= 0).all()

    field = fo.OracleField({k: v.detach().cpu() for k, v in m.state_dict().items()}, m.bound, m.num_instances, density_scale=m.density_scale)
    rng = np.random.RandomState(0)
    for cas in range(C):
        cells = rng.randint(0, G ** 3, size=20000)
        x = fo.extra_state_sweep_points(cells, cas, G, m.bound, noises[cas].numpy())
        with torch.no_grad():
            sig = field.density(torch.from_numpy(x))["sigma"].numpy() * m.density_scale
        # first update from an all-zero grid: grid = max(0 * decay, sigma) = sigma; fp16 autocast MLP on the device vs fp32 here
        np.testing.assert_allclose(grid[cas, cells], sig, rtol=2e-2, atol=1e-3)
    # the EMA -> mean -> threshold -> packbits tail, recomputed from the device grid: identity EMA (tmp == grid), bit-exact bits
    g2, mean, bits = fo.update_grid_ema(np.zeros_like(grid), grid, 0.95, m.density_thresh)
    assert np.array_equal(g2, grid)
    assert abs(float(m.mean_density) - mean) < 1e-5 * max(1.0, mean)
    assert np.array_equal(m.density_bitfield.cpu().numpy(), bits)


def test_run_non_cuda_ray_matches_reference_python_renderer(cuda):
    """NeRFRenderer.run (cuda_ray=False, mask_renderer.py:89-231) through the staged render() on the GPU against the outputs of
    the REFERENCE's own Python renderer (tests/golden/ref_run.npz: NeRFNetwork.render imported unmodified, CPU, fp32).  The
    modular field (GridEncoder / SHEncoder kernels + nn.Linear, fp32) is used: `run` calls density / color / mask separately."""
    import os
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_run.npz"))
    K, bound, H, W, T, seed = g["cfg"]
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")}
    gen = torch.Generator().manual_seed(int(seed))
    n_rows = int(sd["encoder.offsets"][-1])
    for name in ("encoder.embeddings", "encoder_mask.embeddings"):
        sd[name] = (torch.rand(n_rows, 2, generator=gen) * 2 - 1) * 0.5
    m = NeRFNetwork(bound=float(bound), cuda_ray=False, num_instances=int(K))
    m.load_state_dict(sd)
    m = m.to(cuda).eval()
    o, d = torch.from_numpy(g["rays_o"]).to(cuda), torch.from_numpy(g["rays_d"]).to(cuda)
    with torch.no_grad():
        res = m.render(o[None], d[None], staged=True, max_ray_batch=100, render_mask=True, num_steps=int(T), upsample_steps=0, perturb=False, bg_color=1)
    np.testing.assert_allclose(res["image"].cpu().numpy(), g["image"], rtol=0, atol=1e-3)
    np.testing.assert_allclose(res["depth"].cpu().numpy(), g["depth"], rtol=0, atol=1e-3)
    p1 = torch.softmax(res["instance_mask_logits"].cpu(), -1).numpy()
    p0 = torch.softmax(torch.from_numpy(g["logits"]), -1).numpy()
    np.testing.assert_allclose(p1, p0, rtol=0, atol=1e-3)
    # observed differences are ~1e-6 (fp32 on both sides); also exercise the hierarchical branch (upsample_steps > 0): finite, same shapes
    with torch.no_grad():
        r2 = m.render(o[None], d[None], staged=True, max_ray_batch=100, render_mask=True, num_steps=int(T), upsample_steps=16, perturb=False, bg_color=1)
    assert r2["image"].shape == res["image"].shape and bool(torch.isfinite(r2["image"]).all()) and bool(torch.isfinite(r2["instance_mask_logits"]).all())


def test_background_model_fused_vs_loop(cuda):
    """bg_radius > 0 (network_mask.py:95-114, 268; mask_renderer.py:246-249): the background colour comes from sph_from_ray ->
    2-D hash grid + SH -> bg_net and is mixed in by run_cuda's `(1 - weights_sum) * bg_color` tail, so the one-launch renderer
    and the alive-ray loop (modular field) must agree; it must also differ from the constant-background render."""
    from instance_nerf_b200 import synthetic
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork
    torch.manual_seed(0)
    m = NeRFNetwork(bound=8.0, cuda_ray=True, num_instances=8, density_scale=0.05, density_thresh=10, bg_radius=12.0)
    synthetic.randomize_tables(m, 0)
    with torch.no_grad():
        m.encoder_bg.embeddings.uniform_(-1.0, 1.0)
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    with torch.no_grad():
        m.density_grid.copy_(torch.from_numpy(grid)); m.density_bitfield.copy_(torch.from_numpy(bits))
    m = m.to(cuda).eval()
    o, d = (t.to(cuda) for t in make_rays(sc, 48, 64))
    kw = dict(staged=True, render_mask=True, perturb=False, dt_gamma=1 / 128, max_steps=1024, T_thresh=1e-4)
    with torch.no_grad():
        assert m.fused_render_available(True)
        a = m.render(o[None], d[None], **kw)
        m.use_fused = False
        with torch.autocast("cuda", dtype=torch.float16):
            b = m.render(o[None], d[None], **kw)
        m.use_fused = True
        m.bg_radius = -1
        c = m.render(o[None], d[None], bg_color=1, **kw)
    torch.testing.assert_close(a["image"], b["image"].float(), rtol=0, atol=2e-3)
    torch.testing.assert_close(a["depth"], b["depth"].float(), rtol=0, atol=1e-3)
    assert float((a["image"] - c["image"]).abs().max()) > 0.05      # thin medium: the background shows through
