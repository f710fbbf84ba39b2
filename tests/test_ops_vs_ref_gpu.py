"""GPU parity: every libinerf_b200 op against the reference's own kernels on the same inputs, whose outputs are recorded
in tests/golden/recorded_test_ops_vs_ref_gpu.npz (helpers.Recorded).

Bar (BASELINE.json north_star): integer / index / marched-sample streams bit-exact; floating-point
compositing / encoding within the stated tolerance (hash encode and SH are in fact bit-exact too)."""
import numpy as np
import pytest
import torch

from helpers import adversarial_rays, bits_equal, make_rays, scene_arrays

pytestmark = pytest.mark.gpu


def _dev(*ts, device):
    return [t.to(device).contiguous() for t in ts]


@pytest.mark.parametrize("bound", [8.0, 2.0, 3.0])
def test_near_far_bit_exact(recorded, cuda, bound):
    from instance_nerf_b200 import raymarching as rm
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = make_rays(sc, 60, 80)
    ao, ad = adversarial_rays(bound)
    o, d = _dev(torch.cat([o, ao]), torch.cat([d, ad]), device=cuda)
    aabb = torch.tensor([-bound] * 3 + [bound] * 3, dtype=torch.float32, device=cuda)
    n1, f1 = rm.near_far_from_aabb(o, d, aabb, 0.2)
    recorded.exact("nears", n1)
    recorded.exact("fars", f1)


def test_morton_packbits_bit_exact(recorded, cuda):
    from instance_nerf_b200 import raymarching as rm
    g = torch.Generator().manual_seed(0)
    coords = torch.randint(0, 128, (100003, 3), generator=g, dtype=torch.int32).to(cuda)
    i1 = rm.morton3D(coords)
    recorded.exact("morton", i1)
    c1 = rm.morton3D_invert(i1)
    assert torch.equal(c1, coords)
    # known answers (SURVEY.md section 8c)
    ka = rm.morton3D(torch.tensor([[1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=torch.int32, device=cuda))
    assert ka.tolist() == [1, 2, 4]

    grid = (torch.rand(4, 128 ** 3, generator=g) * 20 - 2).to(cuda)
    for thresh in (0.0, 5.0, 10.0):
        b1 = rm.packbits(grid, thresh)
        recorded.exact(f"packbits_{thresh}", b1)


def _march(cuda, o, d, bits, bound, cascade, dt_gamma, max_steps, perturb_seed):
    from instance_nerf_b200 import raymarching as rm
    N = o.shape[0]
    aabb = torch.tensor([-bound] * 3 + [bound] * 3, dtype=torch.float32, device=cuda)
    nears, fars = rm.near_far_from_aabb(o, d, aabb, 0.2)
    if perturb_seed is None:
        noises = torch.zeros(N, device=cuda)
    else:
        noises = torch.rand(N, generator=torch.Generator().manual_seed(perturb_seed)).to(cuda)
    counter = torch.zeros(2, dtype=torch.int32, device=cuda)
    xyzs, dirs, deltas, rays = rm.march_rays_train(o, d, bound, bits, cascade, 128, nears, fars, counter, -1, False, 128, True,
                                                   dt_gamma, max_steps, noises=noises)
    torch.cuda.synchronize()
    return xyzs, dirs, deltas, rays, counter


@pytest.mark.parametrize("cfg", [
    dict(bound=8.0, dt_gamma=1 / 128, max_steps=1024, seed=None),
    dict(bound=8.0, dt_gamma=1 / 128, max_steps=1024, seed=2),
    dict(bound=8.0, dt_gamma=0.0, max_steps=512, seed=3),
    dict(bound=3.0, dt_gamma=1 / 128, max_steps=1024, seed=4),   # non power-of-two bound: mip_rbound = 1/3 is inexact
    dict(bound=2.0, dt_gamma=1 / 256, max_steps=256, seed=5),
    dict(bound=1.0, dt_gamma=0.0, max_steps=128, seed=6),
    dict(bound=8.0, dt_gamma=1 / 128, max_steps=1024, seed=7, big=True),
    dict(bound=3.0, dt_gamma=1 / 128, max_steps=64, seed=8, big=True),
    dict(bound=8.0, dt_gamma=1 / 128, max_steps=37, seed=9),      # max_steps cuts rays short inside a 32-candidate batch
])
def test_march_rays_train_bit_exact(recorded, cuda, cfg):
    """12 288 + adversarial rays -> the one-warp-per-ray kernels (k_march_train_warp); with cfg["big"] 30 720 rays -> the
    thread-per-ray kernels (raymarch.cu use_warp_march)."""
    bound = cfg["bound"]
    sc, cascade, grid, bits = scene_arrays(16, bound, 0)
    o, d = make_rays(sc, *((160, 192) if cfg.get("big") else (96, 128)))
    ao, ad = adversarial_rays(bound)
    o, d = _dev(torch.cat([o, ao]), torch.cat([d, ad]), device=cuda)
    bits_t = torch.from_numpy(bits).to(cuda)
    xyzs, dirs, deltas, rays, counter = _march(cuda, o, d, bits_t, bound, cascade, cfg["dt_gamma"], cfg["max_steps"], cfg["seed"])
    recorded.exact("counter", counter)
    total = int(counter[0])
    assert total > 1000
    # the reference's stream in canonical order (helpers.canonicalize), bit-exact
    recorded.exact("rays", rays)
    recorded.exact("xyzs", xyzs[:total]); recorded.exact("dirs", dirs[:total]); recorded.exact("deltas", deltas[:total])
    assert float(xyzs[total:].abs().sum()) == 0.0                # padding rows are zero


def test_march_rays_train_budget_and_empty(cuda):
    """mean_count budget (rays past M dropped) and N == 0."""
    from instance_nerf_b200 import raymarching as rm
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = _dev(*make_rays(sc, 32, 32), device=cuda)
    bits_t = torch.from_numpy(bits).to(cuda)
    aabb = torch.tensor([-8.0] * 3 + [8.0] * 3, device=cuda)
    nears, fars = rm.near_far_from_aabb(o, d, aabb, 0.2)
    counter = torch.zeros(2, dtype=torch.int32, device=cuda)
    xyzs, dirs, deltas, rays = rm.march_rays_train(o, d, 8.0, bits_t, cascade, 128, nears, fars, counter, 1000, False, 128, False, 1 / 128, 1024)
    assert xyzs.shape[0] == 1024
    r = rays.cpu().numpy()
    kept = (r[:, 1] + r[:, 2] <= 1024) & (r[:, 2] > 0)
    last = (r[kept, 1] + r[kept, 2]).max()
    assert float(xyzs[last:].abs().sum()) == 0.0 and float(xyzs[:last].abs().sum()) > 0
    e = torch.empty(0, 3, device=cuda)
    x2, _, _, r2 = rm.march_rays_train(e, e, 8.0, bits_t, cascade, 128, torch.empty(0, device=cuda), torch.empty(0, device=cuda),
                                      None, -1, False, 128, True, 1 / 128, 1024)
    assert r2.shape == (0, 3) and x2.shape[0] == 128


@pytest.mark.parametrize("n_step", [1, 3, 8])
def test_march_rays_infer_bit_exact(recorded, cuda, n_step):
    from instance_nerf_b200 import raymarching as rm
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = _dev(*make_rays(sc, 64, 64), device=cuda)
    N = o.shape[0]
    bits_t = torch.from_numpy(bits).to(cuda)
    aabb = torch.tensor([-8.0] * 3 + [8.0] * 3, device=cuda)
    nears, fars = rm.near_far_from_aabb(o, d, aabb, 0.2)
    g = torch.Generator().manual_seed(7)
    alive = torch.randperm(N, generator=g)[: N // 2].int().to(cuda)
    n_alive = alive.shape[0]
    rays_t = (nears + torch.rand(N, generator=g).to(cuda) * 2.0).contiguous()
    x1, d1, l1 = rm.march_rays(n_alive, n_step, alive, rays_t, o, d, 8.0, bits_t, cascade, 128, nears, fars, 128, False, 1 / 128, 1024)
    recorded.exact("xyzs", x1); recorded.exact("dirs", d1); recorded.exact("deltas", l1)


def _fake_field(M, K, cuda, seed):
    g = torch.Generator().manual_seed(seed)
    sigmas = torch.exp(torch.randn(M, generator=g) * 1.5 + 1.0).to(cuda)
    rgbs = torch.rand(M, 3, generator=g).to(cuda)
    masks = (torch.randn(M, K, generator=g) * 2).to(cuda) if K else None
    return sigmas, rgbs, masks


@pytest.mark.parametrize("K", [0, 16, 32, 40])
def test_composite_train_fwd_bwd(recorded, cuda, K):
    from instance_nerf_b200 import raymarching as rm
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = _dev(*make_rays(sc, 48, 64), device=cuda)
    bits_t = torch.from_numpy(bits).to(cuda)
    xyzs, dirs, deltas, rays, counter = _march(cuda, o, d, bits_t, 8.0, cascade, 1 / 128, 1024, 11)
    M, N = xyzs.shape[0], rays.shape[0]
    sigmas, rgbs, masks = _fake_field(M, K, cuda, 5)
    sigmas.requires_grad_(True); rgbs.requires_grad_(True)
    T_thresh = 1e-4
    g = torch.Generator().manual_seed(9)
    gws = torch.randn(N, generator=g).to(cuda); gim = torch.randn(N, 3, generator=g).to(cuda)
    if K == 0:
        ws, dp, im = rm.composite_rays_train(sigmas, rgbs, deltas, rays, T_thresh)
        (ws * gws).sum().add((im * gim).sum()).backward()
    else:
        masks.requires_grad_(True)
        gmo = torch.randn(N, K, generator=g).to(cuda)
        ws, dp, im, mo = rm.composite_rays_with_masks_train(sigmas, rgbs, masks, deltas, rays, T_thresh)
        ((ws * gws).sum() + (im * gim).sum() + (mo * gmo).sum()).backward()
        recorded.close("mask_out", mo, rtol=1e-5, atol=1e-5)
        recorded.close("grad_masks", masks.grad, rtol=1e-5, atol=1e-6)
    # tolerance: fp32 compositing, identical operation order for the forward -> tight
    recorded.close("weights_sum", ws, rtol=1e-6, atol=1e-6)
    recorded.close("depth", dp, rtol=1e-5, atol=1e-5)
    recorded.close("image", im, rtol=1e-5, atol=1e-6)
    recorded.close("grad_rgbs", rgbs.grad, rtol=1e-5, atol=1e-6)
    recorded.close("grad_sigmas", sigmas.grad, rtol=1e-3, atol=1e-4)   # K-term sum is re-associated (warp reduce)


@pytest.mark.parametrize("K", [0, 32, 40])
def test_composite_train_bwd_dense_needs_no_zero_fill(cuda, K):
    """inerf_composite_rays_with_masks_train_backward_dense: NaN-poisoned gradient buffers come back equal, bit for bit, to
    the zero-filled contract of raymarching.cu:828-951 (checked against the reference kernel's output above), and the sigma / rgb
    gradients may be left out."""
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = _dev(*make_rays(sc, 48, 64), device=cuda)
    bits_t = torch.from_numpy(bits).to(cuda)
    xyzs, dirs, deltas, rays, counter = _march(cuda, o, d, bits_t, 8.0, cascade, 1 / 128, 1024, 11)
    M, N = int(counter[0].item()), rays.shape[0]          # the dense part of the stream: no alignment rows
    deltas = deltas[:M].contiguous()
    sigmas, rgbs, masks = _fake_field(M, K, cuda, 5)
    sigmas = sigmas * 4                                    # early termination on most rays: long zero tails
    T = 1e-4
    g = torch.Generator().manual_seed(9)
    gws = torch.randn(N, generator=g).to(cuda); gim = torch.randn(N, 3, generator=g).to(cuda)
    gmo = torch.randn(N, max(K, 1), generator=g).to(cuda)
    ws = torch.empty(N, device=cuda); dp = torch.empty(N, device=cuda); im = torch.empty(N, 3, device=cuda); mo = torch.empty(N, max(K, 1), device=cuda)
    st = stream_ptr(cuda)
    if K:
        call("inerf_composite_rays_with_masks_train_forward", ptr(sigmas), ptr(rgbs), ptr(masks), ptr(deltas), ptr(rays), M, N, K, T, ptr(ws), ptr(dp), ptr(im), ptr(mo), st)
    else:
        call("inerf_composite_rays_train_forward", ptr(sigmas), ptr(rgbs), ptr(deltas), ptr(rays), M, N, T, ptr(ws), ptr(dp), ptr(im), st)
    gs0 = torch.zeros(M, device=cuda); gr0 = torch.zeros(M, 3, device=cuda); gm0 = torch.zeros(M, max(K, 1), device=cuda)
    if K:
        call("inerf_composite_rays_with_masks_train_backward", ptr(gws), ptr(gim), ptr(gmo), ptr(sigmas), ptr(rgbs), ptr(masks), ptr(deltas),
             ptr(rays), ptr(ws), ptr(im), ptr(mo), M, N, K, T, ptr(gs0), ptr(gr0), None, ptr(gm0), st)
    else:
        call("inerf_composite_rays_train_backward", ptr(gws), ptr(gim), ptr(sigmas), ptr(rgbs), ptr(deltas), ptr(rays), ptr(ws), ptr(im), M, N, T,
             ptr(gs0), ptr(gr0), st)
    assert float((gs0 == 0).float().mean()) > 0.2        # the case really has terminated rays
    nan = float("nan")
    gs1 = torch.full((M,), nan, device=cuda); gr1 = torch.full((M, 3), nan, device=cuda); gm1 = torch.full((M, max(K, 1)), nan, device=cuda)
    call("inerf_composite_rays_with_masks_train_backward_dense", ptr(gws), ptr(gim), ptr(gmo) if K else None, ptr(sigmas), ptr(rgbs),
         ptr(masks) if K else None, ptr(deltas), ptr(rays), ptr(ws), ptr(im), ptr(mo) if K else None, M, N, K, T, ptr(gs1), ptr(gr1),
         ptr(gm1) if K else None, st)
    assert bits_equal(gs1, gs0) and bits_equal(gr1, gr0)
    if K:
        assert bits_equal(gm1, gm0)
        gm2 = torch.full((M, K), nan, device=cuda)       # instance stage: sigma / colour frozen, their gradients left out
        call("inerf_composite_rays_with_masks_train_backward_dense", ptr(gws), ptr(gim), ptr(gmo), ptr(sigmas), ptr(rgbs), ptr(masks),
             ptr(deltas), ptr(rays), ptr(ws), ptr(im), ptr(mo), M, N, K, T, None, None, ptr(gm2), st)
        assert bits_equal(gm2, gm0)


@pytest.mark.parametrize("K", [0, 32])
@pytest.mark.parametrize("n_step", [1, 4, 8])
def test_composite_infer(recorded, cuda, K, n_step):
    from instance_nerf_b200 import raymarching as rm
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = _dev(*make_rays(sc, 48, 48), device=cuda)
    N = o.shape[0]
    bits_t = torch.from_numpy(bits).to(cuda)
    aabb = torch.tensor([-8.0] * 3 + [8.0] * 3, device=cuda)
    nears, fars = rm.near_far_from_aabb(o, d, aabb, 0.2)
    alive = torch.arange(N, dtype=torch.int32, device=cuda)
    rays_t = nears.clone()
    xyzs, dirs, deltas = rm.march_rays(N, n_step, alive, rays_t, o, d, 8.0, bits_t, cascade, 128, nears, fars, 128, False, 1 / 128, 1024)
    M = xyzs.shape[0]
    sigmas, rgbs, masks = _fake_field(M, K, cuda, 3)
    sigmas = sigmas * 20
    st = [torch.zeros(N, device=cuda), torch.zeros(N, device=cuda), torch.zeros(N, 3, device=cuda)]
    a1, t1 = alive.clone(), rays_t.clone()
    if K == 0:
        rm.composite_rays(N, n_step, a1, t1, sigmas, rgbs, deltas, *st, 1e-2)
    else:
        mo1 = torch.zeros(N, K, device=cuda)
        rm.composite_rays_with_masks(N, n_step, K, a1, t1, sigmas, rgbs, masks, deltas, *st, mo1, 1e-2)
        recorded.close("mask_out", mo1, rtol=1e-5, atol=1e-5)
    recorded.exact("alive", a1)                # which rays die: exact
    recorded.exact("rays_t", t1)
    for name, x in zip(("weights_sum", "depth", "image"), st):
        recorded.close(name, x, rtol=1e-5, atol=1e-6)
    out, n_out = rm.compact_alive(a1, N)
    want = a1[a1 >= 0]
    assert int(n_out) == want.shape[0] and torch.equal(out[: want.shape[0]], want)


def _grid_setup(cuda, dtype, B=20000, bound=8.0, seed=0):
    from instance_nerf_b200.gridencoder import GridEncoder
    enc = GridEncoder(desired_resolution=2048 * bound).to(cuda)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        enc.embeddings.copy_(((torch.rand(enc.embeddings.shape, generator=g) - 0.5)).to(cuda))
    x = torch.rand(B, 3, generator=g).to(cuda)
    x[:16] = torch.tensor([0.0, 1.0, 0.5]).to(cuda)     # boundary values
    x[16:24, 0] = 1.5                                     # out of range -> zeros
    table = enc.embeddings.detach().to(dtype).contiguous()
    return enc, x.contiguous(), table


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_grid_encode_forward_backward_bit_exact(recorded, cuda, dtype):
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    enc, x, table = _grid_setup(cuda, dtype)
    B, L, C = x.shape[0], 16, 2
    S = float(np.log2(enc.per_level_scale))
    out1 = torch.empty(B, L * C, device=cuda, dtype=dtype)
    call("inerf_grid_encode_forward", ptr(x), ptr(table), ptr(enc.offsets), ptr(out1), B, 3, C, L, S, 16, None, 0, 0, 0,
         0 if dtype == torch.float32 else 1, 1, stream_ptr(cuda))
    recorded.exact("encoding", out1)              # the reference's [L, B, C] output as [B, L * C]
    assert float(out1[16:24].abs().sum()) == 0.0
    # backward: atomics make the summation order racy in both implementations -> tolerance
    grad = torch.randn(B, L * C, generator=torch.Generator().manual_seed(1)).to(cuda).to(dtype)
    g1 = torch.zeros_like(table)
    call("inerf_grid_encode_backward", ptr(grad), ptr(x), None, ptr(enc.offsets), ptr(g1), B, 3, C, L, S, 16, None, None, 0, 0, 0,
         0 if dtype == torch.float32 else 1, 1, stream_ptr(cuda))
    tol = dict(rtol=1e-4, atol=1e-5) if dtype == torch.float32 else dict(rtol=2e-2, atol=2e-2)
    recorded.close("grad_table", g1.float(), **tol)
    # the generic kernels (any D / C / layout; here the reference's [L, B, C] layout) next to the D=3, C=2 fast path above
    out2 = torch.empty(L, B, C, device=cuda, dtype=dtype)
    call("inerf_grid_encode_forward", ptr(x), ptr(table), ptr(enc.offsets), ptr(out2), B, 3, C, L, S, 16, None, 0, 0, 0,
         0 if dtype == torch.float32 else 1, 0, stream_ptr(cuda))
    assert bits_equal(out2.permute(1, 0, 2).reshape(B, L * C).contiguous(), out1)
    g2 = torch.zeros_like(table)
    call("inerf_grid_encode_backward", ptr(grad.view(B, L, C).permute(1, 0, 2).contiguous()), ptr(x), None, ptr(enc.offsets), ptr(g2), B, 3, C, L,
         S, 16, None, None, 0, 0, 0, 0 if dtype == torch.float32 else 1, 0, stream_ptr(cuda))
    recorded.close("grad_table", g2.float(), **tol)      # the same reference gradient as the fast path's


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_grid_encode_ray_sorted_stream(recorded, cuda, dtype):
    """Samples in marcher order (consecutive samples of a ray in consecutive rows): the fast-path backward reduces runs of
    lanes that fall into the same cell inside the warp before touching the table gradient.  Forward stays bit-exact;
    backward is compared with the reference kernel's output; in fp16, both against the fp32 result of the same scatter."""
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    from instance_nerf_b200 import raymarching as rm
    enc, _, table = _grid_setup(cuda, dtype, B=64)
    sc, cascade, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = _dev(*make_rays(sc, 48, 64), device=cuda)
    aabb = torch.tensor([-8.0] * 3 + [8.0] * 3, device=cuda)
    nears, fars = rm.near_far_from_aabb(o, d, aabb, 0.2)
    xyzs, _, _, _ = rm.march_rays_train(o, d, 8.0, torch.from_numpy(bits).to(cuda), cascade, 128, nears, fars, None, -1, False, -1, True,
                                        1 / 128, 1024)
    x = ((xyzs + 8.0) / 16.0).contiguous()
    B, L, C = x.shape[0], 16, 2
    assert B > 100000
    S = float(np.log2(enc.per_level_scale))
    code = 0 if dtype == torch.float32 else 1
    out1 = torch.empty(B, L * C, device=cuda, dtype=dtype)
    call("inerf_grid_encode_forward", ptr(x), ptr(table), ptr(enc.offsets), ptr(out1), B, 3, C, L, S, 16, None, 0, 0, 0, code, 1, stream_ptr(cuda))
    recorded.exact("encoding", out1)
    grad = (torch.randn(B, L * C, generator=torch.Generator().manual_seed(3)) * 0.01).to(cuda).to(dtype)
    g1 = torch.zeros_like(table)
    call("inerf_grid_encode_backward", ptr(grad), ptr(x), None, ptr(enc.offsets), ptr(g1), B, 3, C, L, S, 16, None, None, 0, 0, 0, code, 1,
         stream_ptr(cuda))
    if dtype == torch.float32:
        recorded.close("grad_table", g1, rtol=1e-3, atol=1e-5)
    else:
        # fp16 table gradients: hundreds of samples land on one coarse entry; the reference adds individually rounded halves in a
        # racy order, the fast path rounds each warp-level run once -> compare both against the fp32 result of the same scatter.
        # e_ref is that error as recorded (helpers.Recorded) for this input.
        g32 = torch.zeros(table.shape, device=cuda, dtype=torch.float32)
        call("inerf_grid_encode_backward", ptr(grad.float()), ptr(x), None, ptr(enc.offsets), ptr(g32), B, 3, C, L, S, 16, None, None, 0, 0, 0,
             0, 1, stream_ptr(cuda))
        e_ours = (g1.float() - g32).abs().max().item()
        e_ref = float(recorded.value("fp16_scatter_error", e_ours))
        assert e_ours <= max(2.0 * e_ref, 2e-3), (e_ours, e_ref)


def test_grid_encoder_module_autograd(cuda):
    """constant table -> output equals the constant (weights sum to 1); gradcheck-style finite difference on the table."""
    from instance_nerf_b200.gridencoder import GridEncoder
    enc = GridEncoder(num_levels=4, base_resolution=4, log2_hashmap_size=8, desired_resolution=32).to(cuda)
    with torch.no_grad():
        enc.embeddings.fill_(0.25)
    x = (torch.rand(257, 3, device=cuda) * 2 - 1)
    y = enc(x, bound=1)
    torch.testing.assert_close(y, torch.full_like(y, 0.25), rtol=1e-5, atol=1e-6)
    with torch.no_grad():
        enc.embeddings.copy_(torch.randn_like(enc.embeddings))
    w = torch.randn(257, 8, device=cuda)
    (enc(x, bound=1) * w).sum().backward()
    g = enc.embeddings.grad.clone()
    idx = torch.randint(0, enc.embeddings.numel(), (20,))
    for i in idx.tolist():
        r, c = divmod(i, 2)
        with torch.no_grad():
            old = enc.embeddings[r, c].item()
            enc.embeddings[r, c] = old + 1e-2
            up = (enc(x, bound=1) * w).sum().item()
            enc.embeddings[r, c] = old - 1e-2
            dn = (enc(x, bound=1) * w).sum().item()
            enc.embeddings[r, c] = old
        assert abs((up - dn) / 2e-2 - g[r, c].item()) < 2e-2 * max(1.0, abs(g[r, c].item()))


def test_sh_bit_exact(recorded, cuda):
    from instance_nerf_b200.shencoder import SHEncoder
    g = torch.Generator().manual_seed(0)
    d = torch.nn.functional.normalize(torch.randn(25600, 3, generator=g), dim=-1).to(cuda)
    for degree in (1, 2, 3, 4):
        y1 = SHEncoder(degree=degree)(d)
        recorded.exact(f"degree_{degree}", y1)


def test_occupancy_ema_pack(recorded, cuda):
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork
    m = NeRFNetwork(bound=8, cuda_ray=True, num_instances=4, density_thresh=10).to(cuda)
    g = torch.Generator().manual_seed(0)
    grid = (torch.rand(m.density_grid.shape, generator=g) * 30 - 3).to(cuda)
    grid[grid < -2] = -1
    tmp = (torch.rand(m.density_grid.shape, generator=g) * 40 - 8).to(cuda)
    m.density_grid.copy_(grid)
    # reference formulation (mask_renderer.py:532-540)
    want = grid.clone()
    valid = (want >= 0) & (tmp >= 0)
    want[valid] = torch.maximum(want[valid] * 0.95, tmp[valid])
    mean = torch.mean(want.clamp(min=0)).item()
    m.ema_update_(tmp, 0.95)
    assert bits_equal(want, m.density_grid)
    assert abs(m.mean_density - mean) < 1e-5 * max(1, abs(mean))
    recorded.exact("bitfield", m.density_bitfield)       # the reference's packbits of `want` at min(mean, 10)


def test_grad_total_variation_vs_reference_kernel(recorded, cuda):
    """inerf_grad_total_variation (gridencoder.h:15, gridencoder.cu:504-642) against the reference kernel on the same points:
    the contributions are identical, colliding points add with atomics in a racy order in both -> 1e-5 relative."""
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    from instance_nerf_b200.gridencoder import GridEncoder
    enc, x, table = _grid_setup(cuda, torch.float32, B=20000)
    L, C = 16, 2
    S = float(np.log2(enc.per_level_scale))
    g1 = torch.zeros_like(table)
    call("inerf_grad_total_variation", ptr(x), ptr(table), ptr(g1), ptr(enc.offsets), 1e-3, x.shape[0], 3, C, L, S, 16, 0, 0, 0, stream_ptr(cuda))
    assert float(g1.abs().sum()) > 0
    recorded.close("grad_table", g1, rtol=1e-5, atol=1e-9)
    # module API (grid.py:163-185): adds into embeddings.grad, needs an existing gradient, maps [-bound, bound] -> [0, 1]
    with pytest.raises(ValueError):
        enc.grad_total_variation(1e-3, inputs=x * 2 - 1, bound=1)
    enc.embeddings.grad = torch.zeros_like(enc.embeddings)
    enc.grad_total_variation(1e-3, inputs=x * 2 - 1, bound=1)
    torch.testing.assert_close(enc.embeddings.grad, g1, rtol=1e-4, atol=1e-8)      # (x*2-1+1)/2 re-rounds a few coordinates
    # 2-D table (the background encoder's shape: D = 2, 4 levels) through the pybind-shaped shim
    import instance_nerf_b200.backend as backend
    e2 = GridEncoder(input_dim=2, num_levels=4, log2_hashmap_size=19, desired_resolution=2048).to(cuda)
    g = torch.Generator().manual_seed(4)
    with torch.no_grad():
        e2.embeddings.copy_((torch.rand(e2.embeddings.shape, generator=g) - 0.5).to(cuda))
    x2 = torch.rand(5000, 2, generator=g).to(cuda)
    S2 = float(np.log2(e2.per_level_scale))
    h1 = torch.zeros_like(e2.embeddings)
    backend.gridencoder.grad_total_variation(x2, e2.embeddings.detach(), h1, e2.offsets, 1e-2, 5000, 2, 2, 4, S2, 16, 0, False)
    recorded.close("grad_table_2d", h1, rtol=1e-5, atol=1e-9)
