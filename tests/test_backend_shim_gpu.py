"""GPU parity at the FFI boundary itself: `instance_nerf_b200.backend` exposes the reference's pybind prototypes
(raymarching.h:5-22, gridencoder.h:12-15, shencoder.h:9-10); every function is called with the SAME argument list as the
reference's own module, and the caller-allocated outputs are compared with what the reference's module wrote on the same
inputs (tests/golden/recorded_test_backend_shim_gpu.npz, helpers.Recorded)."""
import numpy as np
import pytest
import torch

from helpers import adversarial_rays, canonicalize, make_rays, scene_arrays

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ours():
    import instance_nerf_b200.backend as ours
    return ours


def _scene(cuda, bound=8.0):
    sc, cascade, grid, bits = scene_arrays(16, bound, 0)
    o, d = make_rays(sc, 40, 56)
    ao, ad = adversarial_rays(bound)
    o, d = torch.cat([o, ao]).to(cuda).contiguous(), torch.cat([d, ad]).to(cuda).contiguous()
    return o, d, torch.from_numpy(bits).to(cuda), cascade


def test_raymarching_prototypes(ours, recorded, cuda):
    names = sorted(vars(ours.raymarching))
    assert names == list(recorded.value("exports", names))      # the public names of the reference's _raymarching module
    mod = ours.raymarching
    bound, dt_gamma, max_steps = 8.0, 1 / 128, 512
    o, d, bits, C = _scene(cuda, bound)
    N = o.shape[0]
    aabb = torch.tensor([-bound] * 3 + [bound] * 3, device=cuda)
    nears, fars = torch.empty(N, device=cuda), torch.empty(N, device=cuda)
    mod.near_far_from_aabb(o, d, aabb, N, 0.2, nears, fars)
    coords = torch.empty(N, 2, device=cuda)
    mod.sph_from_ray(o, d, 20.0, N, coords)
    M = N * max_steps
    xyzs, dirs, deltas = torch.zeros(M, 3, device=cuda), torch.zeros(M, 3, device=cuda), torch.zeros(M, 2, device=cuda)
    rays = torch.empty(N, 3, dtype=torch.int32, device=cuda)
    counter = torch.zeros(2, dtype=torch.int32, device=cuda)
    noises = torch.rand(N, generator=torch.Generator().manual_seed(3)).to(cuda)
    mod.march_rays_train(o, d, bits, bound, dt_gamma, max_steps, N, C, 128, M, nears, fars, xyzs, dirs, deltas, rays, counter, noises)
    torch.cuda.synchronize()
    stream = canonicalize(rays, xyzs, dirs, deltas)
    recorded.exact("nears", nears)
    recorded.exact("fars", fars)
    recorded.close("sph_coords", coords, rtol=1e-6, atol=1e-6, equal_nan=True)   # rays that miss the sphere give NaN in both
    recorded.exact("counter", counter)
    for name, a in zip(("rays", "xyzs", "dirs", "deltas"), stream):
        recorded.exact(name, a)

    # compositing (train) with and without masks, forward + backward, same canonical stream
    crays, cx, cd, cl = stream
    total, K = cx.shape[0], 7
    g = torch.Generator().manual_seed(5)
    sig = torch.exp(torch.randn(total, generator=g) + 1.5).to(cuda)
    rgb = torch.rand(total, 3, generator=g).to(cuda)
    msk = torch.randn(total, K, generator=g).to(cuda)
    rays_t, dl = torch.from_numpy(crays).to(cuda), torch.from_numpy(cl).to(cuda)
    gws, gim, gmo = torch.randn(N, generator=g).to(cuda), torch.randn(N, 3, generator=g).to(cuda), torch.randn(N, K, generator=g).to(cuda)
    ws, dp, im, mo = (torch.empty(N, device=cuda), torch.empty(N, device=cuda), torch.empty(N, 3, device=cuda), torch.empty(N, K, device=cuda))
    mod.composite_rays_with_masks_train_forward(sig, rgb, msk, dl, rays_t, total, N, K, 1e-4, ws, dp, im, mo)
    gs, gr, gm, acc = torch.zeros(total, device=cuda), torch.zeros(total, 3, device=cuda), torch.zeros(total, K, device=cuda), torch.zeros(N, K, device=cuda)
    mod.composite_rays_with_masks_train_backward(gws, gim, gmo, sig, rgb, msk, dl, rays_t, ws, im, mo, total, N, K, 1e-4, gs, gr, acc, gm)
    ws2, dp2, im2 = torch.empty(N, device=cuda), torch.empty(N, device=cuda), torch.empty(N, 3, device=cuda)
    mod.composite_rays_train_forward(sig, rgb, dl, rays_t, total, N, 1e-4, ws2, dp2, im2)
    gs2, gr2 = torch.zeros(total, device=cuda), torch.zeros(total, 3, device=cuda)
    mod.composite_rays_train_backward(gws, gim, sig, rgb, dl, rays_t, ws2, im2, total, N, 1e-4, gs2, gr2)
    for i, a in enumerate((ws, dp, im, mo, gs, gr, gm, ws2, dp2, im2, gs2, gr2)):
        recorded.close(f"composite_train_{i}", a, rtol=2e-4, atol=2e-5)   # fp32, different summation order inside a ray

    # inference marching + compositing, 2 chunks of n_step = 4
    alive0 = torch.arange(N, dtype=torch.int32, device=cuda)
    alive, rt = alive0.clone(), nears.clone()
    ws, dp, im, mo = torch.zeros(N, device=cuda), torch.zeros(N, device=cuda), torch.zeros(N, 3, device=cuda), torch.zeros(N, K, device=cuda)
    ws1, dp1, im1 = torch.zeros(N, device=cuda), torch.zeros(N, device=cuda), torch.zeros(N, 3, device=cuda)
    alive1, rt1 = alive0.clone(), nears.clone()
    for it in range(2):
        n_step = 4
        na = alive.shape[0]
        x, dd, dl2 = torch.zeros(na * n_step, 3, device=cuda), torch.zeros(na * n_step, 3, device=cuda), torch.zeros(na * n_step, 2, device=cuda)
        mod.march_rays(na, n_step, alive, rt, o, d, bound, dt_gamma, max_steps, C, 128, bits, nears, fars, x, dd, dl2, torch.zeros(na, device=cuda))
        gg = torch.Generator().manual_seed(10 + it)
        s2 = torch.exp(torch.randn(na * n_step, generator=gg) + 2.5).to(cuda)
        c2 = torch.rand(na * n_step, 3, generator=gg).to(cuda)
        m2 = torch.randn(na * n_step, K, generator=gg).to(cuda)
        if it == 0:
            recorded.exact("infer_xyzs", x)
            recorded.exact("infer_deltas", dl2)
        rt1.copy_(rt); alive1 = alive.clone()
        mod.composite_rays_with_masks(na, n_step, K, 1e-2, alive, rt, s2, c2, m2, dl2, ws, dp, im, mo)
        mod.composite_rays(na, n_step, 1e-2, alive1, rt1, s2, c2, dl2, ws1, dp1, im1)
        last = (alive.clone(), alive1.clone())
        alive = alive[alive >= 0].contiguous()      # the reference loop compacts between iterations (mask_renderer.py:370)
    recorded.exact("infer_alive_masks", last[0])
    recorded.exact("infer_alive", last[1])
    for i, a in enumerate((rt, ws, dp, im, mo, ws1, im1)):
        recorded.close(f"infer_{i}", a, rtol=1e-5, atol=1e-6)

    # morton / packbits
    g2 = torch.Generator().manual_seed(0)
    c3 = torch.randint(0, 128, (4099, 3), generator=g2, dtype=torch.int32).to(cuda)
    grid = (torch.rand(2, 128 ** 3, generator=g2) * 12 - 1).to(cuda)
    idx = torch.empty(4099, dtype=torch.int32, device=cuda)
    mod.morton3D(c3, 4099, idx)
    back = torch.empty(4099, 3, dtype=torch.int32, device=cuda)
    mod.morton3D_invert(idx, 4099, back)
    bf = torch.empty(2 * 128 ** 3 // 8, dtype=torch.uint8, device=cuda)
    mod.packbits(grid, bf.shape[0], 4.5, bf)
    recorded.exact("morton", idx)
    recorded.exact("morton_invert", back)
    recorded.exact("packbits", bf)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16])
def test_gridencoder_and_shencoder_prototypes(ours, recorded, cuda, dtype):
    from oracle.field_oracle import level_offsets
    offsets, pls = level_offsets(desired_resolution=2048 * 2)
    T, B, L, C = int(offsets[-1]), 1237, 16, 2
    g = torch.Generator().manual_seed(1)
    table = ((torch.rand(T, C, generator=g) - 0.5)).to(cuda).to(dtype)
    x01 = torch.rand(B, 3, generator=g).to(cuda)
    off = torch.from_numpy(offsets).to(cuda)
    S = float(np.log2(pls))
    grad = torch.randn(L, B, C, generator=g).to(cuda).to(dtype)
    out = torch.empty(L, B, C, device=cuda, dtype=dtype)
    ours.gridencoder.grid_encode_forward(x01, table, off, out, B, 3, C, L, S, 16, None, 0, False, 0)
    gt = torch.zeros(T, C, device=cuda, dtype=dtype)
    ours.gridencoder.grid_encode_backward(grad, x01, table, off, gt, B, 3, C, L, S, 16, None, None, 0, False, 0)
    recorded.exact("encoding", out)                                       # forward: bit-exact in both dtypes
    tol = dict(rtol=1e-5, atol=1e-6) if dtype == torch.float32 else dict(rtol=2e-2, atol=2e-2)   # atomics: summation order differs
    recorded.close("grad_table", gt.float(), **tol)

    if dtype == torch.float32:
        dirs = torch.nn.functional.normalize(torch.randn(777, 3, generator=g), dim=-1).to(cuda)
        gsh = torch.randn(777, 16, generator=g).to(cuda)
        o16 = torch.empty(777, 16, device=cuda)
        dy = torch.empty(777, 48, device=cuda)
        ours.shencoder.sh_encode_forward(dirs, o16, 777, 3, 4, dy)
        gi = torch.zeros(777, 3, device=cuda)
        ours.shencoder.sh_encode_backward(gsh, dirs, 777, 3, 4, dy, gi)
        recorded.exact("sh", o16)
        recorded.close("sh_dy", dy, rtol=1e-6, atol=1e-6)
        recorded.close("sh_grad_inputs", gi, rtol=1e-5, atol=1e-6)
