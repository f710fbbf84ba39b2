"""CPU suite: pins the oracle (oracle/raymarch_oracle.c, oracle/field_oracle.py) against golden vectors produced by
the reference itself -- tests/golden/ref_kernels.npz (the reference's CUDA kernels run on a B200,
make_golden_gpu.py) and tests/golden/ref_run.npz (the reference's Python renderer, make_golden_cpu.py)."""
import os

import numpy as np
import pytest
import torch

from helpers import bits_equal, scene_arrays
from oracle import field_oracle as fo
from oracle import raymarch_oracle as ro

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def gk():
    return np.load(os.path.join(GOLD, "ref_kernels.npz"))


@pytest.mark.parametrize("tag", ["b8", "b3"])
def test_near_far_and_march_stream_bit_exact(gk, tag):
    bound, dt_gamma, max_steps, cascade = gk[f"{tag}_cfg"]
    bound, max_steps, cascade = float(bound), int(max_steps), int(cascade)
    sc, c2, grid, bits = scene_arrays(16, bound, 0)
    assert c2 == cascade
    o, d = gk[f"{tag}_rays_o"], gk[f"{tag}_rays_d"]
    aabb = np.array([-bound] * 3 + [bound] * 3, np.float32)
    nears, fars = ro.near_far_from_aabb(o, d, aabb, 0.2)
    assert bits_equal(nears, gk[f"{tag}_nears"]) and bits_equal(fars, gk[f"{tag}_fars"])
    xyzs, dirs, deltas, rays, counter = ro.march_rays_train(o, d, bits, bound, float(dt_gamma), max_steps, cascade, 128, nears, fars,
                                                           gk[f"{tag}_noises"])
    assert np.array_equal(counter, gk[f"{tag}_counter"])
    assert np.array_equal(rays, gk[f"{tag}_rays"])                       # (ray, offset, count): bit-exact
    assert bits_equal(xyzs, gk[f"{tag}_xyzs"]) and bits_equal(deltas, gk[f"{tag}_deltas"])
    # dirs are the ray direction repeated per sample
    rep = np.repeat(d, rays[:, 2], axis=0)
    assert bits_equal(dirs, rep)


def test_march_budget_drops_tail_rays(gk):
    bound, dt_gamma, max_steps, cascade = gk["b8_cfg"]
    sc, _, grid, bits = scene_arrays(16, 8.0, 0)
    o, d = gk["b8_rays_o"], gk["b8_rays_d"]
    M = 1000
    xyzs, dirs, deltas, rays, counter = ro.march_rays_train(o, d, bits, 8.0, float(dt_gamma), int(max_steps), int(cascade), 128, gk["b8_nears"],
                                                           gk["b8_fars"], gk["b8_noises"], M=M)
    kept = rays[:, 1] + rays[:, 2] <= M
    full = gk["b8_xyzs"]
    for (n, off, cnt), k in zip(rays, kept):
        if cnt and k:
            assert bits_equal(xyzs[off:off + cnt], full[off:off + cnt])
        elif cnt and off < M:
            assert not xyzs[off:min(off + cnt, M)].any()                 # dropped ray: rows stay zero (raymarching.cu:416)


def test_march_rays_inference_bit_exact(gk):
    bound, dt_gamma, max_steps, cascade = gk["b8_cfg"]
    sc, _, grid, bits = scene_arrays(16, 8.0, 0)
    alive = gk["inf_alive"]
    x, dd, dl = ro.march_rays(alive.shape[0], 3, alive, gk["inf_rays_t"], gk["b8_rays_o"], gk["b8_rays_d"], 8.0, float(dt_gamma), int(max_steps),
                              int(cascade), 128, bits, gk["b8_nears"], gk["b8_fars"], np.zeros(alive.shape[0], np.float32))
    assert bits_equal(x, gk["inf_xyzs"]) and bits_equal(dl, gk["inf_deltas"])


def test_morton_packbits(gk):
    assert np.array_equal(ro.morton3D(gk["morton_coords"]), gk["morton_idx"])
    assert np.array_equal(ro.morton3D_invert(gk["morton_idx"]), gk["morton_coords"])
    assert ro.morton3D(np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1]], np.int32)).tolist() == [1, 2, 4]      # known answers
    ii = np.stack(np.meshgrid(*[np.arange(0, 128, 9)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(np.int32)
    assert np.array_equal(ro.morton3D_invert(ro.morton3D(ii)), ii)                                          # invert o encode = id
    assert np.array_equal(ro.packbits(gk["pack_grid"], 5.0), gk["pack_bits"])


def test_composite_forward_backward(gk):
    """fp32 compositing: the device uses __expf (ex2.approx), the CPU expf -> tolerance 1e-5 (stated)."""
    rays, deltas = gk["b8_rays"], gk["b8_deltas"]
    sig, rgb, msk = gk["cmp_sig"], gk["cmp_rgb"], gk["cmp_msk"]
    ws, depth, image, mask_out = ro.composite_rays_train_forward(sig, rgb, msk, deltas, rays, 1e-4)
    np.testing.assert_allclose(ws, gk["cmp_ws"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(depth, gk["cmp_depth"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(image, gk["cmp_image"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(mask_out, gk["cmp_mask_out"], rtol=1e-5, atol=1e-5)
    ws2, _, image2, _ = ro.composite_rays_train_forward(sig, rgb, None, deltas, rays, 1e-4)
    np.testing.assert_allclose(ws2, gk["cmp_ws_plain"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(image2, gk["cmp_image_plain"], rtol=1e-5, atol=1e-6)
    gs, gr, gm = ro.composite_rays_train_backward(gk["cmp_gws"], gk["cmp_gim"], gk["cmp_gmo"], sig, rgb, msk, deltas, rays, gk["cmp_ws"],
                                                  gk["cmp_image"], gk["cmp_mask_out"], 1e-4)
    np.testing.assert_allclose(gr, gk["cmp_gr"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(gm, gk["cmp_gm"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(gs, gk["cmp_gs"], rtol=2e-3, atol=2e-4)


def test_composite_matches_autograd_of_segment_formulation(gk):
    """Independent cross-check (SURVEY.md section 8c): w = alpha * cumprod(1 - alpha) with break-after-accumulate;
    autograd of that formulation gives the backward."""
    rays, deltas = gk["b8_rays"][:40], torch.from_numpy(gk["b8_deltas"])
    sig = torch.from_numpy(gk["cmp_sig"]).double().requires_grad_(True)
    rgb = torch.from_numpy(gk["cmp_rgb"]).double().requires_grad_(True)
    gim = torch.from_numpy(gk["cmp_gim"]).double()
    loss = 0
    for n, off, cnt in rays:
        if cnt == 0:
            continue
        a = 1 - torch.exp(-sig[off:off + cnt] * deltas[off:off + cnt, 0].double())
        T = torch.cumprod(torch.cat([torch.ones(1, dtype=torch.double), 1 - a[:-1]]), 0)
        T_after = T * (1 - a)
        stop = torch.nonzero(T_after < 1e-4)
        last = int(stop[0]) + 1 if len(stop) else cnt
        w = (a * T)[:last]
        loss = loss + ((w[:, None] * rgb[off:off + last]).sum(0) * gim[n]).sum()
    loss.backward()
    M = int(rays[-1, 1] + rays[-1, 2])
    gs, gr, _ = ro.composite_rays_train_backward(np.zeros_like(gk["cmp_gws"]), gk["cmp_gim"], None, gk["cmp_sig"], gk["cmp_rgb"], None,
                                                 gk["b8_deltas"], rays, gk["cmp_ws_plain"], gk["cmp_image_plain"], None, 1e-4)
    np.testing.assert_allclose(gr[:M], rgb.grad.numpy()[:M], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(gs[:M], sig.grad.numpy()[:M], rtol=2e-3, atol=2e-4)


def test_grid_encode_and_sh_against_reference_kernels(gk):
    offsets, pls = fo.level_offsets(desired_resolution=2048 * 2)
    T = int(offsets[-1])
    table = torch.rand(T, 2, generator=torch.Generator().manual_seed(int(gk["enc_table_seed"][0]))) - 0.5
    x01 = torch.from_numpy(gk["enc_x01"])
    out = fo.grid_encode(x01, table, offsets, pls, scales=gk["enc_scales_b2"])
    # fp32, same operation order as the device (FMA emulated in double) -> agreement to the last bits
    np.testing.assert_allclose(out.numpy(), gk["enc_out"], rtol=1e-6, atol=2e-7)
    # with the host's own exp2 a few level scales differ by one ulp: still within 2e-4 (stated)
    np.testing.assert_allclose(fo.grid_encode(x01, table, offsets, pls).numpy(), gk["enc_out"], rtol=0, atol=2e-4)
    assert not out[2].any()                                              # out-of-range input -> zeros
    gt = fo.grid_encode_backward(x01, torch.from_numpy(gk["enc_grad"]), T, offsets, pls, scales=gk["enc_scales_b2"])
    rows = gk["enc_gtab_rows"]
    np.testing.assert_allclose(gt[rows].numpy(), gk["enc_gtab_vals"], rtol=1e-4, atol=1e-6)
    mask = np.ones(T, bool); mask[rows] = False
    assert float(gt[mask].abs().sum()) == 0.0
    sh = fo.sh_encode(torch.from_numpy(gk["sh_dirs"]), 4)
    np.testing.assert_allclose(sh.numpy(), gk["sh_out"], rtol=1e-6, atol=1e-7)


# Level modes of GridEncoder(desired_resolution=2048 * bound) with the device's level scales: 0 dense, 1 hashed.  At bounds 1-3
# level 4 is dense and 5-7 hashed, so every fused kernel runs its mixed-quarter (generic per-level) path on levels 4-7.
LEVEL_CLASSES = {
    1: ("0000011111111111", ["dense", "mixed", "hashed", "hashed"]),
    2: ("0000011111111111", ["dense", "mixed", "hashed", "hashed"]),
    3: ("0000011111111111", ["dense", "mixed", "hashed", "hashed"]),
    8: ("0000111111111111", ["dense", "hashed", "hashed", "hashed"]),
}


@pytest.mark.parametrize("bound", sorted(LEVEL_CLASSES))
def test_level_classes_from_recorded_scales(gk, bound):
    offsets, _ = fo.level_offsets(desired_resolution=2048 * bound)
    modes, classes = fo.level_modes(offsets, gk[f"enc_scales_b{bound}"])
    assert ("".join(map(str, modes)), classes) == LEVEL_CLASSES[bound]


def test_fma_f32_rounds_once():
    """pos = fmaf(x01, scale, 0.5): a * b = 2^-25 + 2^-57 (641 * 6700417 = 2^32 + 1) puts the float64 sum exactly on the float32
    midpoint 0.5 + 2^-25; the exact value lies above it, so one rounding gives 0.5 + 2^-24 where float64-then-float32 gives 0.5."""
    a, b = np.float32(641 * 2.0 ** -30), np.float32(6700417 * 2.0 ** -27)
    assert np.float32(float(a) * float(b) + 0.5) == np.float32(0.5)
    assert fo.fma_f32(np.array([a]), b, 0.5)[0] == np.float32(0.5 + 2.0 ** -24)
    assert fo.fma_f32(np.array([-a]), b, 0.5)[0] == np.float32(0.5 - 2.0 ** -25)
    x = np.random.RandomState(0).rand(10000).astype(np.float32)
    assert np.array_equal(fo.fma_f32(x, np.float32(47.502937), 0.5), (x.astype(np.float64) * float(np.float32(47.502937)) + 0.5).astype(np.float32))


def _f16_error_bound(x01, table, offsets, scales):
    """|fp16 encode - exact| <= 16 half-ulps of the largest partial sum: 8 product roundings + 8 accumulation roundings."""
    big = np.abs(fo.grid_encode(torch.from_numpy(x01), torch.from_numpy(np.abs(table)), offsets, 2.0, scales=scales).numpy())
    return 16 * 2.0 ** -11 * np.maximum(big, 2.0 ** -14)


def test_grid_encode_half_matches_reference_kernel_fp32(gk):
    """The fp16 oracle on the reference kernel's bound-2 inputs against the reference's fp32 output: within fp16 error, so its
    corner indices and weights are the reference's at bound 2 (dense, mixed and hashed quarters)."""
    offsets, _ = fo.level_offsets(desired_resolution=2048 * 2)
    T = int(offsets[-1])
    table = (torch.rand(T, 2, generator=torch.Generator().manual_seed(int(gk["enc_table_seed"][0]))) - 0.5).numpy()
    x01, scales = gk["enc_x01"], gk["enc_scales_b2"]
    h = fo.grid_encode_half(x01, table.astype(np.float16), offsets, scales)
    assert h.dtype == np.float16 and h.shape == gk["enc_out"].shape
    err = np.abs(h.astype(np.float64) - gk["enc_out"])
    assert (err <= _f16_error_bound(x01, table, offsets, scales)).all(), float(err.max())
    assert float(err.mean()) < 1e-4
    assert not h[2].any()                                                 # out-of-range input -> zeros


def test_grid_encode_half_non_power_of_two_hashed_levels(gk):
    """Hashed levels whose size is not a power of two (mode 2: `% size`) inside the mixed quarter and a hashed one: the fp16
    oracle against the fp32 one, within fp16 error."""
    offsets, pls = fo.level_offsets(desired_resolution=2048 * 2)
    scales = gk["enc_scales_b2"]
    sizes = np.diff(offsets.astype(np.int64))
    for l, n in ((6, 3 << 17), (7, 5 << 16), (13, 3 << 17)):
        sizes[l] = n
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    modes, classes = fo.level_modes(offs, scales)
    assert [modes[l] for l in (4, 5, 6, 7, 13)] == [0, 1, 2, 2, 2] and classes == ["dense", "mixed", "hashed", "mixed"]
    g = torch.Generator().manual_seed(11)
    table = ((torch.rand(int(offs[-1]), 2, generator=g) - 0.5).numpy()).astype(np.float16)
    x01 = torch.rand(2000, 3, generator=g).numpy()
    h = fo.grid_encode_half(x01, table, offs, scales)
    ref = fo.grid_encode(torch.from_numpy(x01), torch.from_numpy(table.astype(np.float32)), offs, pls, scales=scales).numpy()
    err = np.abs(h.astype(np.float64) - ref)
    assert (err <= _f16_error_bound(x01, table.astype(np.float32), offs, scales)).all(), float(err.max())
    # the `% size` levels really differ from a power-of-two mask of the same size
    idx, _ = fo.level_corners_np(x01, offs, scales, 6)
    rel = idx - offs[6]
    assert (rel < sizes[6]).all() and (rel >= 1 << 18).any()


def test_grid_encode_constant_table_and_gradcheck():
    """Analytic checks of SURVEY.md section 8c: constant table -> constant output; fp64 finite differences."""
    offsets, pls = fo.level_offsets(num_levels=4, base_resolution=4, log2_hashmap_size=8, desired_resolution=32)
    T = int(offsets[-1])
    x01 = torch.rand(64, 3, generator=torch.Generator().manual_seed(0))
    out = fo.grid_encode(x01, torch.full((T, 2), 0.25), offsets, pls, 4)
    np.testing.assert_allclose(out.numpy(), 0.25, rtol=1e-6)
    table = torch.randn(T, 2, generator=torch.Generator().manual_seed(1))
    w = torch.randn(64, 8, generator=torch.Generator().manual_seed(2))
    g = fo.grid_encode_backward(x01, w, T, offsets, pls, 4)
    for r, c in [(0, 0), (5, 1), (40, 0), (T - 9, 1)]:
        tp, tm = table.clone(), table.clone()
        tp[r, c] += 1e-2; tm[r, c] -= 1e-2
        fd = ((fo.grid_encode(x01, tp, offsets, pls, 4) * w).sum() - (fo.grid_encode(x01, tm, offsets, pls, 4) * w).sum()) / 2e-2
        assert abs(fd.item() - g[r, c].item()) < 1e-3 * max(1, abs(fd.item()))


def test_oracle_run_matches_reference_python_renderer():
    g = np.load(os.path.join(GOLD, "ref_run.npz"))
    K, bound, H, W, T, seed = g["cfg"]
    K, T = int(K), int(T)
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")}
    gen = torch.Generator().manual_seed(int(seed))
    n_rows = int(sd["encoder.offsets"][-1])
    for name in ("encoder.embeddings", "encoder_mask.embeddings"):
        sd[name] = (torch.rand(n_rows, 2, generator=gen) * 2 - 1) * 0.5
    field = fo.OracleField(sd, float(bound), K)
    o, d = torch.from_numpy(g["rays_o"]), torch.from_numpy(g["rays_d"])
    res = field.render(o[None], d[None], max_ray_batch=100, render_mask=True, num_steps=T, bg_color=1)
    np.testing.assert_allclose(res["image"].numpy(), g["image"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(res["depth"].numpy(), g["depth"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(res["instance_mask_logits"].numpy(), g["logits"], rtol=1e-4, atol=1e-5)


def test_update_grid_ema_restatement():
    rng = np.random.RandomState(0)
    grid = (rng.rand(2, 4096) * 30 - 3).astype(np.float32); grid[grid < -2] = -1
    tmp = (rng.rand(2, 4096) * 40 - 8).astype(np.float32)
    g, mean, bits = fo.update_grid_ema(grid, tmp, 0.95, 10.0)
    valid = (grid >= 0) & (tmp >= 0)
    assert np.array_equal(g[~valid], grid[~valid])
    assert np.all(g[valid] >= tmp[valid]) and np.all(g[valid] >= grid[valid] * np.float32(0.95))
    assert np.array_equal(bits, ro.packbits(g, min(mean, 10.0)))


def test_extra_state_sweep_points_restatement():
    """oracle/field_oracle.extra_state_sweep_points (mask_renderer.py:470-494) against the literal construction: build the
    whole meshgrid block as the reference does, index it through the C oracle's Morton codes, pick the same cells."""
    G, bound = 32, 8.0
    ii = np.arange(G, dtype=np.int32)
    X, Y, Z = np.meshgrid(ii, ii, ii, indexing="ij")                        # custom_meshgrid(xs, ys, zs)
    coords = np.stack([X.reshape(-1), Y.reshape(-1), Z.reshape(-1)], -1)     # [G^3, 3], row = (x * G + y) * G + z
    indices = ro.morton3D(coords).astype(np.int64)                           # raymarching.morton3D(coords)
    assert np.array_equal(ro.morton3D_invert(indices.astype(np.int32)), coords)
    noise = np.random.RandomState(3).rand(G ** 3, 3).astype(np.float32)
    xyzs = (2 * coords.astype(np.float32) / (G - 1) - 1).astype(np.float32)
    for cas in (0, 2, 3):
        b = min(2 ** cas, bound)
        hgs = b / G
        cas_xyzs = xyzs * np.float32(b - hgs) + (noise * 2 - 1) * np.float32(hgs)     # :485-489
        by_cell = np.empty_like(cas_xyzs)
        by_cell[indices] = cas_xyzs                                          # what tmp_grid[cas, indices] = sigma(cas_xyzs) pairs up
        cells = np.random.RandomState(cas).randint(0, G ** 3, size=500)
        got = fo.extra_state_sweep_points(cells, cas, G, bound, noise)
        np.testing.assert_allclose(got, by_cell[cells], rtol=0, atol=1e-6)


# ---------------------------------------------------------------------------------------------------------------------
# oracle/host_oracle.py against tests/golden/ref_host.npz = the reference's own host-side functions run on the CPU
# (tests/golden/make_golden_host.py): get_rays, MaskTrainer.train_step's loss, mark_untrained_grid, update_extra_state.
def _host_gold():
    return np.load(os.path.join(GOLD, "ref_host.npz"))


def _gold_model_sd(g):
    """State dict of the golden's reference network: small tensors stored, both hash tables regenerated from the seed."""
    K, bound, seed = g["model_cfg"]
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")}
    gen = torch.Generator().manual_seed(int(seed))
    n_rows = int(sd["encoder.offsets"][-1])
    for name in ("encoder.embeddings", "encoder_mask.embeddings"):
        sd[name] = (torch.rand(n_rows, 2, generator=gen) * 2 - 1) * 0.5
    return sd, int(K), float(bound)


@pytest.mark.parametrize("case", ["full", "uniform", "patch", "emap"])
def test_host_oracle_get_rays_matches_reference(case):
    from instance_nerf_b200 import synthetic
    from oracle import host_oracle as ho
    g = _host_gold()
    B, H, W, N, patch, seed, emap = (int(v) for v in g[f"rays_{case}_cfg"])
    poses = torch.from_numpy(g["poses"])[:B]
    error_map = ((torch.arange(B * 128 * 128) % 97).float() + 1).view(B, -1) / 97.0 if emap else None
    r = ho.get_rays(poses, synthetic.intrinsics(H, W), H, W, N, error_map=error_map, patch_size=patch, generator=torch.Generator().manual_seed(seed))
    for k in ("rays_o", "rays_d", "inds", "inds_coarse"):
        if f"rays_{case}_{k}" in g.files:
            assert np.array_equal(r[k].contiguous().numpy(), g[f"rays_{case}_{k}"]), (case, k)
        else:
            assert k not in r


def test_host_oracle_mask_loss_matches_reference_train_step():
    from oracle import host_oracle as ho
    g = _host_gold()
    K, patch = int(g["model_cfg"][0]), int(g["loss_patch"])
    depth, labels = torch.from_numpy(g["loss_depth"]), torch.from_numpy(g["loss_labels"])
    m3_logits, m3_labels = torch.from_numpy(g["m3_logits"]), torch.from_numpy(g["m3_labels"])
    for tag in ("ce", "reg", "all"):
        want, reg_w, m3_w = g[f"loss_{tag}"]
        logits = torch.from_numpy(g["loss_logits"]).clone().requires_grad_(True)
        loss = ho.mask_train_loss(logits, depth, labels, patch, K, float(reg_w), m3_logits, m3_labels, float(m3_w))
        (grad,) = torch.autograd.grad(loss, logits)
        assert abs(float(loss) - float(want)) < 1e-6 * max(1.0, abs(float(want))), tag
        np.testing.assert_allclose(grad.numpy(), g[f"loss_{tag}_grad"], rtol=1e-5, atol=1e-8)
    assert abs(float(ho.mask_train_loss(torch.from_numpy(g["loss_logits"]), depth, torch.full_like(labels, -1), patch, K, 0.0)) - float(g["loss_unlabelled"])) == 0.0
    np.testing.assert_allclose(float(torch.nn.functional.cross_entropy(m3_logits, m3_labels)), float(g["m3_loss"]), rtol=1e-6)


def test_host_oracle_mask3d_logits_match_reference_network():
    """The 3D-mask query (nerf/utils.py:1250-1260: density -> geo_feat -> mask) through the oracle field vs the reference net."""
    g = _host_gold()
    sd, K, bound = _gold_model_sd(g)
    field = fo.OracleField(sd, bound, K)
    x = torch.from_numpy(g["m3_coords"])
    with torch.no_grad():
        logits = field.mask(x, geo_feat=field.density(x)["geo_feat"])
    np.testing.assert_allclose(logits.numpy(), g["m3_logits"], rtol=1e-4, atol=1e-5)


def test_host_oracle_occupancy_update_matches_reference():
    """Full sweep and partial update of update_extra_state with the reference's recorded draws: the restated sample points
    are bit-identical, the EMA / mean / packbits tail (field_oracle.update_grid_ema) reproduces grid, mean and bitfield."""
    from oracle import host_oracle as ho
    g = _host_gold()
    C, G, bound = int(g["occ_cfg"][0]), int(g["occ_cfg"][1]), float(g["occ_cfg"][2])
    ii = np.arange(G, dtype=np.int32)
    X, Y, Z = np.meshgrid(ii, ii, ii, indexing="ij")
    mesh = np.stack([X.ravel(), Y.ravel(), Z.ravel()], -1)
    for tag in ("full", "partial"):
        tmp = -np.ones((C, G ** 3), np.float32)
        for c in range(C):
            if tag == "full":
                coords, indices = mesh, ro.morton3D(mesh).astype(np.int64)
            else:
                indices, coords = ho.partial_cells(g["occ_partial_grid_in"][c], g["occ_partial_coords"][c], g["occ_partial_picks"][c])
            pts = ho.sweep_points(coords, c, G, bound, g[f"occ_{tag}_noise"][c])
            assert np.array_equal(pts.view(np.uint32), g[f"occ_{tag}_points"][c].view(np.uint32)), (tag, c)
            tmp[c, indices] = g[f"occ_{tag}_sigma"][c]      # density_scale = 1; duplicates: last write wins, as index_put on the CPU
        grid, mean, bits = fo.update_grid_ema(g[f"occ_{tag}_grid_in"], tmp, 0.95, 0.5)
        assert np.array_equal(grid.view(np.uint32), g[f"occ_{tag}_grid_out"].view(np.uint32)), tag
        assert abs(mean - float(g[f"occ_{tag}_mean"])) < 1e-6 * max(1.0, mean)
        assert np.array_equal(bits, g[f"occ_{tag}_bits"]), tag
    # the recorded densities are the reference network's: the oracle field reproduces them at the recorded points
    sd, K, b = _gold_model_sd(g)
    field = fo.OracleField(sd, b, K)
    with torch.no_grad():
        sig = field.density(torch.from_numpy(g["occ_partial_points"][1]))["sigma"]
    np.testing.assert_allclose(sig.numpy(), g["occ_partial_sigma"][1], rtol=1e-4, atol=1e-6)


def test_host_oracle_mark_untrained_grid_matches_reference():
    from oracle import host_oracle as ho
    g = _host_gold()
    C, G, bound = int(g["occ_cfg"][0]), int(g["occ_cfg"][1]), float(g["occ_cfg"][2])
    got = ho.mark_untrained_grid(np.zeros((C, G ** 3), np.float32), g["mark_poses"], tuple(g["mark_intr"]), bound, G)
    want = g["mark_grid"]
    assert 0 < int((want == -1).sum()) < want.size
    assert np.array_equal(got, want)


def test_checkpoint_layout_matches_reference_and_round_trips(tmp_path):
    """nerf/checkpoint.py against the reference's checkpoint contents: the product network's state dict has exactly the
    names / shapes / dtypes of the REFERENCE network's (recorded from the reference class in tests/golden/ref_host.npz), a
    checkpoint in the reference trainer's dict layout (nerf/utils.py:1100-1140) loads strictly, and save -> load round-trips."""
    import json
    from instance_nerf_b200.nerf import checkpoint
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork
    g = _host_gold()
    layout = json.loads(str(g["ref_sd_layout"]))
    K, bound, _ = g["model_cfg"]
    m = NeRFNetwork(bound=float(bound), cuda_ray=True, num_instances=int(K), density_scale=1, density_thresh=0.5)
    ours = [[k, list(v.shape), str(v.dtype)] for k, v in m.state_dict().items()]
    assert sorted(ours) == sorted(layout)
    # a reference-trainer checkpoint: {'epoch', 'global_step', 'stats', 'mean_count', 'mean_density', 'model'}
    gen = torch.Generator().manual_seed(3)
    ref_sd = {k: (torch.rand(shape, generator=gen) if "float" in dt else torch.zeros(shape, dtype=getattr(torch, dt.split(".")[1])))
              for k, shape, dt in layout}
    path = tmp_path / "ngp_ep0003.pth"
    torch.save({"epoch": 3, "global_step": 300, "stats": {"loss": [1.0]}, "mean_count": 4242, "mean_density": 0.25, "model": ref_sd}, path)
    r = checkpoint.load_checkpoint(str(path), m)
    assert r["missing_keys"] == [] and r["unexpected_keys"] == [] and r["epoch"] == 3 and r["global_step"] == 300
    assert m.mean_count == 4242 and m.mean_density == 0.25
    for k, v in m.state_dict().items():
        assert torch.equal(v, ref_sd[k]), k
    # "best" checkpoints drop density_grid (utils.py:1150-1152)
    p2 = tmp_path / "best.pth"
    checkpoint.save_checkpoint(str(p2), m, epoch=4, global_step=400, best=True)
    m2 = NeRFNetwork(bound=float(bound), cuda_ray=True, num_instances=int(K))
    r2 = checkpoint.load_checkpoint(str(p2), m2, model_only=True)
    assert r2["missing_keys"] == ["density_grid"] and r2["unexpected_keys"] == []
    assert torch.equal(m2.encoder_mask.embeddings, m.encoder_mask.embeddings) and m2.mean_count == 4242


def test_dense_renderer_helpers_known_answers():
    """nerf/renderer.py helpers of the dense (non-cuda_ray) path (mask_renderer.py:13-47, 131-137): closed forms on the CPU.
    (The whole `run()` is compared with the reference's renderer on the GPU, tests/test_field_gpu.py.)"""
    from instance_nerf_b200.nerf.renderer import alpha_weights, sample_pdf
    # constant density: w_i = (1 - a) a'^i with a = exp(-delta sigma), up to the 1e-15 guard
    z = torch.linspace(1.0, 2.0, 11).repeat(3, 1)
    sigma = torch.full((3, 11), 2.0)
    w, deltas = alpha_weights(z, torch.full((3, 1), 0.1), sigma, density_scale=1.5)
    a = torch.exp(torch.tensor(-0.1 * 1.5 * 2.0))
    want = (1 - a) * a ** torch.arange(11, dtype=torch.float32)
    torch.testing.assert_close(w[0], want, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(deltas[1], torch.full((11,), 0.1), rtol=1e-5, atol=1e-6)
    assert float(w.sum(-1)[0]) < 1.0
    # uniform pdf over equal bins + deterministic u: the samples are u mapped linearly onto [bins[0], bins[-1]]
    bins = torch.linspace(0.0, 1.0, 9).repeat(2, 1)
    s = sample_pdf(bins, torch.ones(2, 8), 16, det=True)
    torch.testing.assert_close(s[0], torch.linspace(0.5 / 16, 1 - 0.5 / 16, 16), rtol=0, atol=1e-5)
    # all the mass in one bin: every sample falls inside it
    wts = torch.full((1, 8), 0.0)
    wts[0, 5] = 1.0
    s = sample_pdf(bins[:1], wts, 32, det=True)
    inside = (s >= bins[0, 5] - 1e-4) & (s <= bins[0, 6] + 1e-4)
    assert float(inside.float().mean()) > 0.9 and bool((s[0, 1:] >= s[0, :-1]).all())
    torch.manual_seed(0)
    r = sample_pdf(bins, torch.rand(2, 8) + 0.1, 64, det=False)
    assert r.shape == (2, 64) and float(r.min()) >= 0.0 and float(r.max()) <= 1.0
