"""The hash encode of every fused kernel and of the op-level kernels, bit for bit against the fp16 CPU oracle
(oracle/field_oracle.grid_encode_half), which shares no code with the kernels, at every level class.

`encode4_regs` (field_device.cuh) runs one of three paths per quarter of 4 levels: straight-line dense code, straight-line
hashed code with a power-of-two mask, or the generic per-level path of a mixed quarter, which also holds the `% size` fallback
of a hashed level whose size is not a power of two.  At bound 8 (the benchmark) no quarter is mixed; at bounds 1-3 (the
reference's default is 2) levels 4-7 are one dense level and three hashed ones.  The tests here read the encoder features
the training forwards save (`x0_save`, `xs_save`), the features of the op-level encode, and the table gradient the backward
kernels scatter, and compare each with the oracle; level tables that grid.py never produces (non-power-of-two hashed sizes,
an all-dense quarter above level 3) go in through the C ABI."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import field_oracle as fo
from test_oracle_cpu import LEVEL_CLASSES

pytestmark = pytest.mark.gpu

K = 8
BOUNDS = (1.0, 2.0, 3.0, 8.0)
VD = (0.3, -0.5, 0.8)


def _model(cuda, bound, tables="random"):
    """Instance-stage network at `bound`: tables U(-0.5, 0.5) ("random") or the module's own +-1e-4 initialisation ("init",
    where most fp16 products are subnormal, as in an untrained network)."""
    from instance_nerf_b200 import synthetic
    from instance_nerf_b200.nerf.network_mask import NeRFNetwork
    torch.manual_seed(0)
    m = NeRFNetwork(bound=bound, cuda_ray=True, num_instances=K, density_scale=1.0, density_thresh=10)
    if tables == "random":
        synthetic.randomize_tables(m, 1)
    return m.to(cuda).eval()


def _device_scales(enc, cuda):
    """Level scales as the kernels compute them: exp2f(l * S) on the device (torch.exp2 of a CUDA float32 tensor), then
    * H - 1 with one rounding (exact in float64: H is a power of two)."""
    S = float(np.log2(enc.per_level_scale))
    t = torch.exp2(torch.arange(enc.num_levels, dtype=torch.float32, device=cuda) * S).cpu().numpy()
    return (t.astype(np.float64) * enc.base_resolution - 1.0).astype(np.float32)


def _points(bound, scales, seed=0):
    """float32 [B, 3], B = 128 k + r with r != 0: random points in the box; points on its faces (x01 = 0 or 1); coordinates
    whose x01 * scale + 0.5 is an integer at level 4 (the dense level of the mixed quarter at bounds 1-3: fr = 0, half the
    corners get weight 0) with their fp32 neighbours; points outside the box."""
    rng = np.random.RandomState(seed)
    b = np.float32(bound)
    inside = ((rng.rand(128 * 9, 3) * 2 - 1) * bound).astype(np.float32)
    face = rng.choice(np.array([-b, b], np.float32), size=(64, 3))
    one_face = inside[:96].copy()
    one_face[np.arange(96), rng.randint(0, 3, 96)] = rng.choice(np.array([-b, b], np.float32), size=96)
    # level-4 grid planes: x01 * s4 + 0.5 = k, searched over a few fp32 steps around each plane
    s4 = np.float32(scales[4])
    k = np.arange(1, int(np.ceil(s4)) + 1, dtype=np.float64)
    x = ((k - 0.5) / float(s4) * 2 * bound - bound).astype(np.float32)
    cand = [x]
    for direction in (np.inf, -np.inf):
        y = x
        for _ in range(4):
            y = np.nextafter(y, np.float32(direction)).astype(np.float32)
            cand.append(y)
    cand = np.concatenate(cand)
    pos = fo.fma_f32(fo.x01_like_torch_cuda(cand, bound), s4, 0.5)
    on_plane = cand[pos == np.floor(pos)]
    assert on_plane.size >= 8, "no fp32 coordinate lands on a level-4 grid plane"
    edge = np.unique(np.concatenate([on_plane, np.nextafter(on_plane, np.float32(np.inf)), np.nextafter(on_plane, np.float32(-np.inf))]))
    edge = edge[np.abs(edge) <= b].astype(np.float32)
    planes = rng.choice(edge, size=(256, 3)).astype(np.float32)
    plane_mix = inside[96:352].copy()
    plane_mix[:, rng.randint(0, 3)] = rng.choice(edge, size=256)
    outside = ((rng.rand(40, 3) * 2 - 1) * bound).astype(np.float32)
    outside[np.arange(40), rng.randint(0, 3, 40)] = np.array([1.01, -1.01, 1.5, -2.0], np.float32)[rng.randint(0, 4, 40)] * b
    outside[:2] = [[np.nextafter(b, np.float32(np.inf)), 0, 0], [0, np.nextafter(-b, np.float32(-np.inf)), 0]]
    pts = np.concatenate([inside, face, one_face, planes, plane_mix, outside]).astype(np.float32)
    if pts.shape[0] % 128 == 0:
        pts = pts[:-1]
    return np.ascontiguousarray(pts)


def _assert_bits(got, want, x01, what):
    g = got.detach().cpu().contiguous().numpy().view(np.uint16)
    w = np.ascontiguousarray(want).view(np.uint16)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    bad = np.argwhere(g != w)
    if bad.size:
        r, c = bad[0]
        raise AssertionError(f"{what}: {len(bad)} of {g.size} features differ from the fp16 oracle; first at row {r} level {c // 2} "
                             f"channel {c % 2}: x01 {x01[r].tolist()}, got {got[r, c].item()!r}, want {float(want[r, c])!r}; "
                             f"levels with differences: {sorted(set((bad[:, 1] // 2).tolist()))}")


def _fused_features(desc, x):
    """inerf_field_forward_train -> x0_save[:, :32] (mask-table features) and inerf_field_forward_train_rgb ->
    xs_save[:, :32] (sigma-table features), fp16."""
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    B, dev = x.shape[0], x.device
    d = torch.nn.functional.normalize(torch.tensor(VD, device=dev), dim=0).expand(B, 3).contiguous()
    sig, rgb = torch.empty(B, device=dev), torch.empty(B, 3, device=dev)
    masks = torch.empty(B, K, device=dev)
    x0 = torch.empty(B, 48, dtype=torch.float16, device=dev)
    xs = torch.empty(B, 64, dtype=torch.float16, device=dev)
    call("inerf_field_forward_train", ctypes.byref(desc), ptr(x), ptr(d), B, ptr(sig), ptr(rgb), ptr(masks), ptr(x0), stream_ptr(dev))
    call("inerf_field_forward_train_rgb", ctypes.byref(desc), ptr(x), ptr(d), B, ptr(sig), ptr(rgb), ptr(xs), stream_ptr(dev))
    return x0[:, :32], xs[:, :32]


def _check_fused_features(desc, packed, offsets, scales, bound, x, cuda):
    x01 = fo.x01_like_torch_cuda(x, bound)
    fm, fs = _fused_features(desc, torch.from_numpy(x).to(cuda))
    want_s = fo.grid_encode_half(x01, packed[:, 0:2], offsets, scales)
    want_m = fo.grid_encode_half(x01, packed[:, 2:4], offsets, scales)
    _assert_bits(fs, want_s, x01, "sigma-table features (xs_save)")
    _assert_bits(fm, want_m, x01, "mask-table features (x0_save)")
    return want_s, want_m


# ---- 1. geometry guard ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bound", BOUNDS)
def test_level_classes_of_the_model(cuda, bound):
    """The model's own level table with the device's scales has the quarter classes the CPU suite pins (a mixed quarter at
    bounds 1-3); the device scales are the ones recorded from exp2f in tests/golden/ref_kernels.npz."""
    import os
    m = _model(cuda, bound, "init")
    scales = _device_scales(m.encoder, cuda)
    gk = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_kernels.npz"))
    assert np.array_equal(scales.view(np.uint32), gk[f"enc_scales_b{int(bound)}"].view(np.uint32))
    assert torch.equal(m.encoder.offsets, m.encoder_mask.offsets)
    modes, classes = fo.level_modes(m.encoder.offsets.cpu().numpy(), scales)
    assert ("".join(map(str, modes)), classes) == LEVEL_CLASSES[int(bound)]


# ---- 2. the x01 the kernels compute (`inv2b`) is the one PyTorch computes on the device --------------------------------------
def test_x01_of_torch_cuda_division(cuda):
    """grid.py:149 `(x + bound) / (2 * bound)` on a CUDA tensor at bound 3 (not a power of two) equals fl(fl(x + b) * fl(1 / 2b))
    bit for bit, which is what every fused kernel computes; the CPU division differs in the last bit for many points."""
    g = torch.Generator().manual_seed(2)
    x = (torch.rand(1 << 18, 3, generator=g) * 2 - 1) * 3.0
    x[:4] = torch.tensor([[-3.0, 3.0, 0.0], [1.0, -1.0, 2.5], [2.9999998, -2.9999998, 1e-7], [0.1, 0.2, 0.3]])
    got = ((x.to(cuda) + 3.0) / (2 * 3.0)).cpu().numpy()
    want = fo.x01_like_torch_cuda(x.numpy(), 3.0)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    true_div = (x.numpy() + np.float32(3.0)) / np.float32(6.0)
    assert (true_div != want).mean() > 0.05     # a correctly rounded division differs: this check can tell the two apart


# ---- 3. fused features, bit for bit ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("tables", ["random", "init"])
@pytest.mark.parametrize("bound", BOUNDS)
def test_fused_features_bit_identical_to_fp16_oracle(cuda, bound, tables):
    m = _model(cuda, bound, tables)
    scales = _device_scales(m.encoder, cuda)
    x = _points(bound, scales)
    assert x.shape[0] % 128 != 0
    packed = m._packed_tables().cpu().numpy()
    want_s, _ = _check_fused_features(m._field_desc(), packed, m.encoder.offsets.cpu().numpy(), scales, bound, x, cuda)
    if tables == "init":      # the untrained network: fp16 subnormal features are part of what is compared
        a = np.abs(want_s.astype(np.float32))
        assert ((a > 0) & (a < 2.0 ** -14)).mean() > 0.1


# ---- 4. op-level encode ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bound", [1.0, 2.0, 3.0])
def test_op_level_encode_matches_oracles(cuda, bound):
    """inerf_grid_encode_forward through the D = 3, C = 2 fast path ([B, L*C]) and the generic kernel ([L, B, C]): fp16 bit for
    bit against the fp16 oracle, fp32 within 1e-6 relative of the fp32 oracle."""
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    from instance_nerf_b200.gridencoder import GridEncoder
    enc = GridEncoder(desired_resolution=2048 * bound).to(cuda)
    with torch.no_grad():
        enc.embeddings.copy_((torch.rand(enc.embeddings.shape, generator=torch.Generator().manual_seed(4)) - 0.5).to(cuda))
    scales = _device_scales(enc, cuda)
    x = _points(bound, scales, seed=1)
    x01 = fo.x01_like_torch_cuda(x, bound)
    xd = torch.from_numpy(x01).to(cuda)
    B, L, C = x.shape[0], 16, 2
    S = float(np.log2(enc.per_level_scale))
    offs = enc.offsets.cpu().numpy()
    for dtype, code in ((torch.float16, 1), (torch.float32, 0)):
        table = enc.embeddings.detach().to(dtype).contiguous()
        if dtype == torch.float16:
            want = fo.grid_encode_half(x01, table.cpu().numpy(), offs, scales)
        else:
            want = fo.grid_encode(torch.from_numpy(x01), table.cpu(), offs, enc.per_level_scale, scales=scales).numpy()
        for layout in (1, 0):
            out = torch.empty((B, L * C) if layout else (L, B, C), dtype=dtype, device=cuda)
            call("inerf_grid_encode_forward", ptr(xd), ptr(table), ptr(enc.offsets), ptr(out), B, 3, C, L, S, 16, None, 0, 0, 0, code, layout,
                 stream_ptr(cuda))
            got = out if layout else out.permute(1, 0, 2).reshape(B, L * C)
            if dtype == torch.float16:
                _assert_bits(got, want, x01, f"fp16 encode, layout {layout}")
            else:
                np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-6, atol=2e-7, err_msg=f"fp32 encode, layout {layout}")


# ---- 5. level tables grid.py never produces, through the C ABI --------------------------------------------------------------
def _level_table(offsets, scales, kind):
    """Offsets from the bound-2 geometry with (i) "mode2": hashed levels of non-power-of-two sizes in quarters 1 and 3, or
    (ii) "dense_q1": levels 4-7 enlarged to r1^3 entries, so quarter 1 is all dense.  Every offset stays a multiple of 8
    (grid.py rounds the level sizes so; the backward's 16-byte RED assumes even offsets)."""
    sizes = np.diff(np.asarray(offsets, np.int64))
    if kind == "mode2":
        for l, n in ((6, 3 << 17), (7, 5 << 16), (13, 3 << 17)):
            sizes[l] = n
    else:
        for l in range(4, 8):
            r1 = int(np.ceil(float(scales[l]))) + 2
            sizes[l] = -(-r1 ** 3 // 8) * 8
    offs = np.concatenate([[0], np.cumsum(sizes)])
    assert offs[-1] < 2 ** 31 and not (offs % 8).any()
    modes, classes = fo.level_modes(offs, scales)
    if kind == "mode2":
        assert [modes[l] for l in (6, 7, 13)] == [2, 2, 2] and classes == ["dense", "mixed", "hashed", "mixed"]
    else:
        assert classes == ["dense", "dense", "hashed", "hashed"]
    return offs.astype(np.int32)


def _custom_desc(m, offs, seed, cuda):
    """The model's descriptor with its level table and packed fp16 table replaced -> (desc, packed numpy, keep-alive)."""
    g = torch.Generator().manual_seed(seed)
    packed = ((torch.rand(int(offs[-1]), 4, generator=g) - 0.5)).half().to(cuda)
    offs_d = torch.from_numpy(offs).to(cuda)
    desc = m._field_desc()
    desc.table_packed = packed.data_ptr()
    desc.offsets = offs_d.data_ptr()
    return desc, packed.cpu().numpy(), (packed, offs_d)


@pytest.mark.parametrize("kind", ["mode2", "dense_q1"])
def test_custom_level_tables_fused_features_and_extraction(cuda, kind):
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    bound = 2.0
    m = _model(cuda, bound)
    scales = _device_scales(m.encoder, cuda)
    offs = _level_table(m.encoder.offsets.cpu().numpy(), scales, kind)
    desc, packed, keep = _custom_desc(m, offs, 5, cuda)
    _check_fused_features(desc, packed, offs, scales, bound, _points(bound, scales, seed=2), cuda)
    # inerf_extract_volume with the same tables: bit-identical to inerf_field_forward at the voxel points
    X, Y, Z = 21, 13, 29
    bbox = np.array([-bound] * 3 + [bound] * 3, np.float32)
    n = X * Y * Z
    xyzs = torch.empty(n, 3, device=cuda)
    call("inerf_volume_points", bbox.ctypes.data, X, Y, Z, None, m.cascade, m.grid_size, bound, ptr(xyzs), None, stream_ptr(cuda))
    vd = (np.array(VD) / np.linalg.norm(VD)).astype(np.float32)
    d = torch.from_numpy(vd).to(cuda).expand(n, 3).contiguous()
    s_ref, c_ref, k_ref = torch.empty(n, device=cuda), torch.empty(n, 3, device=cuda), torch.empty(n, K, device=cuda)
    call("inerf_field_forward", ctypes.byref(desc), ptr(xyzs), ptr(d), n, ptr(s_ref), ptr(c_ref), ptr(k_ref), stream_ptr(cuda))
    thr = float(s_ref.median())
    sig, rgb = torch.empty(n, device=cuda), torch.empty(n, 3, device=cuda)
    lab = torch.empty(n, dtype=torch.int32, device=cuda)
    n_live = torch.zeros(1, dtype=torch.int32, device=cuda)
    call("inerf_extract_volume", ctypes.byref(desc), bbox.ctypes.data, X, Y, Z, None, m.cascade, m.grid_size, vd.ctypes.data, thr,
         ptr(sig), ptr(rgb), ptr(lab), None, ptr(n_live), stream_ptr(cuda))
    torch.cuda.synchronize()
    assert int(n_live.item()) == n
    assert torch.equal(sig.view(torch.int32), s_ref.view(torch.int32))
    assert torch.equal(rgb.view(torch.int32), c_ref.view(torch.int32))
    assert torch.equal(lab, torch.where(s_ref >= thr, torch.argmax(k_ref, dim=-1).to(torch.int32) + 1, 0))
    del keep


# ---- 6. backward scatter: indices and weights of the table gradient ---------------------------------------------------------
def _check_scatter(grad, x01, offs, scales, g_known=None, what=""):
    """grad [T, 2] fp32 table gradient of ONE point at x01: its nonzero rows are exactly the oracle's corners with w != 0, and
    within each level every corner row holds fl32(w_c * g_l) (summed over corners that hash to the same row), g_l being the
    level's feature gradient -- given, or recovered from the corner with the largest weight."""
    want_rows = set()
    for l in range(len(offs) - 1):
        idx, w = fo.level_corners_np(x01[None], offs, scales, l)
        idx, w = idx[0], w[0]
        want_rows |= set(idx[w != 0].tolist())
        rows, inv, mult = np.unique(idx, return_inverse=True, return_counts=True)
        for ch in range(2):
            got = grad[rows, ch]

            def expected(g):
                e = np.zeros(len(rows), np.float32)
                for c in range(8):
                    e[inv[c]] = np.float32(e[inv[c]] + np.float32(np.float64(w[c]) * np.float64(g)))
                return e

            if g_known is not None:
                cands = [np.float32(g_known[l, ch])]
            else:
                single = [c for c in range(8) if mult[inv[c]] == 1]
                c0 = max(single, key=lambda c: w[c])
                g0 = np.float32(np.float64(grad[idx[c0], ch]) / np.float64(w[c0]))
                cands = [g0]
                for direction in (np.inf, -np.inf):
                    y = g0
                    for _ in range(3):
                        y = np.nextafter(y, np.float32(direction))
                        cands.append(y)
            ok = False
            for g in cands:
                e = expected(g)
                exact = mult <= 2      # two terms add in either order to the same fp32 sum
                if np.array_equal(e[exact].view(np.uint32), got[exact].view(np.uint32)) and np.allclose(e[~exact], got[~exact], rtol=1e-6, atol=0):
                    ok = True
                    break
            assert ok, f"{what}: level {l} channel {ch}: table gradient {got.tolist()} at rows {rows.tolist()} is not fl32(w * g) " \
                       f"for weights {w.tolist()}"
    got_rows = set(np.flatnonzero((grad != 0).any(axis=1)).tolist())
    assert got_rows == want_rows, f"{what}: rows written but not corners: {sorted(got_rows - want_rows)[:8]}, corners not written: " \
                                  f"{sorted(want_rows - got_rows)[:8]}"


@pytest.mark.parametrize("case", ["b2", "b8", "b2_mode2"])
def test_backward_scatter_matches_oracle_corners(cuda, case):
    """inerf_field_backward_mask, inerf_field_backward_rgb and the op-level inerf_grid_encode_backward with one live row: the
    scatter's indices and weights against the oracle's corners, without trusting level_corners."""
    from instance_nerf_b200._lib import call, lib, ptr, stream_ptr
    bound = 8.0 if case == "b8" else 2.0
    m = _model(cuda, bound)
    scales = _device_scales(m.encoder, cuda)
    offs = m.encoder.offsets.cpu().numpy()
    if case == "b2_mode2":
        offs = _level_table(offs, scales, "mode2")
        desc, _, keep = _custom_desc(m, offs, 6, cuda)
    else:
        desc, keep = m._field_desc(), None
    T = int(offs[-1])
    offs_d = torch.from_numpy(offs).to(cuda)
    # one point in the box; one with x01 * scale + 0.5 an integer on level 4 in every axis (zero weights on the +1 corners)
    s4 = np.float32(scales[4])
    pts = [np.array([0.37, -0.81, 0.52], np.float32) * np.float32(bound)]
    k = np.float64(np.floor(float(s4) * 0.3)) + 0.5
    c = np.float32(k / float(s4) * 2 * bound - bound)
    for _ in range(64):
        if fo.fma_f32(fo.x01_like_torch_cuda(np.array([c]), bound), s4, 0.5)[0] % 1 == 0:
            break
        c = np.nextafter(c, np.float32(np.inf))
    else:
        raise AssertionError("no fp32 coordinate on a level-4 grid plane")
    pts.append(np.array([c, c, c], np.float32))
    gen = torch.Generator().manual_seed(7)
    wb_rgb = torch.empty(int(lib().inerf_field_rgb_bwd_weights_bytes()), dtype=torch.uint8, device=cuda)
    call("inerf_field_pack_weights_rgb_bwd_device", *[ptr(l.weight.detach()) for l in (*m.sigma_net, *m.color_net)], ptr(wb_rgb), stream_ptr(cuda))
    _, wb_mask = m._packed_weights(want_bwd=True)
    for p in pts:
        x01 = fo.x01_like_torch_cuda(p, bound)
        x = torch.from_numpy(p[None]).to(cuda)
        d = torch.nn.functional.normalize(torch.tensor([VD], device=cuda), dim=-1)
        sig, rgb, masks = torch.empty(1, device=cuda), torch.empty(1, 3, device=cuda), torch.empty(1, K, device=cuda)
        x0 = torch.empty(1, 48, dtype=torch.float16, device=cuda)
        xs = torch.empty(1, 64, dtype=torch.float16, device=cuda)
        call("inerf_field_forward_train", ctypes.byref(desc), ptr(x), ptr(d), 1, ptr(sig), ptr(rgb), ptr(masks), ptr(x0), stream_ptr(cuda))
        # instance head
        gt = torch.zeros(T, 2, device=cuda)
        gw = [torch.zeros(64, 47, device=cuda), torch.zeros(64, 64, device=cuda), torch.zeros(K, 64, device=cuda)]
        g_masks = torch.randn(1, K, generator=gen).to(cuda)
        call("inerf_field_backward_mask", ctypes.byref(desc), ptr(wb_mask), ptr(x), ptr(x0), ptr(g_masks), 1, ptr(gt), *[ptr(t) for t in gw],
             stream_ptr(cuda))
        _check_scatter(gt.cpu().numpy(), x01, offs, scales, what=f"backward_mask {case} {p.tolist()}")
        # stage-1 field
        call("inerf_field_forward_train_rgb", ctypes.byref(desc), ptr(x), ptr(d), 1, ptr(sig), ptr(rgb), ptr(xs), stream_ptr(cuda))
        gt = torch.zeros(T, 2, device=cuda)
        gw = [torch.zeros(64, 32, device=cuda), torch.zeros(16, 64, device=cuda), torch.zeros(64, 31, device=cuda),
              torch.zeros(64, 64, device=cuda), torch.zeros(3, 64, device=cuda)]
        g_s, g_c = torch.randn(1, generator=gen).to(cuda), torch.randn(1, 3, generator=gen).to(cuda)
        call("inerf_field_backward_rgb", ctypes.byref(desc), ptr(wb_rgb), ptr(x), ptr(xs), ptr(sig), ptr(rgb), ptr(g_s), ptr(g_c), 1, ptr(gt),
             *[ptr(t) for t in gw], stream_ptr(cuda))
        _check_scatter(gt.cpu().numpy(), x01, offs, scales, what=f"backward_rgb {case} {p.tolist()}")
        # op-level backward (fast path, fp32): the feature gradient is given
        g_feat = torch.randn(1, 32, generator=gen)
        gt = torch.zeros(T, 2, device=cuda)
        xd = torch.from_numpy(x01[None]).to(cuda)
        S = float(np.log2(m.encoder.per_level_scale))
        call("inerf_grid_encode_backward", ptr(g_feat.to(cuda)), ptr(xd), None, ptr(offs_d), ptr(gt), 1, 3, 2, 16, S, 16, None, None, 0, 0, 0, 0, 1,
             stream_ptr(cuda))
        _check_scatter(gt.cpu().numpy(), x01, offs, scales, g_known=g_feat.numpy().reshape(16, 2), what=f"grid_encode_backward {case} {p.tolist()}")
    del keep
