"""Volume extraction (NeRFRenderer.extract_volume -> inerf_volume_points / inerf_extract_volume) on the GPU: the voxel points,
the fused kernel against the fused field forward on the same points (bit for bit), occupancy gating, the modular fallback,
the stage-1 network, no host sync, and the label volume projected into views against the C oracle."""
import numpy as np
import pytest
import torch

from helpers import bits_equal
from test_field_gpu import build_model

pytestmark = pytest.mark.gpu

SUB = (-2.9, -1.45, -2.4, 2.5, 1.3, 2.2)     # a sub-box of the synthetic room (bound 8; scaled by bound / 8 at other bounds)
SHAPE = (37, 20, 53)                          # non-cubic, no axis a multiple of 4 or 8
VD = tuple(float(v) for v in (np.array([0.3, -0.5, 0.8]) / np.linalg.norm([0.3, -0.5, 0.8])).astype(np.float32))


def _points(m, shape, bbox, bits=True):
    """inerf_volume_points -> (xyzs [n, 3], occupied [n] bool)"""
    from instance_nerf_b200._lib import call, ptr, stream_ptr
    X, Y, Z = shape
    dev = m.aabb_infer.device
    xyzs = torch.empty(X * Y * Z, 3, dtype=torch.float32, device=dev)
    occ = torch.empty(X * Y * Z, dtype=torch.uint8, device=dev)
    bb = np.ascontiguousarray(bbox, dtype=np.float32)
    call("inerf_volume_points", bb.ctypes.data, X, Y, Z, ptr(m.density_bitfield) if bits else None, m.cascade, m.grid_size,
         float(m.bound), ptr(xyzs), ptr(occ), stream_ptr(dev))
    return xyzs, occ.bool()


def test_volume_points_formula(cuda):
    from instance_nerf_b200.projection import voxel_points
    m, _ = build_model(cuda, 4)
    xyzs, occ = _points(m, SHAPE, SUB)
    b = np.asarray(SUB, np.float32)
    lo, hi = b[:3], b[3:]
    axes = [lo[a] + (np.arange(n, dtype=np.float32) / np.float32(n)) * (hi[a] - lo[a]) for a, n in enumerate(SHAPE)]   # fp32, IEEE
    ref = np.stack(np.meshgrid(*axes, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    assert bits_equal(xyzs, ref)
    np.testing.assert_allclose(xyzs.cpu().numpy().astype(np.float64), voxel_points(SHAPE, SUB), rtol=0, atol=1e-6 * m.bound)
    _, all_live = _points(m, SHAPE, SUB, bits=False)
    assert bool(all_live.all()) and 0 < int(occ.sum()) < occ.numel()


def _expected(m, xyzs, thr):
    s, c, k = m.forward_fused(xyzs, torch.tensor(VD, device=xyzs.device).expand(xyzs.shape[0], 3).contiguous())
    s = s * float(m.density_scale)
    lab = torch.where(s >= thr, torch.argmax(k, dim=-1).to(torch.int32) + 1, 0)
    return s, c, lab


@pytest.mark.parametrize("K,density_scale,bound", [(32, 1.0, 8.0), (16, 25.0, 8.0), (2, 1.0, 8.0), (48, 1.0, 8.0), (16, 25.0, 2.0)],
                         ids=["32-1.0", "16-25.0", "2-1.0", "48-1.0", "16-25.0-bound2"])
def test_dense_bit_identical_to_field_forward(cuda, K, density_scale, bound):
    m, _ = build_model(cuda, K, bound=bound, density_scale=density_scale)
    sub = tuple(v * bound / 8 for v in SUB)
    xyzs, _ = _points(m, SHAPE, sub)
    s_ref = m.forward_fused(xyzs, torch.tensor(VD, device=cuda).expand(xyzs.shape[0], 3).contiguous(), want_masks=False)[0]
    thr = float((s_ref * density_scale).median())       # both sides of the label test are populated
    v = m.extract_volume(SHAPE, bbox=sub, view_dir=VD, sigma_thresh=thr, skip_empty=False)
    s, c, lab = _expected(m, xyzs, thr)
    assert v["sigma"].shape == SHAPE and v["rgb"].shape == (*SHAPE, 3) and v["label"].shape == SHAPE and v["label"].dtype == torch.int32
    assert bits_equal(v["sigma"].view(-1), s)
    assert bits_equal(v["rgb"].view(-1, 3), c)
    assert torch.equal(v["label"].view(-1), lab)
    assert int(v["n_live"].item()) == xyzs.shape[0]
    assert 0.3 < float((lab > 0).float().mean()) < 0.7 and len(torch.unique(lab)) > min(K, 3)


def test_occupancy_gating(cuda):
    m, sc = build_model(cuda, 32)
    thr = 1.0
    xyzs, occ = _points(m, SHAPE, SUB)
    g = m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=thr)
    d = m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=thr, skip_empty=False)
    gs, gc, gl = g["sigma"].view(-1), g["rgb"].view(-1, 3), g["label"].view(-1)
    assert int(g["n_live"].item()) == int(occ.sum())
    assert bool((gs[~occ] == 0).all()) and bool((gc[~occ] == 0).all()) and bool((gl[~occ] == 0).all())
    assert bits_equal(gs[occ], d["sigma"].view(-1)[occ])
    assert bits_equal(gc[occ], d["rgb"].view(-1, 3)[occ])
    assert torch.equal(gl[occ], d["label"].view(-1)[occ])

    # independently of the device cell lookup: deep inside a solid -> live, far from every solid -> empty.  The analytic grid
    # marks a cell when its box touches a solid; the coarsest cell these points use is 2 * 4 / 128 (|p| < 4: cascade <= 2).
    p = xyzs.cpu().numpy().astype(np.float64)
    live = occ.cpu().numpy()
    margin = 2 * 8.0 / 128 * 1.01
    inside_deep = np.zeros(len(p), bool)
    near_any = np.zeros(len(p), bool)
    for _, lo, hi in sc.solids:
        inside_deep |= np.all((p - lo > margin) & (hi - p > margin), axis=1)
        near_any |= np.max(np.maximum(np.maximum(lo - p, p - hi), 0.0), axis=1) <= margin
    assert inside_deep.sum() > 100 and (~near_any).sum() > 100
    assert live[inside_deep].all()
    assert not live[~near_any].any()

    # an all-ones bitfield evaluates every voxel: bit-identical to skip_empty=False
    m.density_bitfield.fill_(255)
    a = m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=thr)
    for key in ("sigma", "rgb", "label"):
        assert bits_equal(a[key], d[key]), key
    assert int(a["n_live"].item()) == int(np.prod(SHAPE))


def test_fallback_matches_fused(cuda):
    """The modular path (inerf_volume_points -> forward under fp16 autocast -> torch rules) that serves networks without the
    fused kernel, against the fused kernel: within the tolerances of test_field_fused_vs_modular."""
    m, _ = build_model(cuda, 16, density_scale=25.0)
    thr = 5.0
    f = m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=thr)
    m.use_fused = False
    try:
        r = m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=thr, chunk=10000)
    finally:
        m.use_fused = True
    assert torch.equal(f["n_live"], r["n_live"])
    torch.testing.assert_close(f["sigma"], r["sigma"], rtol=2e-2, atol=1e-3 * 25.0)
    torch.testing.assert_close(f["rgb"], r["rgb"], rtol=0, atol=2e-3)
    agree = float((f["label"] == r["label"]).float().mean())
    assert agree >= 0.99, agree
    assert float((f["label"] > 0).float().mean()) > 0.05


def test_stage1_network(cuda):
    from helpers import scene_arrays
    from instance_nerf_b200 import synthetic
    from instance_nerf_b200.nerf.network import NeRFNetwork
    torch.manual_seed(0)
    m = NeRFNetwork(bound=8.0, cuda_ray=True, density_scale=3.0, density_thresh=10)
    synthetic.randomize_tables(m, 0)
    _, _, grid, bits = scene_arrays(16, 8.0, 0)
    with torch.no_grad():
        m.density_grid.copy_(torch.from_numpy(grid)); m.density_bitfield.copy_(torch.from_numpy(bits))
    m = m.to(cuda).eval()
    with pytest.raises(ValueError):
        m.extract_volume(8)
    v = m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=1.0, skip_empty=False, labels=False)
    assert "label" not in v
    xyzs, _ = _points(m, SHAPE, SUB)
    with torch.no_grad():
        s, c = m(xyzs, torch.tensor(VD, device=cuda).expand(xyzs.shape[0], 3).contiguous())
    assert bits_equal(v["sigma"].view(-1), s * 3.0)
    assert bits_equal(v["rgb"].view(-1, 3), c)


def test_fused_call_does_not_sync(cuda):
    m, _ = build_model(cuda, 32)
    m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=1.0)      # packs tables / weights, loads the module
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        v = m.extract_volume(SHAPE, bbox=SUB, view_dir=VD, sigma_thresh=1.0)
        w = m.extract_volume(SHAPE, bbox=SUB, sigma_thresh=1.0, skip_empty=False)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert isinstance(v["n_live"], torch.Tensor) and v["n_live"].is_cuda
    assert "rgb" not in w and int(w["n_live"].item()) == int(np.prod(SHAPE))


def test_label_volume_projects_like_the_oracle(cuda):
    from oracle import raymarch_oracle as ro
    from instance_nerf_b200 import synthetic
    from instance_nerf_b200.nerf.utils import get_rays
    from instance_nerf_b200.projection import project_masks
    K = 8
    m, sc = build_model(cuda, K)
    v = m.extract_volume((48, 24, 40), view_dir=None, sigma_thresh=1.0, bbox=SUB)
    lab = v["label"]
    assert int(lab.min()) >= 0 and int(lab.max()) <= K and int((lab > 0).sum()) > 0
    poses = torch.from_numpy(synthetic.camera_poses(sc, 2, 1)).to(cuda)
    H, W = 40, 56
    intr = synthetic.intrinsics(H, W)
    frames, maps = project_masks(lab, v["bbox"], poses, intr, H, W)
    assert frames == [0, 1]
    assert int(maps.min()) >= 0 and int(maps.max()) <= K
    for f in frames:
        r = get_rays(poses[f][None], intr, H, W, -1)
        l0, _ = ro.project_labels(r["rays_o"].cpu().numpy().reshape(-1, 3), r["rays_d"].cpu().numpy().reshape(-1, 3), lab.cpu().numpy(),
                                  np.asarray(v["bbox"], np.float32))
        assert np.array_equal(maps[f].cpu().numpy().reshape(-1), l0)
    assert int((maps > 0).sum()) > 0
